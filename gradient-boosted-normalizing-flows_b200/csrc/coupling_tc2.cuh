// Pipelined tcgen05 / TMEM / bulk-TMA coupling-stack kernel (GBNF_GEMM_F16_TC*, coupling_network_depth == 1,
// hidden width a multiple of 128 up to 512).  Rows, activations and accumulators never leave the SM, and -- unlike
// coupling_tc.cuh -- the hidden activations never touch SHARED memory either: they are packed to fp16 in tensor memory
// and fed back to tcgen05.mma as the A operand from TMEM.  Shared memory then only carries the weight stream (written
// once by TMA, read once by the tensor pipe), which is what bounds a 128-row tile on one SM (measured: 128 B/clk of
// shared-memory bandwidth, 42 B/clk of L2->SM ingest, tools/tc_probe2.cu).
//
//   TMEM map (512 columns, T2Geom below):
//     A1 = columns [0, h/2): the layer-2 A operand, k-quarter q (128 K elements) at [64 q, 64 q + 64)
//     two accumulator slots after it (128 + 128 columns; 128 + 64 when h = 512) and the last-layer accumulator (64)
//     layer 1 (K = |z1|, A0 from smem):  chunk q (N = 128) -> L1 slot q & 1; epilogue: bias + act -> fp16 pairs -> A1 quarter q
//     layer 2 (K = h, A1 from TMEM):     chunk j (N = 128 or 64) -> slot j & 1; chunk 0 is accumulated k-quarter by k-quarter
//                                        behind the layer-1 epilogue, later chunks run one ahead of the epilogue;
//                                        epilogue: bias + act -> fp16 pairs packed IN PLACE = k-piece j of the last layer's A
//     last layer (N <= 64, A2 from TMEM): K-streamed piece by piece into the last-layer accumulator
//   Every reuse of a TMEM region is ordered either by the in-order tensor pipe or by an epilogue -> MMA mbarrier.
//
//   weights: layer 1 [128-col chunk][k-slab][128 x 16], layer 2 [chunk (128 / 64 wide)][k-slab][width x 16], last layer
//   [k-slab][Np x 16], fp16 canonical K-major slabs; one ring stage (<= 32 KB) = W1 of all layer-1 chunks, 32 KB of one
//   layer-2 chunk, or the k-slabs of one last-layer piece.  Producer and MMA warp walk the same fixed schedule.
//
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (both run warp-uniform control flow and issue from one elected
// lane, see ptx::elect_one), warps 2..17 = epilogue: four threads per row (column groups g = 0..3), each TMEM lane
// quadrant served by four warps.
#pragma once
#include "coupling_tc.cuh"

namespace gbnf {

constexpr int kT2Chunk = 128;        // layer-1 chunk = k-quarter of layer 2 = wide layer-2 chunk
constexpr int kT2Piece = 64;         // narrow layer-2 chunk (h = 512 only)
constexpr int kT2Threads = 576;       // 2 control warps + 16 epilogue warps
constexpr int kT2EpiThreads = 512;
constexpr int kT2MaxStages = 8;
constexpr uint32_t kT2W3Bytes = 16384;      // one last-layer piece: <= 8 k-slabs of [64 x 16]
constexpr uint32_t kT2StageBytes = 32768;   // ring slot: up to 16 layer-2 k-slabs; fewer, larger handshakes (see acquire())
constexpr uint32_t kT2TraceUnit = 37;

struct Tc2Misc {
  uint64_t full[kT2MaxStages];
  uint64_t empty[kT2MaxStages];
  uint64_t a0r;       // epilogue -> MMA : A0 written, every TMEM region of the previous pass drained        (8 arrivals)
  uint64_t a1r[4];    // epilogue -> MMA : A1 k-quarter q packed into T(q)[0:64], hole H(q) free               (4 arrivals)
  uint64_t sr[3];     // epilogue -> MMA : A2 piece stored in hole i, its accumulator drained                  (4 arrivals)
  uint64_t l1f[4];    // MMA -> epilogue : layer-1 chunk q accumulated        (tcgen05.commit)
  uint64_t l2f[3];    // MMA -> epilogue : layer-2 chunk in hole i accumulated
  uint64_t l3f;       // MMA -> epilogue : last layer accumulated
  uint64_t w3full[2]; // producer -> MMA : last-layer weights of a piece landed in their own double buffer (outside the ring)
  uint64_t w3empty[2];// MMA -> producer : that buffer may be refilled
  uint32_t tmem_base;
  uint32_t last_flag;
  int meta[2][8];     // per step (double buffered): in_dim, out_dim, Kp of layer 1, Np of the last layer (net 0, 1), bias offsets
                      // (net 0, 1), offset of the gather-order tables (t2_stage_meta)
  float coef[kMaxComponents];
};

constexpr uint32_t kT2MiscBytes = 1536;
static_assert(sizeof(Tc2Misc) <= kT2MiscBytes, "misc region too small");

__host__ __device__ inline uint32_t t2_bias_stride(int h) { return (uint32_t)(2 * h + 64); }   // floats per bias buffer

// Eligibility of a configuration for the pipelined kernel (host).
inline bool tc2_eligible(const ModelDims& md, const std::vector<StepDesc>& steps) {
  if (md.nlayers != 3 || md.h % kT2Chunk != 0 || md.h > 512 || md.D > kTcMaxD) return false;
  for (const StepDesc& s : steps)
    for (int n = 0; n < md.nnets; ++n) {
      if (s.layer[n][0].Kp > 32) return false;          // one ring stage holds W1 of all (<= 4) layer-1 chunks
      if (s.layer[n][2].Np > 64) return false;          // last-layer accumulator is the 64-column hole H(3)
    }
  return true;
}

// Shared-memory plan of the pipelined kernel: no A1 image, the space goes to the weight ring.
inline bool tc2_make_plan(const ModelDims& md, const std::vector<StepDesc>& steps, TcPlan* p) {
  int k0p = 16, out_max = 1;
  for (const StepDesc& s : steps) {
    k0p = std::max(k0p, s.layer[0][0].Kp);
    out_max = std::max(out_max, s.out_dim);
  }
  auto al = [](uint32_t v) { return (v + 127u) & ~127u; };
  p->K0p = k0p; p->out_max = out_max;
  uint32_t o = 0;
  p->off_zs = o;   o = al(o + kTcRows * md.Dv * 4);
  p->off_a0 = o;   o = al(o + (k0p / 16) * 4096);        // also hosts the per-row partial sums at the end of a component (6 x 128 floats)
  p->off_a1 = o;   o = al(o + kTcRows * md.D * 4);       // here: the untransformed x tile (reloaded into zs per component)
  p->off_sh = o;   o = al(o + (md.nnets == 2 ? kTcRows * out_max * 4 : 0));
  p->off_misc = o; o = al(o + kT2MiscBytes);
  p->off_bias = o; o = al(o + 2 * t2_bias_stride(md.h) * 4);   // b1 | b2 | b3 of the current and of the next pass
  p->off_tab = o;  o = al(o + 2 * 2 * kEpPad * 16);       // gather-order tables of the current and the next step
  p->off_w3 = o;   o = al(o + 2 * kT2W3Bytes);            // last-layer weights of two pieces (their own double buffer)
  p->off_ring = o;
  const uint32_t limit = 227 * 1024;
  p->nst = std::min<int>(kT2MaxStages, (limit - o) / kT2StageBytes);
  p->smem_bytes = o + (size_t)p->nst * kT2StageBytes;
  p->tmem_cols = 512;
  return p->nst >= 3;
}

// Epilogue warp -> MMA warp handoff: every lane has fenced its own writes, one lane arrives for the warp.
__device__ __forceinline__ void t2_warp_arrive(uint64_t* bar, int lane) {
  __syncwarp();
  if (lane == 0) ptx::mbar_arrive(bar);
}
// mbarrier wait polled by one lane per warp (256 spinning threads would compete with the MMA operand reads for shared memory)
__device__ __forceinline__ void t2_wait(uint64_t* bar, uint32_t parity, int* err, int code, int lane) {
  (void)lane;
  ptx::mbar_wait(bar, parity, err, code);   // all lanes poll: ~50 cycles less latency than one polling lane + __syncwarp
  __syncwarp();
}
// the four epilogue warps that share a TMEM lane quadrant (= the four threads of every row in it)
__device__ __forceinline__ void t2_quad_bar(int quad) { asm volatile("bar.sync %0, 128;" ::"r"(2 + quad) : "memory"); }
__device__ __forceinline__ void t2_epi_bar() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

// N (16 or 32) accumulator values of one row -> bias + activation -> N / 2 packed fp16 pairs
// (ReLU activations are unbounded: a value that is not finite in fp16 raises status word 2, see CouplingArgs::error_flag)
template <int ACT, int TANH_MODE, int N>
__device__ __forceinline__ void t2_act_pack(const uint32_t (&r)[N], const float* __restrict__ bias, uint32_t* p, int* status) {
  if (ACT == 2) {
    float mx = 0.f;
#pragma unroll
    for (int q = 0; q < N; ++q) mx = fmax_nan(mx, __uint_as_float(r[q]) + bias[q]);
    if (!(mx <= 65504.f)) *reinterpret_cast<volatile int*>(status + 2) = 1;
  }
#pragma unroll
  for (int q = 0; q < N / 4; ++q) {
    const float4 b = *reinterpret_cast<const float4*>(bias + 4 * q);      // staged in shared memory (broadcast read)
    float v0 = __uint_as_float(r[4 * q + 0]) + b.x, v1 = __uint_as_float(r[4 * q + 1]) + b.y;
    float v2 = __uint_as_float(r[4 * q + 2]) + b.z, v3 = __uint_as_float(r[4 * q + 3]) + b.w;
    tc_act4<ACT, TANH_MODE>(v0, v1, v2, v3);
    p[2 * q + 0] = pack_half2(v0, v1);
    p[2 * q + 1] = pack_half2(v2, v3);
  }
}

// ---- per-row epilogue code shared by the persistent tensor-core kernels (coupling_tc2/3/4/5.cuh): 512 epilogue threads,
//      four per row (column group g), et = epilogue thread index ----

// x tile of 128 rows -> xs (row-major, D floats a row, zero beyond row B; INV: from row row_end on), 8 independent loads in flight
// per thread
template <int INV = 0>
__device__ __forceinline__ void t2_load_x_tile(float* xs, const CouplingArgs& a, int D, long long row0, int et, long long row_end = 0) {
  const int total = kTcRows * D;
  const long long gbase = row0 * D;
  const long long glimit = (INV ? row_end : a.B) * (long long)D;
  for (int i0 = et; i0 < total; i0 += 8 * kT2EpiThreads) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * kT2EpiThreads;
      v[u] = (i < total && gbase + i < glimit) ? __ldg(a.x + gbase + i) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * kT2EpiThreads;
      if (i < total) xs[i] = v[u];
    }
  }
}

// ActNorm / eval-BatchNorm affine fused into the gather of z1 -> A0 (fp16, canonical layout, zero padded): this thread's
// 8-element chunks g, g + 4, ... of nch.  Forward: the row keeps the normalised value.  INV: the MLP input is z1 as it
// stands and the row keeps the un-normalised value (inverse tables).  FEED: the MLP input is z1 as it stands and the row is
// left untouched (a second network on the same z1, coupling_tc3.cuh).
template <int INV = 0, int FEED = 0>
__device__ __forceinline__ void t2_gather_z1(float* zrow, const float4* tab1, int in_dim, int nch, int g, int row,
                                             unsigned char* A0, int* status) {
  for (int ch = g; ch < nch; ch += 4) {
    // loads first, stores last: the compiler cannot prove that the gathered columns are distinct, so an interleaved
    // load / store sequence would be serialised on shared-memory latency
    float4 t[8];
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) t[e] = tab1[ch * 8 + e];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = zrow[__float_as_int(t[e].w)];
    if (FEED) {
      // the row keeps its values
    } else if (INV) {
#pragma unroll
      for (int e = 0; e < 8; ++e) if (ch * 8 + e < in_dim) zrow[__float_as_int(t[e].w)] = (v[e] + t[e].x) * t[e].y + t[e].z;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = (v[e] + t[e].x) * t[e].y + t[e].z;
#pragma unroll
      for (int e = 0; e < 8; ++e) if (ch * 8 + e < in_dim) zrow[__float_as_int(t[e].w)] = v[e];   // never write the scratch column
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = (ch * 8 + e < in_dim) ? v[e] : 0.f;
    {   // a value that fp16 cannot hold (|v| > 65504, inf, NaN) would silently become inf / NaN in the GEMM operand
      const float mx = fmax_nan(fmax_nan(fmax_nan(fabsf(v[0]), fabsf(v[1])), fmax_nan(fabsf(v[2]), fabsf(v[3]))),
                                fmax_nan(fmax_nan(fabsf(v[4]), fabsf(v[5])), fmax_nan(fabsf(v[6]), fabsf(v[7]))));
      if (!(mx <= 65504.f)) *reinterpret_cast<volatile int*>(status + 2) = 1;
    }
    st_shared_v4(A0 + a_chunk_off(row, ch * 8), pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]),
                 pack_half2(v[6], v[7]));
  }
}

// End of component c for this row: base-density quadratic over the thread's columns [h0col, h1col), the four groups'
// partial sums combined through part (quadratic) / part + 3 kTcRows (log-det) -- A0 is dead by then -- and, by the
// writer's group-0 thread, log q and the total log-det stored to logq / the peer gather buffers / ldj_out and coef[c] + log q
// to the mixture-term scratch.  base_off, ldj_const and base_const are the caller's: it loads them where their latency hides.
__device__ __forceinline__ void t2_component_logq(const CouplingArgs& a, const float* zrow, float lsum, float* part, int row, int g,
                                                  int quad, int h0col, int h1col, int Dv, long long base_off, float ldj_const,
                                                  float base_const, const float* coef, int c, int tile, bool writer) {
  const long long gr = (long long)tile * kTcRows + row;
  float* const part2 = part + 3 * kTcRows;
  float q = 0.f;
  if (a.md.base == GBNF_BASE_STD_NORMAL) {       // mean 0, 1 / (2 var) = 0.5: the same arithmetic as the table path, no loads
    for (int p = h0col; p < h1col; ++p) { const float d = zrow[p]; q = fmaf(d * d, 0.5f, q); }
  } else {
    const float* bm = a.fblob + base_off;
    const float* bi = bm + Dv;
    for (int p = h0col; p < h1col; ++p) { const float d = zrow[p] - __ldg(bm + p); q = fmaf(d * d, __ldg(bi + p), q); }
  }
  if (g > 0) { part[(g - 1) * kTcRows + row] = q; part2[(g - 1) * kTcRows + row] = lsum; }
  t2_quad_bar(quad);
  if (writer && g == 0) {
    q += part[row] + part[kTcRows + row] + part[2 * kTcRows + row];
    const float ldj_tot = (lsum + part2[row] + part2[kTcRows + row] + part2[2 * kTcRows + row]) + ldj_const;
    const float lq = (base_const - q) + ldj_tot;
    if (gr < a.B) {
      if (a.logq) a.logq[gr * a.ld_logq + (c - a.c0)] = lq;
      // component-parallel multi-GPU: the same value straight into every rank's gather buffer (peer memory over NVLink)
      for (int i = 0; i < a.n_peers; ++i) a.logq_peers[i][(long long)(a.peer_col0 + (c - a.c0)) * a.peer_ld + gr] = lq;
      if (a.ldj_out) a.ldj_out[gr] = ldj_tot;
    }
    if (a.G_ll != nullptr && c < a.n_mix) __stcg(a.lse_terms + gr * a.n_mix + c, coef[c] + lq);
  }
}

// End of a component in the inverse direction: the log-det of the inverse map, the four groups' shares combined in
// t2_component_logq's order, stored by the writer's group-0 thread for rows gr < row_end (the end of the work unit).
__device__ __forceinline__ void t2_inverse_ldj(const CouplingArgs& a, float lsum, float* part, int row, int g, int quad,
                                               float ldj_const, long long gr, long long row_end, bool writer) {
  float* const part2 = part + 3 * kTcRows;
  if (g > 0) part2[(g - 1) * kTcRows + row] = lsum;
  t2_quad_bar(quad);
  if (writer && g == 0 && gr < row_end && a.ldj_out)
    a.ldj_out[gr] = (lsum + part2[row] + part2[kTcRows + row] + part2[2 * kTcRows + row]) + ldj_const;
}

// G_ll of the tile's rows: logsumexp over their mixture terms in component order (two passes: exact max, then the sum), by
// the last of the tile's `split` units to arrive.  All 512 epilogue threads of the CTA call it together (the ticket takes
// two epilogue barriers).  gr = tile * kTcRows + row.
__device__ __forceinline__ void t2_tile_logsumexp(const CouplingArgs& a, int tile, long long gr, int g, int et, uint32_t* last_flag) {
  bool last = true;
  if (a.split > 1) {
    if (g == 0) __threadfence();
    t2_epi_bar();
    if (et == 0) *last_flag = (atomicAdd(a.tile_ctr + tile, 1u) == (unsigned)(a.split - 1)) ? 1u : 0u;
    t2_epi_bar();
    last = *last_flag != 0u;
    if (last && et == 0) a.tile_ctr[tile] = 0u;
    if (last && g == 0) __threadfence();
  }
  if (last && g == 0 && gr < a.B) {
    const float* tv = a.lse_terms + gr * a.n_mix;
    float M = -INFINITY;
    bool has_nan = false;
    for (int i = 0; i < a.n_mix; ++i) { const float t = __ldcg(tv + i); M = fmaxf(M, t); has_nan |= (t != t); }
    float S = 0.f;
    for (int i = 0; i < a.n_mix; ++i) { const float t = __ldcg(tv + i); if (t != -INFINITY) S += expf(t - M); }
    // torch.logsumexp semantics: a NaN term -> NaN (fmaxf drops it), +inf -> +inf, all terms -inf -> -inf
    a.G_ll[gr] = has_nan ? __int_as_float(0x7fc00000) : (M == INFINITY || M == -INFINITY) ? M : M + logf(S);
  }
}


// ---- TMEM geometry ---------------------------------------------------------------------------------------------
// A1 (layer-2 A operand, fp16 pairs) occupies columns [0, h/2): k-quarter q at [64 q, 64 q + 64).  Two accumulator slots
// follow; layer-2 chunk j lives in slot j & 1, layer-1 chunk q in L1 slot q & 1 (always 128 wide).  h = 512 leaves only
// 256 columns: slot 0 = 128, slot 1 = 64, last-layer accumulator = 64, and layer 2 is cut into chunks of 128/64/128/64/128
// columns; narrower models use two 128-column slots.  128-column accumulators matter because a tcgen05.mma costs ~44 cycles
// to issue (blocking issue + descriptor arithmetic) but an N=64 MMA executes in 32: only N=128 keeps the pipe busy.
struct T2Geom {
  int NQ, NJ;
  bool tight;
  bool l1_in_slot0;     // layer-1 accumulators share accumulator slot 0 (then layer-2 chunk 0 must wait for them to drain)
  bool l1_even_inplace; // the even layer-1 chunks accumulate inside the A1 region they are packed into
  uint32_t slot_col[2], l1_col[2], la_col;
  __device__ __forceinline__ int cw(int j) const { return (tight && (j & 1)) ? 64 : 128; }
  __device__ __forceinline__ int ccol(int j) const { return tight ? 192 * (j >> 1) + ((j & 1) ? 128 : 0) : 128 * j; }
};
__device__ __forceinline__ T2Geom t2_geom(int h) {
  T2Geom g;
  g.NQ = h / kT2Chunk;
  g.tight = (h == 512);
  g.NJ = g.tight ? 5 : g.NQ;
  const uint32_t a1w = (uint32_t)h >> 1;
  g.slot_col[0] = a1w; g.slot_col[1] = a1w + 128u;
  g.la_col = g.tight ? 448u : a1w + 256u;
  // Layer-1 accumulators (128 columns each, two in flight).  Keeping them OUT of slot 0 lets layer-2 chunk 0 start as soon as
  // the first A1 quarter exists.  h = 512: even chunks use the upper half of the A1 region itself ([128, 256): still unused
  // when chunk 0 accumulates, packed in place by chunk 2), odd chunks use slot 1 + the last-layer accumulator ([384, 512)).
  // h <= 256: slot 1 and the columns behind it are free.  h = 384 has no spare 128 columns: slots 0 / 1 as before.
  if (g.tight)        { g.l1_col[0] = 128u; g.l1_col[1] = 384u; g.l1_in_slot0 = false; g.l1_even_inplace = true; }
  else if (h <= 256)  { g.l1_col[0] = a1w + 128u; g.l1_col[1] = a1w + 256u; g.l1_in_slot0 = false; g.l1_even_inplace = false; }
  else                { g.l1_col[0] = a1w; g.l1_col[1] = a1w + 128u; g.l1_in_slot0 = true; g.l1_even_inplace = false; }
  return g;
}

// ---- the fixed per-pass schedule, walked identically by the TMA producer and the MMA issuer ------------------------
//   L1_STAGE  ()                 ring stage: W1 of all layer-1 chunks (held while the chunks are issued)
//   L1        (chunk q)          MMA only  : A0 x W1 chunk q -> L1 slot q & 1 (chunks >= 2 wait for the slot to be drained)
//   L2        (chunk j, part p)  ring stage: 32 KB of chunk j's weights = one k-quarter of a 128-column chunk, or two
//                                            k-quarters of a 64-column chunk; needs A1 quarters and a free slot
//   L2_DONE   (chunk j)          MMA only  : commit -> epilogue
//   L3_STAGE  (piece j)          ring stage: last-layer k-slabs of piece j, taken (and held) one chunk before they are used:
//                                            waiting for them at the point of use stalled the issuer for a TMA round trip
//   L3        (piece j)          MMA only  : waits for the packed piece, accumulates it, releases the held stage
enum { T2_OP_L1_STAGE = 0, T2_OP_L1, T2_OP_L2, T2_OP_L2_DONE, T2_OP_L3_STAGE, T2_OP_L3 };
template <class F>
__device__ __forceinline__ void t2_schedule(const T2Geom& g, F&& f) {
  f(T2_OP_L1_STAGE, 0, 0);
  f(T2_OP_L1, 0, 0);
  if (g.NQ > 1) f(T2_OP_L1, 1, 0);
  // chunk 0 (always 128 wide: one part per k-quarter) is interleaved with the remaining layer-1 chunks, so that its part q is
  // issued as soon as A1 quarter q exists
#pragma unroll
  for (int q = 0; q < g.NQ; ++q) {
    if (q + 2 < g.NQ) f(T2_OP_L1, q + 2, 0);
    f(T2_OP_L2, 0, q);
  }
  f(T2_OP_L2_DONE, 0, 0);
#pragma unroll
  for (int j = 1; j < g.NJ; ++j) {
    if (j >= 2) f(T2_OP_L3, j - 2, 0);                       // frees slot j & 1 (and the piece's weight stage)
    f(T2_OP_L3_STAGE, j - 1, 0);                             // weights of piece j - 1, a whole chunk before they are used
    const int parts = (g.cw(j) == 128) ? g.NQ : (g.NQ + 1) / 2;
#pragma unroll
    for (int p = 0; p < parts; ++p) f(T2_OP_L2, j, p);
    f(T2_OP_L2_DONE, j, 0);
  }
  if (g.NJ >= 2) f(T2_OP_L3, g.NJ - 2, 0);
  f(T2_OP_L3_STAGE, g.NJ - 1, 0);
  f(T2_OP_L3, g.NJ - 1, 0);
}

// PROF: per-role cycle counters of CTA 0 (gbnf_get_profile).  A clock64() costs ~30 cycles on the latency-bound single-warp
// roles, so the counters are compiled out of the production instantiation.
#define T2_CLOCK() (PROF == 1 ? clock64() : 0LL)
// event trace of ONE coupling pass (unit kT2TraceUnit of CTA 0): a.prof[32 + id] = clock64(), see tools/tc_trace.py
#define T2_TRACE(id) do { if (PROF && a.prof != nullptr && blockIdx.x == 0 && units == kT2TraceUnit && lane == 0) a.prof[32 + (id)] = clock64(); } while (0)
// One thread copies the scalars of a step's descriptor that the epilogue needs into shared memory a step ahead: a
// first-touch global load at the start of a step would sit on the critical path of every coupling pass.
__device__ __forceinline__ void t2_stage_meta(const StepDesc* sd, int nnets, int* m) {
  const int v0 = __ldg(&sd->in_dim), v1 = __ldg(&sd->out_dim), v2 = __ldg(&sd->layer[0][0].Kp);
  const int v3 = __ldg(&sd->layer[0][2].Np), v5 = (int)__ldg(&sd->layer[0][0].b_off);
  int v4 = 0, v6 = 0;
  if (nnets == 2) { v4 = __ldg(&sd->layer[1][2].Np); v6 = (int)__ldg(&sd->layer[1][0].b_off); }
  m[0] = v0; m[1] = v1; m[2] = v2; m[3] = v3; m[4] = v4; m[5] = v5; m[6] = v6; m[7] = (int)__ldg(&sd->ep_off);
}
// The same copy without stalling anybody: threads i = 0..7 each issue one 4-byte cp.async (the low words of the 64-bit
// offsets); the values are visible after the issuing threads' cp.async.wait_all and a CTA barrier.
__device__ __forceinline__ void t2_stage_meta_async(const StepDesc* sd, int nnets, int* m, int i) {
  const void* src = nullptr;
  switch (i) {
    case 0: src = &sd->in_dim; break;
    case 1: src = &sd->out_dim; break;
    case 2: src = &sd->layer[0][0].Kp; break;
    case 3: src = &sd->layer[0][2].Np; break;
    case 4: if (nnets == 2) src = &sd->layer[1][2].Np; break;
    case 5: src = &sd->layer[0][0].b_off; break;
    case 6: if (nnets == 2) src = &sd->layer[1][0].b_off; break;
    case 7: src = &sd->ep_off; break;
    default: break;
  }
  if (src != nullptr) ptx::cp_async4(m + i, src);
}
// b1 | b2 | b3 of one coupling pass (contiguous in fblob, 16-byte aligned) -> a bias buffer, asynchronously
__device__ __forceinline__ void t2_stage_bias_async(float* dst, const float* src, int nfloat, int et) {
  for (int i = et; i < (nfloat >> 2); i += kT2EpiThreads) ptx::cp_async16(dst + 4 * i, src + 4 * i);
}

// PROF: 0 production, 1 cycle counters + event trace, 2 event trace only (near-production timing).
// NQT: h / 128 as a compile-time constant (0 = read it from the model): with a constant geometry the whole schedule unrolls
// into straight-line code, which matters on the MMA-issuer warp where every dependent scalar instruction costs 4-6 cycles
// that are NOT hidden whenever a stage is issue-bound (measured ~400 cycles of bookkeeping per stage in the generic form).
// MV: model variant known at compile time - 1 = Glow / affine coupling / tanh nets (one net per step), 2 = RealNVP with tanh
// s- and t-nets (two nets per step), 0 = read everything from the model: the other coupling variants, activations and net
// counts drop out of the instantiation.
// INV: 1 = inverse direction (sampling): a.x = z in the flow's output column order, work units from `ut` (one component and
// up to 128 rows each, in any component order), steps walked from the last to the first; every pass runs the same MLP(s) on z1
// (which the forward step left untouched), un-does the coupling on z2 and un-does the ActNorm / BatchNorm affine through the
// INVERSE gather-order tables (pack_meta_kernel); writes a.z_out = x and a.ldj_out = log-det of the inverse map.  Upstream:
// FlowStep.decode models/glow.py:344-366, RealNVPFlow.decode models/realnvp.py:97-113.
template <int TANH_MODE, int PROF, int NQT, int MV = 0, int INV = 0>
__global__ void __launch_bounds__(kT2Threads, 1) coupling_tc2_kernel(CouplingArgs a, TcPlan plan, UnitTable ut) {
  extern __shared__ __align__(1024) unsigned char smem[];
  // PTX predicate registers that carry the result of an early mbarrier.test_wait across the MMA block issued in between
  // (warps issue in order: converting the predicate to a value right away would stall the issuer for the ~100-cycle
  // latency of the test; see acquire() below)
  asm volatile(".reg .pred t2_p_full;\n\t.reg .pred t2_p_sr;" ::);
  const ModelDims& md = a.md;
  const int D = md.D, Dv = md.Dv;
  const int nnets = MV == 1 ? 1 : MV == 2 ? 2 : md.nnets;
  float* zs = reinterpret_cast<float*>(smem + plan.off_zs);
  unsigned char* A0 = smem + plan.off_a0;
  float* xs = reinterpret_cast<float*>(smem + plan.off_a1);
  float* sh = reinterpret_cast<float*>(smem + plan.off_sh);
  float* bias_s = reinterpret_cast<float*>(smem + plan.off_bias);
  float4* tab_s = reinterpret_cast<float4*>(smem + plan.off_tab);
  Tc2Misc* misc = reinterpret_cast<Tc2Misc*>(smem + plan.off_misc);
  unsigned char* ring = smem + plan.off_ring;
  unsigned char* w3buf = smem + plan.off_w3;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nst = plan.nst;
  const T2Geom G = t2_geom(NQT ? NQT * kT2Chunk : md.h);
  const int NQ = G.NQ;                     // layer-1 chunks = k-quarters of layer 2
  const int NJ = G.NJ;                     // layer-2 chunks = k-pieces of the last layer
  const int hs = md.h >> 4;                // k-slabs of the h x h layer

  if (threadIdx.x == 0) {
    for (int i = 0; i < nst; ++i) { ptx::mbar_init(&misc->full[i], 1); ptx::mbar_init(&misc->empty[i], 1); }
    ptx::mbar_init(&misc->a0r, 16);
    for (int i = 0; i < 4; ++i) { ptx::mbar_init(&misc->a1r[i], 16); ptx::mbar_init(&misc->l1f[i], 1); }
    for (int i = 0; i < 3; ++i) { ptx::mbar_init(&misc->sr[i], 16); ptx::mbar_init(&misc->l2f[i], 1); }
    ptx::mbar_init(&misc->l3f, 1);
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&misc->w3full[i], 1); ptx::mbar_init(&misc->w3empty[i], 1); }
    ptx::fence_mbar_init();
    if (a.G_ll != nullptr) mixture_coefficients(a.rho, a.n_mix, a.skip_c, a.mix_mode, misc->coef);
  }
  if (warp == 1) ptx::tmem_alloc(&misc->tmem_base, 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tbase = misc->tmem_base;
  const __half* wb = reinterpret_cast<const __half*>(a.wblob);

  if (warp == 0) {
    // ===================================== TMA producer =====================================================
    uint32_t sidx = 0, par = 0, ph_w3 = 0;
    int slot = 0;                                    // ring position kept incrementally: a runtime % or / costs ~100 cycles
    const long long p_t0 = T2_CLOCK();                // on this single latency-bound warp
    long long p_wait = 0;
    auto push = [&](const __half* src, uint32_t bytes) {
      const long long tw = T2_CLOCK();
      t2_wait(&misc->empty[slot], par ^ 1u, a.error_flag, 10, lane);
      p_wait += T2_CLOCK() - tw;
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(&misc->full[slot], bytes);
        ptx::tma_bulk_g2s(ring + (size_t)slot * kT2StageBytes, src, bytes, &misc->full[slot]);
      }
      __syncwarp();
      ++sidx;
      if (++slot == nst) { slot = 0; par ^= 1u; }
    };
    for (int u = blockIdx.x; u < (INV ? inverse_units(a, ut) : a.num_units); u += gridDim.x) {
      const int cb = INV ? __ldg(&ut.unit[u].x) : a.c0 + (u % a.split) * a.comps_per_unit;
      const int ce = INV ? cb + 1 : min(a.c1, cb + a.comps_per_unit);
      for (int c = cb; c < ce; ++c)
        for (int kk = 0; kk < md.K; ++kk) {
          const int k = INV ? md.K - 1 - kk : kk;
          const StepDesc* sd = a.steps + (c * md.K + k);
          for (int net = 0; net < nnets; ++net) {
            const int k0s = __ldg(&sd->layer[net][0].Kp) >> 4;
            const int np3 = __ldg(&sd->layer[net][2].Np);
            const __half* w1 = wb + __ldg(&sd->layer[net][0].w_off);
            const __half* w2 = wb + __ldg(&sd->layer[net][1].w_off);
            const __half* w3 = wb + __ldg(&sd->layer[net][2].w_off);
            t2_schedule(G, [&](int op, int x, int y) {
              if (op == T2_OP_L1_STAGE) {
                push(w1, (uint32_t)(NQ * k0s) * 4096u);
              } else if (op == T2_OP_L2) {
                const __half* base = w2 + (size_t)G.ccol(x) * hs * 16;      // chunk x: [k-slab][width x 16]
                if (G.cw(x) == 128) {
                  push(base + (size_t)(8 * y) * 2048, 32768u);                // k-quarter y: 8 slabs of 128 x 16
                } else {
                  const int q0 = 2 * y, nq = min(2, NQ - q0);
                  push(base + (size_t)(8 * q0) * 1024, (uint32_t)nq * 16384u); // two k-quarters: 16 slabs of 64 x 16
                }
              } else if (op == T2_OP_L3_STAGE) {
                const int b = x & 1;
                t2_wait(&misc->w3empty[b], ((ph_w3 >> b) & 1u) ^ 1u, a.error_flag, 11, lane);
                ph_w3 ^= 1u << b;
                if (ptx::elect_one()) {
                  const uint32_t bytes = (uint32_t)((G.cw(x) >> 4) * np3) * 32u;
                  ptx::mbar_arrive_expect_tx(&misc->w3full[b], bytes);
                  ptx::tma_bulk_g2s(w3buf + (size_t)b * kT2W3Bytes, w3 + (size_t)(G.ccol(x) >> 4) * np3 * 16, bytes, &misc->w3full[b]);
                }
                __syncwarp();
              }
            });
          }
        }
    }
    if (PROF == 1 && a.prof != nullptr && blockIdx.x == 0 && lane == 0) { a.prof[16] = T2_CLOCK() - p_t0; a.prof[17] = p_wait; a.prof[18] = sidx; }
  } else if (warp == 1) {
    // ===================================== MMA issuer =======================================================
    uint32_t units = 0;
    uint32_t ph_sr = 0;                              // phase bits of the three hole barriers (bit i = parity of sr[i])
    int nslot = 0;                                   // next ring slot / its parity, kept incrementally (no runtime % or /)
    uint32_t npar = 0;
    const long long m_t0 = T2_CLOCK();
    long long m_wa = 0, m_wf = 0, m_iss = 0, m_sr = 0, tw, ti;
    const uint64_t a0_desc = ptx::make_smem_desc(ptx::smem_u32(A0));
    const uint64_t ring_desc = ptx::make_smem_desc(ptx::smem_u32(ring));
    const uint64_t w3_desc = ptx::make_smem_desc(ptx::smem_u32(w3buf));
    uint32_t ph_w3f = 0;
    const uint32_t idesc_l1 = ptx::make_idesc_f16(128, kT2Chunk);
    const uint32_t idesc_l2 = ptx::make_idesc_f16(128, kT2Piece);
    int slot = 0;
    // An mbarrier test costs 100-160 cycles on this warp even when the phase has long completed, and tcgen05.mma issue is
    // nearly synchronous with execution (tools/tc_probe3.cu, tc_probe4.cu): every handshake between two MMA blocks idles
    // the tensor pipe.  Hence (1) ring slots are large (up to 16 MMAs per handshake) and (2) the readiness of the NEXT
    // stage is tested (non-blocking) before the current stage's MMAs are issued and only consumed afterwards.
    auto test_full = [&](uint64_t* bar, uint32_t par) {
      asm volatile("mbarrier.test_wait.parity.shared::cta.b64 t2_p_full, [%0], %1;" ::"r"(ptx::smem_u32(bar)), "r"(par) : "memory");
    };
    test_full(&misc->full[0], 0u);
    auto acquire = [&]() -> uint64_t {
      slot = nslot;
      tw = T2_CLOCK();
      uint32_t full_ok;
      asm volatile("selp.u32 %0, 1, 0, t2_p_full;" : "=r"(full_ok));
      if (!full_ok) ptx::mbar_wait(&misc->full[slot], npar, a.error_flag, 21);
      m_wf += T2_CLOCK() - tw;
      ptx::tc_fence_after();
      if (++nslot == nst) { nslot = 0; npar ^= 1u; }
      test_full(&misc->full[nslot], npar);             // result consumed at the next acquire()
      return ring_desc + (uint64_t)((uint32_t)slot * (kT2StageBytes >> 4));
    };
    auto stage_take = [&]() -> uint64_t { return acquire(); };
    auto wait_epi = [&](uint64_t* bar, uint32_t par, int code) {
      tw = T2_CLOCK();
      ptx::mbar_wait(bar, par, a.error_flag, code);
      m_wa += T2_CLOCK() - tw;
      ptx::tc_fence_after();
    };
    for (int u = blockIdx.x; u < (INV ? inverse_units(a, ut) : a.num_units); u += gridDim.x) {
      const int cb = INV ? __ldg(&ut.unit[u].x) : a.c0 + (u % a.split) * a.comps_per_unit;
      const int ce = INV ? cb + 1 : min(a.c1, cb + a.comps_per_unit);
      for (int c = cb; c < ce; ++c)
        for (int kk = 0; kk < md.K; ++kk) {
          const int k = INV ? md.K - 1 - kk : kk;
          const StepDesc* sd = a.steps + (c * md.K + k);
          for (int net = 0; net < nnets; ++net, ++units) {
            const int k0s = __ldg(&sd->layer[net][0].Kp) >> 4;
            const int np3 = __ldg(&sd->layer[net][2].Np);
            const uint32_t idesc_o = ptx::make_idesc_f16(128, np3);
            const uint32_t b3_step = (uint32_t)np3 * 2u;       // (np3 * 32 B) >> 4
            const uint32_t upar = units & 1u;
            uint64_t l1_desc = 0;                              // the held layer-1 weight stage
            int l1_slot = 0;
            int a1_waited = 0;                                 // a1r[0 .. a1_waited) have been observed
            uint32_t sr_pre = 0;                               // an early test of the next piece's barrier is pending in t2_p_sr
            auto need_a1 = [&](int upto) {
              while (a1_waited <= upto) { wait_epi(&misc->a1r[a1_waited], upar, 22); T2_TRACE(5 + a1_waited); ++a1_waited; }
            };

            t2_schedule(G, [&](int op, int x, int y) {
              if (op == T2_OP_L1_STAGE) {
                l1_desc = stage_take();
                l1_slot = slot;
                T2_TRACE(138);
              } else if (op == T2_OP_L1) {
                // layer-1 chunk x: A0 (smem) x W1 chunk -> L1 slot x & 1 (drained by the epilogue of chunk x - 2)
                if (x == 0) { wait_epi(&misc->a0r, upar, 20); T2_TRACE(0); }   // A0 gathered, TMEM of the previous pass drained
                if (x >= 2) need_a1(x - 2);
                ti = T2_CLOCK();
                if (ptx::elect_one()) {
                  const uint32_t d = tbase + G.l1_col[x & 1];
                  const uint64_t bq = l1_desc + (uint64_t)(x * k0s * 256);
                  for (int i = 0; i < k0s; ++i)
                    ptx::umma_f16(d, a0_desc + (uint64_t)(i * 256), bq + (uint64_t)(i * 256), idesc_l1, i > 0 ? 1u : 0u);
                  ptx::umma_commit(&misc->l1f[x]);
                  if (x == NQ - 1) ptx::umma_commit(&misc->empty[l1_slot]);
                }
                __syncwarp();
                m_iss += T2_CLOCK() - ti;
                T2_TRACE(1 + x);
              } else if (op == T2_OP_L2) {
                // layer-2 chunk x (slot x & 1), part y: A1 k-quarters from TMEM x k-slabs of [width x 16]
                const int w = G.cw(x);
                const int q0 = (w == 128) ? y : 2 * y;
                const int nq = (w == 128) ? 1 : min(2, NQ - q0);
                // the A1 quarters of this part, and a slot free of layer-1 accumulators (slot 0 hosted the even chunks)
                need_a1(max(q0 + nq - 1, x == 0 ? (G.l1_in_slot0 ? ((NQ - 1) & ~1) : 0) : NQ - 1));
                if (x == 3) T2_TRACE(130 + 3 * (y & 1));
                const uint64_t bd = stage_take();
                const int cur_slot = slot;
                if (x == 3) T2_TRACE(131 + 3 * (y & 1));
                // The op after the LAST part of chunk x >= 1 is the last-layer piece x - 1: test its barrier
                // now, so that its latency overlaps with the MMAs issued below instead of idling the pipe.
                const bool pre_l3 = (q0 + nq == NQ) && x >= 1;
                if (pre_l3) {
                  const int sn = (x - 1) & 1;
                  asm volatile("mbarrier.test_wait.parity.shared::cta.b64 t2_p_sr, [%0], %1;" ::"r"(ptx::smem_u32(&misc->sr[sn])),
                               "r"((ph_sr >> sn) & 1u) : "memory");
                  sr_pre = 1;
                }
                ti = T2_CLOCK();
                if (ptx::elect_one()) {
                  const uint32_t d = tbase + G.slot_col[x & 1];
                  if (w == 128) {
                    const uint32_t at = tbase + (uint32_t)q0 * 64u;
                    ptx::umma_f16_ts(d, at, bd, idesc_l1, q0 > 0 ? 1u : 0u);
#pragma unroll
                    for (int i = 1; i < 8; ++i) ptx::umma_f16_ts(d, at + 8u * i, bd + (uint64_t)(i * 256), idesc_l1, 1u);
                  } else {
                    for (int qq = 0; qq < nq; ++qq) {
                      const uint32_t at = tbase + (uint32_t)(q0 + qq) * 64u;
                      const uint64_t bq = bd + (uint64_t)(qq * 1024);
                      ptx::umma_f16_ts(d, at, bq, idesc_l2, (q0 + qq) > 0 ? 1u : 0u);
#pragma unroll
                      for (int i = 1; i < 8; ++i) ptx::umma_f16_ts(d, at + 8u * i, bq + (uint64_t)(i * 128), idesc_l2, 1u);
                    }
                  }
                  ptx::umma_commit(&misc->empty[cur_slot]);
                  if (q0 + nq == NQ) ptx::umma_commit(&misc->l2f[x & 1]);      // chunk complete -> epilogue
                }
                __syncwarp();
                m_iss += T2_CLOCK() - ti;
                if (x == 3) T2_TRACE(132 + 3 * (y & 1));
              } else if (op == T2_OP_L2_DONE) {
                T2_TRACE(10 + x);
              } else if (op == T2_OP_L3_STAGE) {
                // producer-only op: the piece's weights go to their own buffer
              } else {
                // last layer, k-piece x held packed in slot x & 1 (128-column chunk: 8 slabs at slot + 8 i; 64-column
                // chunk: 4 slabs at slot + 16 i) -> last-layer accumulator
                const int sl = x & 1;
                const int w = G.cw(x);
                if (x == 1) T2_TRACE(136);
                ti = T2_CLOCK();
                uint32_t sr_ok = 0;
                if (sr_pre) asm volatile("selp.u32 %0, 1, 0, t2_p_sr;" : "=r"(sr_ok));
                sr_pre = 0;
                if (!sr_ok) ptx::mbar_wait(&misc->sr[sl], (ph_sr >> sl) & 1u, a.error_flag, 23);
                ptx::tc_fence_after();
                m_sr += T2_CLOCK() - ti;
                ph_sr ^= 1u << sl;
                if (x == 1) T2_TRACE(137);
                ptx::mbar_wait(&misc->w3full[sl], (ph_w3f >> sl) & 1u, a.error_flag, 24);   // landed a chunk ago
                ptx::tc_fence_after();
                ph_w3f ^= 1u << sl;
                const uint64_t bd = w3_desc + (uint64_t)((uint32_t)sl * (kT2W3Bytes >> 4));
                if (ptx::elect_one()) {
                  const uint32_t at = tbase + G.slot_col[sl], d = tbase + G.la_col;
                  const uint32_t astep = (w == 128) ? 8u : 16u;
                  const int nsl = w >> 4;
                  for (int i = 0; i < nsl; ++i)
                    ptx::umma_f16_ts(d, at + astep * i, bd + (uint64_t)((uint32_t)i * b3_step), idesc_o, (x > 0 || i > 0) ? 1u : 0u);
                  ptx::umma_commit(&misc->w3empty[sl]);
                  if (x == NJ - 1) ptx::umma_commit(&misc->l3f);
                }
                __syncwarp();
                T2_TRACE(20 + x);
              }
            });
          }
        }
    }
    if (PROF == 1 && a.prof != nullptr && blockIdx.x == 0 && lane == 0) {
      a.prof[0] = T2_CLOCK() - m_t0; a.prof[1] = m_wa; a.prof[2] = m_wf; a.prof[3] = units; a.prof[4] = m_iss; a.prof[5] = m_sr;
    }
  } else {
    // ===================================== epilogue / elementwise warps =====================================
    // 16 warps = 4 groups (g) x 4 TMEM lane quadrants: FOUR threads per row, each owning a quarter of every chunk's
    // columns.  Four warps per scheduler hide the tcgen05.ld / st and barrier latencies of one another, which two
    // warps per scheduler could not (measured: 27 % of the MUFU bound with 8 warps).
    const int et = threadIdx.x - 64;
    const int warp_e = et >> 5;
    const int quad = warp & 3;             // TMEM lane quadrant this warp may access
    const int g = warp_e >> 2;             // column group 0..3
    const int row = quad * 32 + lane;
    float* zrow = zs + row * Dv;
    const uint32_t lane_base = tbase + ((uint32_t)(quad * 32) << 16);
    const int dq = (D + 3) >> 2;
    const int h0col = min(D, g * dq), h1col = min(D, (g + 1) * dq);   // column split for elementwise passes
    uint32_t units = 0, stepc = 0;
    uint32_t ph_l2f = 0;
    float* const part = reinterpret_cast<float*>(A0);   // per-row partial sums of a component's log-density (A0 is dead by then)
    const uint32_t bstride = t2_bias_stride(md.h);
    // the first step's gather-order tables, scalars and biases; afterwards every pass stages what the next one needs
    // (cp.async issued while this pass waits for the tensor core, completed and published at the end of the pass)
    if (blockIdx.x < (INV ? inverse_units(a, ut) : a.num_units)) {
      const int cb0 = INV ? __ldg(&ut.unit[blockIdx.x].x) : a.c0 + ((int)blockIdx.x % a.split) * a.comps_per_unit;
      const StepDesc* sd0 = a.steps + cb0 * md.K + (INV ? md.K - 1 : 0);
      if (et < 2 * kEpPad) ptx::cp_async16(tab_s + et, reinterpret_cast<const float4*>(a.fblob + __ldg(&sd0->ep_off)) + (INV ? 2 * kEpPad : 0) + et);
      if (et == 0) t2_stage_meta(sd0, nnets, misc->meta[0]);
      t2_stage_bias_async(bias_s, a.fblob + __ldg(&sd0->layer[0][0].b_off), 2 * md.h + __ldg(&sd0->layer[0][2].Np), et);
    }
    const bool tr = (warp_e & 3) == 0;     // one tracing warp per group
    const long long e_t0 = T2_CLOCK();
    long long e_w1 = 0, e_w2 = 0, e_w3 = 0, e_l1 = 0, e_l2 = 0, e_l3 = 0, e_pro = 0, e_x = 0, e_tmp;
    for (int u = blockIdx.x; u < (INV ? inverse_units(a, ut) : a.num_units); u += gridDim.x) {
      const int tile = u / a.split, cs = u - tile * a.split;
      const int4 un = INV ? __ldg(ut.unit + u) : make_int4(0, 0, 0, 0);   // INV: {component, first row, rows}
      const int cb = INV ? un.x : a.c0 + cs * a.comps_per_unit, ce = INV ? cb + 1 : min(a.c1, cb + a.comps_per_unit);
      const long long row0 = INV ? (long long)un.y : (long long)tile * kTcRows;
      const long long row_end = row0 + un.z;         // INV: end of the unit's rows
      const long long gr = row0 + row;
      for (int c = cb; c < ce; ++c) {
        // ---- x tile: fetched from HBM once per tile (8 independent loads in flight per thread) and kept in shared
        //      memory; every component restarts from it ----
        e_tmp = T2_CLOCK();
        // the component's scalars for the END of the component, fetched now with independent loads: three dependent L2 round
        // trips there (descriptor -> offsets -> constants) would sit on the critical path of every component
        const CompDesc* cdp = a.comps + c;
        const float2 cconst = __ldg(reinterpret_cast<const float2*>(a.fblob + a.cc_off) + c);   // {ldj constant, base constant}
        const long long base_off = (md.base == GBNF_BASE_STD_NORMAL) ? 0LL : __ldg(&cdp->base_off);
        const float ldj_const = cconst.x, base_const = cconst.y;
        t2_epi_bar();                                // previous component's readers are done with zs / part
        if (c == cb) {
          t2_load_x_tile<INV>(xs, a, D, row0, et, row_end);
          t2_epi_bar();
        }
        if (INV) {   // z arrives in the flow's OUTPUT column order: logical column p lives at physical column sigma[p]
          const int* sig = a.iblob + __ldg(&cdp->sigma_off);
          for (int p = h0col; p < h1col; ++p) zrow[__ldg(sig + p)] = xs[row * D + p];
        } else {
          for (int p = h0col; p < h1col; ++p) zrow[p] = xs[row * D + p];   // this thread's quarter of its own row (no div / mod)
        }
        if (g == 0) for (int p = D; p < Dv; ++p) zrow[p] = 0.f;           // scratch column(s): target of padded table entries
        ptx::cp_async_wait_all();                    // (first component of the launch: the prologue's staging copies)
        t2_epi_bar();
        e_x += T2_CLOCK() - e_tmp;
        float lsum = 0.f;                            // this thread's share of the data-dependent log-det
        for (int kk = 0; kk < md.K; ++kk, ++stepc) {
          const int k = INV ? md.K - 1 - kk : kk;
          e_tmp = T2_CLOCK();
          if (tr) T2_TRACE(72 + 40 * (g & 1));
          if (PROF && tr && g == 0 && a.prof != nullptr && blockIdx.x == 0 && units == kT2TraceUnit + 1 && lane == 0) a.prof[32 + 201] = clock64();
          const StepDesc* sd = a.steps + (c * md.K + k);
          const int* meta = misc->meta[stepc & 1u];                          // staged a step ahead
          const int out_dim = meta[1], in_dim = meta[0];
          const float4* tab1 = tab_s + (stepc & 1u) * (2 * kEpPad);          // staged by the previous step
          const float4* tab2 = tab1 + kEpPad;
          // the step after this one (next k, next component, or the first step of this CTA's next tile)
          const int kfirst = INV ? md.K - 1 : 0;
          const StepDesc* sd_next = (kk + 1 < md.K) ? (INV ? sd - 1 : sd + 1)
                                    : (c + 1 < ce) ? a.steps + (c + 1) * md.K + kfirst
                                    : (u + (int)gridDim.x < (INV ? inverse_units(a, ut) : a.num_units))
                                        ? a.steps + (INV ? __ldg(&ut.unit[u + gridDim.x].x)
                                                         : a.c0 + ((u + (int)gridDim.x) % a.split) * a.comps_per_unit) * md.K + kfirst
                                        : nullptr;
          // ---- ActNorm / eval-BatchNorm affine fused into the gather of z1 -> A0 ----
          t2_gather_z1<INV>(zrow, tab1, in_dim, meta[2] >> 3, g, row, A0, a.error_flag);
          e_pro += T2_CLOCK() - e_tmp;
          if (tr) T2_TRACE(73 + 40 * (g & 1));
          for (int net = 0; net < nnets; ++net, ++units) {
            const int act_kind = MV ? 1 : (md.act == GBNF_ACT_TANH) ? 1 : (md.act == GBNF_ACT_RELU) ? 2 : (net == 0 ? 2 : 1);
            const float* bias_c = bias_s + (units & 1u) * bstride;           // staged by the previous pass
            const float* b1 = bias_c + g * 32;
            const float* bias = bias_c + 2 * md.h;
            const uint32_t upar = units & 1u;
            const int np3 = meta[3 + net];
            // hand A0 (and every drained TMEM region) to the MMA warp
            ptx::fence_proxy_async_smem();
            ptx::tc_fence_before();
            t2_warp_arrive(&misc->a0r, lane);
            if (tr) T2_TRACE(40 + 40 * (g & 1));
            if (PROF && tr && g == 0 && a.prof != nullptr && blockIdx.x == 0 && units == kT2TraceUnit + 1 && lane == 0) a.prof[32 + 200] = clock64();
            // ---- staging for the NEXT pass, entirely off the critical path (a first-touch global load here, or in the
            //      chunk epilogues, would stall all four warps of a scheduler for an L2 round trip): the next step's scalars
            //      now; its tables and the next pass's biases once those scalars are visible (after layer 1, below) ----
            if (net == 0 && sd_next != nullptr && et < 8) t2_stage_meta_async(sd_next, nnets, misc->meta[(stepc + 1) & 1u], et);
            // ---- layer 1: chunk q in L1 slot q & 1 (128 columns, 32 per thread) -> act -> fp16 pairs written to the A1
            //      region [64 q, 64 q + 64) (normally a different TMEM region; see T2Geom::l1_even_inplace) ----
            for (int q = 0; q < NQ; ++q) {
              e_tmp = T2_CLOCK();
              t2_wait(&misc->l1f[q], upar, a.error_flag, 30, lane);
              if (tr) T2_TRACE(41 + 40 * (g & 1) + q);
              e_w1 += T2_CLOCK() - e_tmp;
              ptx::tc_fence_after();
              e_tmp = T2_CLOCK();
              uint32_t p[16];
              {
                uint32_t r[32];
                ptx::tmem_ld32(lane_base + G.l1_col[q & 1] + (uint32_t)g * 32u, r);
                ptx::tmem_ld_wait();
                if (PROF && warp_e == 0 && q == 1) T2_TRACE(120);
                if (act_kind == 1) t2_act_pack<1, TANH_MODE>(r, b1 + q * kT2Chunk, p, a.error_flag);
                else               t2_act_pack<2, TANH_MODE>(r, b1 + q * kT2Chunk, p, a.error_flag);
                if (PROF && warp_e == 0 && q == 1) T2_TRACE(121);
              }
              if (G.l1_even_inplace && !(q & 1)) t2_quad_bar(quad);   // packed quarter may overlap the row's unread accumulator
              ptx::tmem_st16(lane_base + (uint32_t)q * 64u + (uint32_t)g * 16u, p);
              ptx::tmem_st_wait();
              if (PROF && warp_e == 0 && q == 1) T2_TRACE(122);
              ptx::tc_fence_before();
              t2_warp_arrive(&misc->a1r[q], lane);
              if (tr) T2_TRACE(45 + 40 * (g & 1) + q);
              e_l1 += T2_CLOCK() - e_tmp;
            }
            // the epilogue now idles until layer-2 chunk 0 completes: publish the next step's scalars and start the copies
            // that depend on them (biases b1 | b2 | b3 of the next pass are contiguous in fblob)
            ptx::cp_async_wait_all();
            t2_epi_bar();
            if (net + 1 < nnets) {
              t2_stage_bias_async(bias_s + ((units + 1) & 1u) * bstride, a.fblob + meta[5 + net + 1], 2 * md.h + meta[3 + net + 1], et);
            } else if (sd_next != nullptr) {
              const int* mn = misc->meta[(stepc + 1) & 1u];
              t2_stage_bias_async(bias_s + ((units + 1) & 1u) * bstride, a.fblob + mn[5], 2 * md.h + mn[3], et);
              if (et >= kT2EpiThreads - 2 * kEpPad) {
                const int i = et - (kT2EpiThreads - 2 * kEpPad);
                ptx::cp_async16(tab_s + ((stepc + 1) & 1u) * (2 * kEpPad) + i, reinterpret_cast<const float4*>(a.fblob + mn[7]) + (INV ? 2 * kEpPad : 0) + i);
              }
            }
            // ---- layer 2: chunk j in slot j & 1 -> act -> fp16 pairs packed in place = k-piece j of the last layer's A
            //      operand.  128-column chunk: 32 columns per thread compacted into slot[0:64) (the quadrant's four warps
            //      synchronise between reading and overwriting); 64-column chunk: 16 columns per thread packed into the first
            //      8 of the thread's own columns (no hazard) ----
            for (int j = 0; j < NJ; ++j) {
              const int sl = j & 1;
              e_tmp = T2_CLOCK();
              t2_wait(&misc->l2f[sl], (ph_l2f >> sl) & 1u, a.error_flag, 31, lane);
              ph_l2f ^= 1u << sl;
              if (tr) T2_TRACE(50 + 40 * (g & 1) + j);
              e_w2 += T2_CLOCK() - e_tmp;
              ptx::tc_fence_after();
              e_tmp = T2_CLOCK();
              const uint32_t sc = lane_base + G.slot_col[sl];
              const float* bj = bias_c + md.h + G.ccol(j);
              if (G.cw(j) == 128) {
                uint32_t p[16];
                {
                  uint32_t r[32];
                  ptx::tmem_ld32(sc + (uint32_t)g * 32u, r);
                  ptx::tmem_ld_wait();
                  if (act_kind == 1) t2_act_pack<1, TANH_MODE>(r, bj + g * 32, p, a.error_flag);
                  else               t2_act_pack<2, TANH_MODE>(r, bj + g * 32, p, a.error_flag);
                }
                t2_quad_bar(quad);             // all four threads of the row have read their columns
                ptx::tmem_st16(sc + (uint32_t)g * 16u, p);
              } else {
                uint32_t p[8];
                {
                  uint32_t r[16];
                  ptx::tmem_ld16(sc + (uint32_t)g * 16u, r);
                  ptx::tmem_ld_wait();
                  if (act_kind == 1) t2_act_pack<1, TANH_MODE>(r, bj + g * 16, p, a.error_flag);
                  else               t2_act_pack<2, TANH_MODE>(r, bj + g * 16, p, a.error_flag);
                }
                ptx::tmem_st8(sc + (uint32_t)g * 16u, p);
              }
              ptx::tmem_st_wait();
              ptx::tc_fence_before();
              t2_warp_arrive(&misc->sr[sl], lane);
              if (tr) T2_TRACE(60 + 40 * (g & 1) + j);
              e_l2 += T2_CLOCK() - e_tmp;
            }
            // ---- last layer: coupling transform on this thread's 16-column slice of H(3); branch-free over the padded
            //      gather-order tables (padded entries hit the scratch column and are masked out of the log-det) ----
            e_tmp = T2_CLOCK();
            t2_wait(&misc->l3f, upar, a.error_flag, 32, lane);
            if (tr) T2_TRACE(70 + 40 * (g & 1));
            e_w3 += T2_CLOCK() - e_tmp;
            ptx::tc_fence_after();
            e_tmp = T2_CLOCK();
            const int c0 = g * 16;
            if (c0 < np3) {
              uint32_t r[16];
              ptx::tmem_ld16(lane_base + G.la_col + (uint32_t)c0, r);
              ptx::tmem_ld_wait();
              // every branch: gather the affected z2 columns first, store them last (see the gather above)
              if (MV == 1 || (MV == 0 && md.kind == GBNF_KIND_GLOW && md.coupling == GBNF_COUPLING_AFFINE)) {
                const float2* bias2 = reinterpret_cast<const float2*>(bias);
                float4 t[8];
                float z[8];
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) t[jj] = tab2[g * 8 + jj];
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) z[jj] = zrow[__float_as_int(t[jj].w)];
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                  const int j = g * 8 + jj;
                  const float2 b = bias2[j];
                  const float shift = __uint_as_float(r[2 * jj]) + b.x;
                  const float raw = __uint_as_float(r[2 * jj + 1]) + b.y;
                  const float s = __fdividef(1.0f, 1.0f + __expf(-(raw + 2.0f)));      // sigmoid(raw + 2), glow.py:333
                  if (INV) {
                    const float y = __fdividef(z[jj], s) - shift;                       // glow.py:354-356
                    z[jj] = (y + t[jj].x) * t[jj].y + t[jj].z;                          // ActNorm reverse, layers.py:505-518
                    lsum -= (j < out_dim) ? __logf(s) : 0.f;                            // glow.py:357
                  } else {
                    const float zn = (z[jj] + t[jj].x) * t[jj].y + t[jj].z;
                    z[jj] = (zn + shift) * s;                                           // glow.py:334-335
                    lsum += (j < out_dim) ? __logf(s) : 0.f;                            // glow.py:338
                  }
                }
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) if (g * 8 + jj < out_dim) zrow[__float_as_int(t[jj].w)] = z[jj];
              } else {
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                  float4 t[8];
                  float z[8];
#pragma unroll
                  for (int jj = 0; jj < 8; ++jj) t[jj] = tab2[c0 + half * 8 + jj];
#pragma unroll
                  for (int jj = 0; jj < 8; ++jj) z[jj] = zrow[__float_as_int(t[jj].w)];
#pragma unroll
                  for (int jj = 0; jj < 8; ++jj) {
                    const int j = c0 + half * 8 + jj;
                    const float acc = __uint_as_float(r[half * 8 + jj]) + bias[j];
                    const float zn = INV ? 0.f : (z[jj] + t[jj].x) * t[jj].y + t[jj].z;
                    if (MV != 2 && md.kind == GBNF_KIND_GLOW) {
                      if (INV) z[jj] = ((z[jj] - acc) + t[jj].x) * t[jj].y + t[jj].z;   // glow.py:350, then ActNorm reverse
                      else     z[jj] = zn + acc;                                        // additive coupling, glow.py:328-329
                    } else if (net == 0) {                                              // RealNVP t_net: keep the shift
                      if (j < out_dim) sh[row * plan.out_max + j] = acc;
                    } else {                                                            // RealNVP s_net: transform
                      const float tt = (j < out_dim) ? sh[row * plan.out_max + j] : 0.f;
                      if (INV) {
                        const float y = (z[jj] - tt) * __expf(-acc);                    // inverse of transformations.py:575
                        z[jj] = (y + t[jj].x) * t[jj].y + t[jj].z;                      // eval-BatchNorm inverse
                        lsum -= (j < out_dim) ? acc : 0.f;
                      } else {
                        z[jj] = tt + zn * __expf(acc);                                  // transformations.py:575
                        lsum += (j < out_dim) ? acc : 0.f;                              // transformations.py:577
                      }
                    }
                  }
                  if ((MV != 2 && md.kind == GBNF_KIND_GLOW) || net == 1) {
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) if (c0 + half * 8 + jj < out_dim) zrow[__float_as_int(t[jj].w)] = z[jj];
                  }
                }
              }
            }
            // z2 updates visible to the row's other threads, and the staged biases / tables / scalars of the next pass to
            // everybody, before the next gather
            if (tr) T2_TRACE(71 + 40 * (g & 1));
            ptx::cp_async_wait_all();
            t2_epi_bar();
            if (tr) T2_TRACE(74 + 40 * (g & 1));
            e_l3 += T2_CLOCK() - e_tmp;
          }
        }
        // ---- component log-density for this row (inverse: the log-det of the inverse map) ----
        if (INV) t2_inverse_ldj(a, lsum, part, row, g, quad, -ldj_const, gr, row_end, true);
        else     t2_component_logq(a, zrow, lsum, part, row, g, quad, h0col, h1col, Dv, base_off, ldj_const, base_const, misc->coef, c,
                                   tile, true);
        if (a.z_out != nullptr && gr < (INV ? row_end : a.B)) {
          if (INV) {   // physical == logical column order at the flow's input
            for (int j = h0col; j < h1col; ++j) a.z_out[gr * D + j] = zrow[j];
          } else {
            const int* sig = a.iblob + __ldg(&cdp->sigma_off);
            for (int j = h0col; j < h1col; ++j) a.z_out[gr * D + j] = zrow[__ldg(sig + j)];
          }
        }
      }
      if (a.G_ll != nullptr) t2_tile_logsumexp(a, tile, gr, g, et, &misc->last_flag);
    }
    if (PROF == 1 && a.prof != nullptr && blockIdx.x == 0 && et == 0) {
      a.prof[8] = T2_CLOCK() - e_t0; a.prof[9] = e_w1 + e_w2 + e_w3; a.prof[10] = e_l1 + e_l2; a.prof[11] = e_l3; a.prof[12] = e_pro + e_x;
      a.prof[13] = e_w1; a.prof[14] = e_w2; a.prof[15] = e_w3; a.prof[19] = e_l1; a.prof[20] = e_l2; a.prof[21] = e_x; a.prof[22] = e_pro;
    }
    ptx::tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tbase, 512);
  }
}

#undef T2_CLOCK
#undef T2_TRACE

template <int T, int P, int Q, int MV = 0, int INV = 0>
inline cudaError_t tc2_configure_one() {
  return cudaFuncSetAttribute(coupling_tc2_kernel<T, P, Q, MV, INV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}
// Instantiations.  Production (PROF = 0): geometry NQT in {4 (h = 512), 2 (h = 256), 0 (read from the model)} x model variant
// MV in {0 generic, 1 Glow / affine / tanh, 2 RealNVP / tanh} x both tanh modes; profiling builds (PROF = 1, 2) only exist for the
// generic variant and NQT in {0, 4}.
#define T2_FOR_PROD(X) X(4, 0) X(2, 0) X(0, 0) X(4, 1) X(2, 1) X(0, 1) X(4, 2) X(2, 2) X(0, 2)
inline cudaError_t tc2_configure() {
  cudaError_t e = cudaSuccess;
#define T2_CFG(T, P, Q) if (e == cudaSuccess) e = tc2_configure_one<T, P, Q>()
  T2_CFG(0, 1, 0); T2_CFG(1, 1, 0); T2_CFG(0, 2, 0); T2_CFG(1, 2, 0);
  T2_CFG(0, 1, 4); T2_CFG(1, 1, 4); T2_CFG(0, 2, 4); T2_CFG(1, 2, 4);
#undef T2_CFG
#define T2_CFG_PROD(Q, MV) if (e == cudaSuccess) e = tc2_configure_one<0, 0, Q, MV>(); if (e == cudaSuccess) e = tc2_configure_one<1, 0, Q, MV>();
  T2_FOR_PROD(T2_CFG_PROD)
#undef T2_CFG_PROD
  if (e == cudaSuccess) e = tc2_configure_one<0, 0, 0, 0, 1>();      // inverse direction: generic geometry / model variant
  if (e == cudaSuccess) e = tc2_configure_one<1, 0, 0, 0, 1>();
  return e;
}

inline int tc2_launch_inverse(const CouplingArgs& a, const TcPlan& p, const UnitTable& ut, int grid, cudaStream_t st) {
  if (p.tanh_mode == 0) coupling_tc2_kernel<0, 0, 0, 0, 1><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p, ut);
  else                  coupling_tc2_kernel<1, 0, 0, 0, 1><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p, ut);
  return 0;
}

inline int tc2_launch(const CouplingArgs& a, const TcPlan& p, int grid, cudaStream_t st, int prof) {
#define T2_GO(T, P, Q) coupling_tc2_kernel<T, P, Q><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p, UnitTable{})
#define T2_GO_Q(T, P) do { if (a.md.h == 512) T2_GO(T, P, 4); else T2_GO(T, P, 0); } while (0)
  if (prof == 1 || prof == 2) {
    if (p.tanh_mode == 0) { if (prof == 1) T2_GO_Q(0, 1); else T2_GO_Q(0, 2); }
    else                  { if (prof == 1) T2_GO_Q(1, 1); else T2_GO_Q(1, 2); }
    return 0;
  }
#undef T2_GO_Q
#undef T2_GO
  const int q = (a.md.h == 512) ? 4 : (a.md.h == 256) ? 2 : 0;
  const int mv = (a.md.kind == GBNF_KIND_GLOW && a.md.coupling == GBNF_COUPLING_AFFINE && a.md.act == GBNF_ACT_TANH && a.md.nnets == 1) ? 1
               : (a.md.kind == GBNF_KIND_REALNVP && a.md.act == GBNF_ACT_TANH && a.md.nnets == 2) ? 2 : 0;
#define T2_GO_PROD(Q, MV) \
  if (q == Q && mv == MV) { \
    if (p.tanh_mode == 0) coupling_tc2_kernel<0, 0, Q, MV><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p, UnitTable{}); \
    else                  coupling_tc2_kernel<1, 0, Q, MV><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p, UnitTable{}); \
    return 0; \
  }
  T2_FOR_PROD(T2_GO_PROD)
#undef T2_GO_PROD
  return -1;
}
#undef T2_FOR_PROD

}  // namespace gbnf
