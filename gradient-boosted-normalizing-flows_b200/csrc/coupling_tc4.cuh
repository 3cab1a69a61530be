// Two-chain variant of the pipelined tcgen05 / TMEM kernel (coupling_tc2.cuh) for the headline shape: Glow steps with an
// affine coupling and ONE tanh MLP of hidden width 512 (BASELINE configurations 3 and 4), forward direction.
//
// Why: at h = 512 the layer-2 A operand of a 128-row tile (A1, 256 TMEM columns) plus the accumulators fill tensor memory, so a
// coupling pass of coupling_tc2_kernel cannot be double buffered and the tensor pipe idles during the pass's two serial ends:
// the layer-1 phase (gather -> K = 32 GEMM -> 128 x 512 tanh, MUFU bound) and the tail (last chunk epilogue -> last last-layer
// piece -> coupling transform -> barrier -> next gather), together ~11 k of a 24.6 k cycle pass (profiles/r01_tc2_timeline.txt).
// Steps of one component depend on each other, but COMPONENTS do not: this kernel gives every CTA two chains X and Y (the two
// halves of a work unit's components, same 128 rows, own z tile / A0 / bias / table buffers) whose passes strictly alternate
// and TIME-SHARE the tensor memory:
//
//   slot s (chain B = s & 1 starts pass P_s; chain A = the other one finishes P_{s-1}):
//     tensor pipe : [L1(0) of P_s] [last last-layer piece of P_{s-1}] [L1(1..3), layer 2 and last-layer pieces 0..3 of P_s]
//     epilogue    : A: last layer-2 chunk -> B: layer-1 chunks 0..3 -> A: coupling transform (reads A's last-layer accumulator, which
//                   no GEMM of B touches before B's first last-layer piece) -> B: layer-2 chunks 0, 1 -> A: end of component / x
//                   reload / gather of A's next pass (= P_{s+1}) and the staging for it -> B: layer-2 chunks 2, 3
//   A's transform, its log-density / mixture bookkeeping, the x reload and the gather of its next pass run while the tensor
//   pipe works through B's layer 2, where the epilogue warps used to wait; only A's last chunk epilogue (1.1 k) and B's layer-1
//   phase (4.8 k, MUFU bound) remain exposed per pass.  Layer-1 accumulators are placed so that this needs no extra tensor
//   memory: chunk 0 -> [128, 256), chunk 1 -> slot 0, chunk 2 -> [128, 256), chunk 3 -> slot 1 + [192, 256) (two N = 64 halves).
//   The instruction footprint is kept small on purpose (one copy of every block, runtime chunk indices, DESIGN 4.1f).
//
// Everything else -- TMEM map, weight image, ring protocol, epilogue arithmetic -- is coupling_tc2_kernel's tight (h = 512)
// geometry with NQ = 4 layer-1 chunks and NJ = 5 layer-2 chunks (128 / 64 / 128 / 64 / 128 columns); results are bitwise
// identical to it (same operands, same accumulation order).  Shapes this kernel does not cover fall back to coupling_tc2_kernel
// on the same packed image: odd component counts per work unit, z_out requested, profiling builds.
#pragma once
#include "coupling_tc2.cuh"

namespace gbnf {

struct Tc4Misc {
  uint64_t full[kT2MaxStages];
  uint64_t empty[kT2MaxStages];
  uint64_t a0r[2];    // epilogue -> MMA : A0 of chain c gathered                                             (16 arrivals)
  uint64_t a1r[4];    // epilogue -> MMA : A1 k-quarter q packed, its layer-1 accumulator drained             (16 arrivals)
  uint64_t sr[2];     // epilogue -> MMA : last-layer A piece packed in slot i                                (16 arrivals)
  uint64_t l1f[4];    // MMA -> epilogue : layer-1 chunk q accumulated                                        (commit)
  uint64_t l2f[2];    // MMA -> epilogue : layer-2 chunk in slot i accumulated                                (commit)
  uint64_t l3f;       // MMA -> epilogue : last layer of a pass accumulated                                   (commit)
  uint64_t l3d;       // epilogue -> MMA : the transform has read the last-layer accumulator ([448, 512) free)   (16 arrivals)
  uint64_t c2r;       // epilogue -> MMA : layer-1 chunk 2's accumulator has been READ ([192, 256) may take half of chunk 3)  (16 arrivals)
  uint64_t w3full[2];
  uint64_t w3empty[2];
  uint32_t tmem_base;
  uint32_t last_flag;
  float coef[kMaxComponents];
};
static_assert(sizeof(Tc4Misc) <= kT2MiscBytes, "misc region too small");

// host: shape eligibility (per handle) -- the launch additionally needs an even number of components in every work unit
inline bool tc4_eligible(const ModelDims& md, const std::vector<StepDesc>& steps) {
  if (!tc2_eligible(md, steps) || steps.empty()) return false;
  if (md.h != 512 || md.nnets != 1 || md.kind != GBNF_KIND_GLOW || md.coupling != GBNF_COUPLING_AFFINE || md.act != GBNF_ACT_TANH) return false;
  const StepDesc& s0 = steps[0];
  for (const StepDesc& s : steps)
    if (s.in_dim != s0.in_dim || s.out_dim != s0.out_dim || s.layer[0][0].Kp != s0.layer[0][0].Kp || s.layer[0][2].Np != s0.layer[0][2].Np)
      return false;
  return true;
}

__host__ __device__ inline uint32_t t4_zs_stride(int Dv) { return ((uint32_t)(kTcRows * Dv * 4) + 127u) & ~127u; }   // bytes

inline bool tc4_make_plan(const ModelDims& md, const std::vector<StepDesc>& steps, TcPlan* p) {
  const int k0p = steps[0].layer[0][0].Kp, np3 = steps[0].layer[0][2].Np;
  auto al = [](uint32_t v) { return (v + 127u) & ~127u; };
  p->K0p = k0p; p->out_max = steps[0].out_dim;
  uint32_t o = 0;
  p->off_zs = o;   o = al(o + 2 * t4_zs_stride(md.Dv));         // z tile of chain X | chain Y
  p->off_a0 = o;   o = al(o + (k0p / 16) * 4096);               // A0: ONE buffer (a chain gathers its next pass after the other chain's layer-1 GEMMs)
  p->off_a1 = o;   o = al(o + 6 * kTcRows * 4);                 // per-row partial sums at a component's end
  p->off_sh = o;
  p->off_misc = o; o = al(o + kT2MiscBytes);
  p->off_bias = o; o = al(o + 2 * t2_bias_stride(md.h) * 4);    // b1 | b2 | b3 of chain X's | chain Y's current pass
  p->off_tab = o;  o = al(o + 6 * kEpPad * 16);                 // z1 tables [chain][pass parity], z2 tables [chain]
  p->off_w3 = o;   o = al(o + 2 * (uint32_t)np3 * 256u);         // last-layer weights of two pieces: <= 8 k-slabs of [np3 x 16] each
  p->off_ring = o;
  const uint32_t limit = 227 * 1024;
  if (o + 4 * kT2StageBytes > limit) return false;            // fewer than four 32 KB stages loses more to L2 -> SM latency than the schedule gains
  p->nst = std::min<int>(kT2MaxStages, (limit - o) / kT2StageBytes);
  p->smem_bytes = o + (size_t)p->nst * kT2StageBytes;
  p->tmem_cols = 512;
  return true;
}

// position of a chain in its pass sequence: work units blockIdx.x, + gridDim.x, ...; chain 0 walks the first half of a unit's
// components, chain 1 the second half; K steps per component
struct T4Pos { int u, c, k, cend; };
__device__ __forceinline__ void t4_pos_unit(const CouplingArgs& a, int chain, T4Pos& p) {
  const int half = a.comps_per_unit >> 1;
  p.c = a.c0 + (p.u % a.split) * a.comps_per_unit + chain * half;
  p.cend = p.c + half;
  p.k = 0;
}
__device__ __forceinline__ void t4_pos_next(const CouplingArgs& a, int chain, T4Pos& p) {
  if (++p.k == a.md.K) {
    p.k = 0;
    if (++p.c == p.cend) {
      p.u += (int)gridDim.x;
      if (p.u < a.num_units) t4_pos_unit(a, chain, p);
    }
  }
}

// tight geometry (coupling_tc2.cuh T2Geom for h = 512)
__device__ __forceinline__ constexpr int t4_cw(int j) { return (j & 1) ? 64 : 128; }
__device__ __forceinline__ constexpr int t4_ccol(int j) { return 192 * (j >> 1) + ((j & 1) ? 128 : 0); }
constexpr uint32_t kT4Slot0 = 256u, kT4Slot1 = 384u, kT4LaCol = 448u;

#define T4_CLK() (PROF ? clock64() : 0LL)
// event trace of ONE slot (kT4TraceSlot) of CTA 0: a.prof[190 + id] = clock64() (tools/tc4_profile.py prints it)
constexpr int kT4TraceSlot = 41;
#define T4_TRACE(id) do { if (PROF && a.prof != nullptr && blockIdx.x == 0 && s == kT4TraceSlot && lane == 0) a.prof[190 + (id)] = clock64(); } while (0)
// PROF = 1: per-role cycle counters of CTA 0 (gbnf_get_profile; tools/tc4_profile.py)
template <int TANH_MODE, int PROF = 0>
__global__ void __launch_bounds__(kT2Threads, 1) coupling_tc4_kernel(CouplingArgs a, TcPlan plan) {
  extern __shared__ __align__(1024) unsigned char smem[];
  asm volatile(".reg .pred t4_p_full;\n\t.reg .pred t4_p_sr;" ::);
  const ModelDims& md = a.md;
  const int D = md.D, Dv = md.Dv, K = md.K;
  constexpr int NQ = 4, NJ = 5, H = 512, hs = H >> 4;
  unsigned char* const zs_b = smem + plan.off_zs;
  unsigned char* const A0_b = smem + plan.off_a0;
  float* const part_s = reinterpret_cast<float*>(smem + plan.off_a1);
  float* const bias_s = reinterpret_cast<float*>(smem + plan.off_bias);
  float4* const tab_s = reinterpret_cast<float4*>(smem + plan.off_tab);
  Tc4Misc* const misc = reinterpret_cast<Tc4Misc*>(smem + plan.off_misc);
  unsigned char* const ring = smem + plan.off_ring;
  unsigned char* const w3buf = smem + plan.off_w3;
  const uint32_t zs_stride = t4_zs_stride(Dv);
  const uint32_t bstride = t2_bias_stride(H);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nst = plan.nst;
  // uniform step geometry (tc4_eligible)
  const int in_dim = __ldg(&a.steps[a.c0 * md.K].in_dim), out_dim = __ldg(&a.steps[a.c0 * md.K].out_dim);
  const int k0p = __ldg(&a.steps[a.c0 * md.K].layer[0][0].Kp), np3 = __ldg(&a.steps[a.c0 * md.K].layer[0][2].Np);
  const int k0s = k0p >> 4;
  const uint32_t w3_stride = (uint32_t)np3 * 256u;     // bytes per last-layer piece buffer
  // passes per chain of this CTA
  const int my_units = (a.num_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int npass = my_units * (a.comps_per_unit >> 1) * K;

  if (threadIdx.x == 0) {
    for (int i = 0; i < nst; ++i) { ptx::mbar_init(&misc->full[i], 1); ptx::mbar_init(&misc->empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&misc->a0r[i], 16); ptx::mbar_init(&misc->sr[i], 16); ptx::mbar_init(&misc->l2f[i], 1);
      ptx::mbar_init(&misc->w3full[i], 1); ptx::mbar_init(&misc->w3empty[i], 1);
    }
    for (int i = 0; i < 4; ++i) { ptx::mbar_init(&misc->a1r[i], 16); ptx::mbar_init(&misc->l1f[i], 1); }
    ptx::mbar_init(&misc->l3f, 1); ptx::mbar_init(&misc->l3d, 16); ptx::mbar_init(&misc->c2r, 16);
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
    uint32_t par = 0, ph_w3 = 0;
    int slot = 0;
    const long long p_t0 = T4_CLK();
    long long p_we = 0, p_w3 = 0, tq;
    auto push = [&](const __half* src, uint32_t bytes) {
      tq = T4_CLK();
      t2_wait(&misc->empty[slot], par ^ 1u, a.error_flag, 10, lane);
      p_we += T4_CLK() - tq;
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(&misc->full[slot], bytes);
        ptx::tma_bulk_g2s(ring + (size_t)slot * kT2StageBytes, src, bytes, &misc->full[slot]);
      }
      __syncwarp();
      if (++slot == nst) { slot = 0; par ^= 1u; }
    };
    T4Pos pX, pY;
    pX.u = pY.u = (int)blockIdx.x;
    t4_pos_unit(a, 0, pX); t4_pos_unit(a, 1, pY);
    // (one copy of the per-pass code for both chains: the kernel's instruction footprint matters, see the note at the epilogue)
#pragma unroll 1
    for (int s = 0; s < 2 * npass; ++s) {
      {
        const int ch = s & 1;
        T4Pos p = ch ? pY : pX;
        const StepDesc* sd = a.steps + (p.c * K + p.k);
        const __half* w1 = wb + __ldg(&sd->layer[0][0].w_off);
        const __half* w2 = wb + __ldg(&sd->layer[0][1].w_off);
        const __half* w3 = wb + __ldg(&sd->layer[0][2].w_off);
        auto stage_w3 = [&](int x) {
          const int b = x & 1;
          tq = T4_CLK();
          t2_wait(&misc->w3empty[b], ((ph_w3 >> b) & 1u) ^ 1u, a.error_flag, 11, lane);
          p_w3 += T4_CLK() - tq;
          ph_w3 ^= 1u << b;
          if (ptx::elect_one()) {
            const uint32_t bytes = (uint32_t)((t4_cw(x) >> 4) * np3) * 32u;
            ptx::mbar_arrive_expect_tx(&misc->w3full[b], bytes);
            ptx::tma_bulk_g2s(w3buf + (size_t)b * w3_stride, w3 + (size_t)(t4_ccol(x) >> 4) * np3 * 16, bytes, &misc->w3full[b]);
          }
          __syncwarp();
        };
        push(w1, (uint32_t)(NQ * k0s) * 4096u);
#pragma unroll
        for (int q = 0; q < NQ; ++q) push(w2 + (size_t)(8 * q) * 2048, 32768u);          // chunk 0, k-quarter q
#pragma unroll
        for (int j = 1; j < NJ; ++j) {
          stage_w3(j - 1);
          const __half* base = w2 + (size_t)t4_ccol(j) * hs * 16;
          if (t4_cw(j) == 128) {
#pragma unroll
            for (int y = 0; y < 4; ++y) push(base + (size_t)(8 * y) * 2048, 32768u);
          } else {
#pragma unroll
            for (int y = 0; y < 2; ++y) push(base + (size_t)(16 * y) * 1024, 32768u);
          }
        }
        stage_w3(NJ - 1);
        t4_pos_next(a, ch, p);
        if (ch) pY = p; else pX = p;
      }
    }
    if (PROF && a.prof != nullptr && blockIdx.x == 0 && lane == 0) { a.prof[16] = T4_CLK() - p_t0; a.prof[17] = p_we; a.prof[18] = p_w3; }
  } else if (warp == 1) {
    // ===================================== MMA issuer =======================================================
    uint32_t ph_sr = 0, ph_w3f = 0;
    int nslot = 0, slot = 0;
    uint32_t npar = 0;
    const uint64_t a0_desc = ptx::make_smem_desc(ptx::smem_u32(A0_b));
    const uint64_t ring_desc = ptx::make_smem_desc(ptx::smem_u32(ring));
    const uint64_t w3_desc = ptx::make_smem_desc(ptx::smem_u32(w3buf));
    const uint32_t idesc_l1 = ptx::make_idesc_f16(128, kT2Chunk);
    const uint32_t idesc_l2 = ptx::make_idesc_f16(128, kT2Piece);
    const uint32_t idesc_o = ptx::make_idesc_f16(128, np3);
    const uint32_t b3_step = (uint32_t)np3 * 2u;
    auto test_full = [&](uint64_t* bar, uint32_t par) {
      asm volatile("mbarrier.test_wait.parity.shared::cta.b64 t4_p_full, [%0], %1;" ::"r"(ptx::smem_u32(bar)), "r"(par) : "memory");
    };
    test_full(&misc->full[0], 0u);
    const long long m_t0 = T4_CLK();
    long long m_a0 = 0, m_full = 0, m_sr = 0, m_l3d = 0, m_a1 = 0, tq;
    auto acquire = [&]() -> uint64_t {
      slot = nslot;
      uint32_t full_ok;
      asm volatile("selp.u32 %0, 1, 0, t4_p_full;" : "=r"(full_ok));
      tq = T4_CLK();
      if (!full_ok) ptx::mbar_wait(&misc->full[slot], npar, a.error_flag, 21);
      m_full += T4_CLK() - tq;
      ptx::tc_fence_after();
      if (++nslot == nst) { nslot = 0; npar ^= 1u; }
      test_full(&misc->full[nslot], npar);
      return ring_desc + (uint64_t)((uint32_t)slot * (kT2StageBytes >> 4));
    };
    auto wait_epi = [&](uint64_t* bar, uint32_t par, int code) {
      ptx::mbar_wait(bar, par, a.error_flag, code);
      ptx::tc_fence_after();
    };
    uint32_t sr_pre = 0;
    // last layer, k-piece x held packed in slot x & 1 -> last-layer accumulator
    uint32_t n_l3d = 0;                       // completions of l3d consumed so far
    auto l3_piece = [&](int x, bool wait_drain) {
      const int sl = x & 1;
      const int w = t4_cw(x);
      if (wait_drain) {                       // piece 0 overwrites [448, 512): the other chain's transform must have read it
        tq = T4_CLK();
        ptx::mbar_wait(&misc->l3d, n_l3d & 1u, a.error_flag, 27);
        m_l3d += T4_CLK() - tq;
        ++n_l3d;
      }
      uint32_t sr_ok = 0;
      if (sr_pre) asm volatile("selp.u32 %0, 1, 0, t4_p_sr;" : "=r"(sr_ok));
      sr_pre = 0;
      tq = T4_CLK();
      if (!sr_ok) ptx::mbar_wait(&misc->sr[sl], (ph_sr >> sl) & 1u, a.error_flag, 23);
      ptx::tc_fence_after();
      ph_sr ^= 1u << sl;
      ptx::mbar_wait(&misc->w3full[sl], (ph_w3f >> sl) & 1u, a.error_flag, 24);
      m_sr += T4_CLK() - tq;
      ptx::tc_fence_after();
      ph_w3f ^= 1u << sl;
      const uint64_t bd = w3_desc + (uint64_t)((uint32_t)sl * (w3_stride >> 4));
      if (ptx::elect_one()) {
        const uint32_t at = tbase + (sl ? kT4Slot1 : kT4Slot0), d = tbase + kT4LaCol;
        const uint32_t astep = (w == 128) ? 8u : 16u;
        const int nsl = w >> 4;
        for (int i = 0; i < nsl; ++i)
          ptx::umma_f16_ts(d, at + astep * i, bd + (uint64_t)((uint32_t)i * b3_step), idesc_o, (x > 0 || i > 0) ? 1u : 0u);
        ptx::umma_commit(&misc->w3empty[sl]);
        if (x == NJ - 1) ptx::umma_commit(&misc->l3f);
      }
      __syncwarp();
    };
#pragma unroll 1
    for (int s = 0; s < 2 * npass; ++s) {
      {
        const int ch = s & 1, n = s >> 1;
        // ---- layer-1 chunk 0 of this pass, then the LAST last-layer piece of the previous pass (other chain) ----
        const uint64_t l1_desc = acquire();
        const int l1_slot = slot;
        tq = T4_CLK();
        wait_epi(&misc->a0r[ch], (uint32_t)n & 1u, 20);
        m_a0 += T4_CLK() - tq;
        auto l1_chunk = [&](int x) {
          if (ptx::elect_one()) {
            const uint64_t bq = l1_desc + (uint64_t)(x * k0s * 256);
            if (x < 3) {
              const uint32_t d = tbase + (x == 1 ? kT4Slot0 : 128u);
              for (int i = 0; i < k0s; ++i)
                ptx::umma_f16(d, a0_desc + (uint64_t)(i * 256), bq + (uint64_t)(i * 256), idesc_l1, i > 0 ? 1u : 0u);
            } else {                          // chunk 3: columns 0..63 -> slot 1 [384, 448), columns 64..127 -> [192, 256)
              for (int i = 0; i < k0s; ++i) {
                ptx::umma_f16(tbase + kT4Slot1, a0_desc + (uint64_t)(i * 256), bq + (uint64_t)(i * 256), idesc_l2, i > 0 ? 1u : 0u);
                ptx::umma_f16(tbase + 192u, a0_desc + (uint64_t)(i * 256), bq + (uint64_t)(i * 256 + 128), idesc_l2, i > 0 ? 1u : 0u);
              }
            }
            ptx::umma_commit(&misc->l1f[x]);
            if (x == NQ - 1) ptx::umma_commit(&misc->empty[l1_slot]);
          }
          __syncwarp();
        };
        auto l2c0_part = [&](int q) {
          const uint64_t bd = acquire();
          const int cur = slot;
          if (ptx::elect_one()) {
            const uint32_t d = tbase + kT4Slot0, at = tbase + (uint32_t)q * 64u;
            ptx::umma_f16_ts(d, at, bd, idesc_l1, q > 0 ? 1u : 0u);
#pragma unroll
            for (int i = 1; i < 8; ++i) ptx::umma_f16_ts(d, at + 8u * i, bd + (uint64_t)(i * 256), idesc_l1, 1u);
            ptx::umma_commit(&misc->empty[cur]);
            if (q == NQ - 1) ptx::umma_commit(&misc->l2f[0]);
          }
          __syncwarp();
        };
        auto wait_a1 = [&](int q) {
          tq = T4_CLK();
          wait_epi(&misc->a1r[q], (uint32_t)ch, 22);             // one completion per pass: parity = s & 1
          m_a1 += T4_CLK() - tq;
        };
        // Layer-1 accumulators: chunk 0 -> [128, 256) (the dead upper half of the other chain's A1), chunk 1 -> slot 0 (free once
        // the other chain's last piece has been multiplied), chunk 2 -> [128, 256) again, chunk 3 -> slot 1 [384, 448) + [192, 256)
        // (the upper half of chunk 2's accumulator, packed in place): the other chain's last-layer accumulator [448, 512) stays
        // untouched until its transform has read it.  Layer-2 chunk 0 starts behind layer-1 chunk 1 and still ends one
        // k-quarter after the last layer-1 epilogue.
        T4_TRACE(0);
        l1_chunk(0);
        T4_TRACE(1);
        if (s > 0) l3_piece(NJ - 1, false);
        T4_TRACE(2);
        l1_chunk(1);
        wait_a1(0);
        T4_TRACE(3);
        l1_chunk(2);
        wait_a1(1);
        T4_TRACE(4);
        l2c0_part(0);
        tq = T4_CLK();
        wait_epi(&misc->c2r, (uint32_t)ch, 28);   // chunk 2's accumulator has been read (well before its activation is done)
        m_a1 += T4_CLK() - tq;
        T4_TRACE(5);
        l1_chunk(3);                           // before the next parts: the in-order pipe would park it behind them
        l2c0_part(1);
        wait_a1(2);
        l2c0_part(2);
        T4_TRACE(6);
        wait_a1(3);
        T4_TRACE(7);
        l2c0_part(3);
        T4_TRACE(8);
        // ---- layer-2 chunks 1..4 with the last-layer pieces 0..3 ----
#pragma unroll
        for (int j = 1; j < NJ; ++j) {
          T4_TRACE(10 + 3 * (j - 1));            // chunk j: before the previous piece
          if (j >= 2) l3_piece(j - 2, j == 2 && s > 0);
          T4_TRACE(11 + 3 * (j - 1));            // piece issued
          const int w = t4_cw(j);
          const int parts = (w == 128) ? 4 : 2;
#pragma unroll
          for (int y = 0; y < parts; ++y) {
            const uint64_t bd = acquire();
            const int cur = slot;
            if (y == parts - 1) {          // the op after this chunk is last-layer piece j - 1: test its barrier under these MMAs
              const int sn = (j - 1) & 1;
              asm volatile("mbarrier.test_wait.parity.shared::cta.b64 t4_p_sr, [%0], %1;" ::"r"(ptx::smem_u32(&misc->sr[sn])),
                           "r"((ph_sr >> sn) & 1u) : "memory");
              sr_pre = 1;
            }
            if (ptx::elect_one()) {
              const uint32_t d = tbase + ((j & 1) ? kT4Slot1 : kT4Slot0);
              if (w == 128) {
                const uint32_t at = tbase + (uint32_t)y * 64u;
                ptx::umma_f16_ts(d, at, bd, idesc_l1, y > 0 ? 1u : 0u);
#pragma unroll
                for (int i = 1; i < 8; ++i) ptx::umma_f16_ts(d, at + 8u * i, bd + (uint64_t)(i * 256), idesc_l1, 1u);
              } else {
#pragma unroll
                for (int qq = 0; qq < 2; ++qq) {
                  const uint32_t at = tbase + (uint32_t)(2 * y + qq) * 64u;
                  const uint64_t bq = bd + (uint64_t)(qq * 1024);
                  ptx::umma_f16_ts(d, at, bq, idesc_l2, (2 * y + qq) > 0 ? 1u : 0u);
#pragma unroll
                  for (int i = 1; i < 8; ++i) ptx::umma_f16_ts(d, at + 8u * i, bq + (uint64_t)(i * 128), idesc_l2, 1u);
                }
              }
              ptx::umma_commit(&misc->empty[cur]);
              if (y == parts - 1) ptx::umma_commit(&misc->l2f[j & 1]);
            }
            __syncwarp();
          }
          T4_TRACE(12 + 3 * (j - 1));            // chunk j issued
        }
        T4_TRACE(22);
        l3_piece(NJ - 2, false);
        T4_TRACE(23);
      }
    }
    if (npass > 0) l3_piece(NJ - 1, false);
    if (PROF && a.prof != nullptr && lane == 0 && blockIdx.x < 256)      // every CTA: total (low word) | ring wait (high word)
      a.prof[32 + blockIdx.x] = ((T4_CLK() - m_t0) & 0xffffffffLL) | ((m_full + m_a0 + m_sr + m_l3d + m_a1) << 32);   // total | all waits
    if (PROF && a.prof != nullptr && blockIdx.x == 0 && lane == 0) {
      a.prof[0] = T4_CLK() - m_t0; a.prof[1] = m_a0; a.prof[2] = m_full; a.prof[3] = m_sr; a.prof[4] = m_l3d; a.prof[5] = m_a1; a.prof[6] = 2 * npass;
    }
  } else {
    // ===================================== epilogue / elementwise warps =====================================
    const int et = threadIdx.x - 64;
    const int warp_e = et >> 5;
    const int quad = warp & 3;
    const int g = warp_e >> 2;
    const int row = quad * 32 + lane;
    const uint32_t lane_base = tbase + ((uint32_t)(quad * 32) << 16);
    const int dq = (D + 3) >> 2;
    const int h0col = min(D, g * dq), h1col = min(D, (g + 1) * dq);
    uint32_t ph_l2f = 0;
    float lsumX = 0.f, lsumY = 0.f;
    uint32_t ngX = 0, ngY = 0;               // passes of the chain gathered so far
    T4Pos pX, pY;                            // the pass of the chain that was gathered last (= the one it finishes next)
    pX.u = pY.u = (int)blockIdx.x;
    t4_pos_unit(a, 0, pX); t4_pos_unit(a, 1, pY);
    const int c0 = g * 16;                   // this thread's 16 columns of the last-layer accumulator
    const long long e_t0 = T4_CLK();
    long long e_l1f = 0, e_l2f = 0, e_l3f = 0, e_fin = 0, e_bar = 0, e_e1 = 0, e_e2 = 0, e_tr = 0, e_ga = 0, tq;

    // ---- x rows of a component's start -> z tile (this thread's quarter of its own row) ----
    auto load_x = [&](const T4Pos& p, float* zrow) {
      const long long gr = (long long)(p.u / a.split) * kTcRows + row;
      float v[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = (h0col + i < h1col && gr < a.B) ? __ldg(a.x + gr * D + h0col + i) : 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) if (h0col + i < h1col) zrow[h0col + i] = v[i];
      if (g == 0) for (int pc = D; pc < Dv; ++pc) zrow[pc] = 0.f;
    };
    // ---- asynchronous staging for pass p of a chain (just gathered, index ng): its biases and z2 table; the z1 table of the
    //      chain's pass after it ----
    // (the descriptor loads are issued by stage_offsets() before the gather so that their L2 round trip hides under it)
    auto stage_offsets = [&](int chain, const T4Pos& p, uint32_t ng, long long& off) {
      off = -1;
      const StepDesc* sd = a.steps + (p.c * K + p.k);
      if (et < 272) off = __ldg(&sd->layer[0][0].b_off);
      else if (et < 272 + kEpPad) off = __ldg(&sd->ep_off);
      else if (et < 272 + 2 * kEpPad && (int)ng + 1 < npass) {
        T4Pos p2 = p;
        t4_pos_next(a, chain, p2);
        off = __ldg(&a.steps[p2.c * K + p2.k].ep_off);
      }
    };
    auto stage = [&](int chain, uint32_t ng, long long off) {
      if (et < 272) {
        if (et < ((2 * H + np3) >> 2)) ptx::cp_async16(bias_s + chain * bstride + 4 * et, a.fblob + off + 4 * et);
      } else if (et < 272 + kEpPad) {
        const int i = et - 272;
        ptx::cp_async16(tab_s + (4 + chain) * kEpPad + i, reinterpret_cast<const float4*>(a.fblob + off) + kEpPad + i);
      } else if (et < 272 + 2 * kEpPad) {
        if (off >= 0) {
          const int i = et - 272 - kEpPad;
          ptx::cp_async16(tab_s + (2 * chain + ((ng + 1) & 1u)) * kEpPad + i, reinterpret_cast<const float4*>(a.fblob + off) + i);
        }
      }
    };
    // ---- layer-1 chunk q of the starting pass: accumulator -> bias + tanh -> fp16 pairs -> A1 quarter q ----
    auto e1_chunk = [&](int q, const float* bias_c, uint32_t par) {
      tq = T4_CLK();
      t2_wait(&misc->l1f[q], par, a.error_flag, 30, lane);
      e_l1f += T4_CLK() - tq;
      tq = T4_CLK();
      ptx::tc_fence_after();
      // accumulator columns of this thread's 32 values: chunks 0, 2 at [128, 256), chunk 1 in slot 0, chunk 3 split (see the MMA warp)
      const uint32_t col = (q == 3) ? (g < 2 ? kT4Slot1 + (uint32_t)g * 32u : 192u + (uint32_t)(g - 2) * 32u)
                                    : ((q == 1) ? kT4Slot0 : 128u) + (uint32_t)g * 32u;
      uint32_t pk[16];
      {
        uint32_t r[32];
        ptx::tmem_ld32(lane_base + col, r);
        ptx::tmem_ld_wait();
        if (q == 2) {                         // chunk 3's second half may now be multiplied into [192, 256): its layer-1 GEMM then
          ptx::tc_fence_before();             // runs under this chunk's activation instead of after it
          t2_warp_arrive(&misc->c2r, lane);
        }
        t2_act_pack<1, TANH_MODE>(r, bias_c + g * 32 + q * kT2Chunk, pk, a.error_flag);
      }
      if (q >= 2) t2_quad_bar(quad);         // chunk 2 and half of chunk 3 accumulate inside the A1 region they are packed into
      ptx::tmem_st16(lane_base + (uint32_t)q * 64u + (uint32_t)g * 16u, pk);
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      t2_warp_arrive(&misc->a1r[q], lane);
      e_e1 += T4_CLK() - tq;
    };
    // ---- layer-2 chunk j: accumulator -> bias + tanh -> fp16 pairs packed in place (k-piece j of the last layer's A) ----
    auto e2_chunk = [&](int j, const float* bias_c) {
      const int sl = j & 1;
      tq = T4_CLK();
      t2_wait(&misc->l2f[sl], (ph_l2f >> sl) & 1u, a.error_flag, 31, lane);
      e_l2f += T4_CLK() - tq;
      tq = T4_CLK();
      ph_l2f ^= 1u << sl;
      ptx::tc_fence_after();
      const uint32_t sc = lane_base + (sl ? kT4Slot1 : kT4Slot0);
      const float* bj = bias_c + H + 192 * (j >> 1) + (sl ? 128 : 0);
      if (sl == 0) {
        uint32_t pk[16];
        {
          uint32_t r[32];
          ptx::tmem_ld32(sc + (uint32_t)g * 32u, r);
          ptx::tmem_ld_wait();
          t2_act_pack<1, TANH_MODE>(r, bj + g * 32, pk, a.error_flag);
        }
        t2_quad_bar(quad);
        ptx::tmem_st16(sc + (uint32_t)g * 16u, pk);
      } else {
        uint32_t pk[8];
        {
          uint32_t r[16];
          ptx::tmem_ld16(sc + (uint32_t)g * 16u, r);
          ptx::tmem_ld_wait();
          t2_act_pack<1, TANH_MODE>(r, bj + g * 16, pk, a.error_flag);
        }
        ptx::tmem_st8(sc + (uint32_t)g * 16u, pk);
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      t2_warp_arrive(&misc->sr[sl], lane);
      e_e2 += T4_CLK() - tq;
    };
    // ---- affine coupling transform of the finishing pass (glow.py:333-338); releases the last-layer accumulator ----
    auto transform = [&](float* zrow, const float4* tab2, const float* bias3, float& lsum, uint32_t par) {
      tq = T4_CLK();
      t2_wait(&misc->l3f, par, a.error_flag, 32, lane);
      e_l3f += T4_CLK() - tq;
      ptx::tc_fence_after();
      uint32_t r[16];
      if (c0 < np3) {
        ptx::tmem_ld16(lane_base + kT4LaCol + (uint32_t)c0, r);
        ptx::tmem_ld_wait();
      }
      ptx::tc_fence_before();
      t2_warp_arrive(&misc->l3d, lane);      // [448, 512) may take the other chain's last layer
      if (c0 < np3) {
        const float2* bias2 = reinterpret_cast<const float2*>(bias3);
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
          const float s = __fdividef(1.0f, 1.0f + __expf(-(raw + 2.0f)));
          const float zn = (z[jj] + t[jj].x) * t[jj].y + t[jj].z;
          z[jj] = (zn + shift) * s;
          lsum += (j < out_dim) ? __logf(s) : 0.f;
        }
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) if (g * 8 + jj < out_dim) zrow[__float_as_int(t[jj].w)] = z[jj];
      }
    };
    // ---- end of a component: log q for this row; chain 1 at the end of a unit: the tile's logsumexp ----
    auto comp_end = [&](int chain, const T4Pos& p, const float* zrow, float lsum, float* part) {
      const int tile = p.u / a.split;
      const long long gr = (long long)tile * kTcRows + row;
      const int c = p.c;
      const float2 cconst = __ldg(reinterpret_cast<const float2*>(a.fblob + a.cc_off) + c);
      const long long base_off = (md.base == GBNF_BASE_STD_NORMAL) ? 0LL : __ldg(&a.comps[c].base_off);
      t2_component_logq(a, zrow, lsum, part, row, g, quad, h0col, h1col, Dv, base_off, cconst.x, cconst.y, misc->coef, c, tile, true);
      if (chain == 1 && c + 1 == p.cend && a.G_ll != nullptr && !a.terms_only) t2_tile_logsumexp(a, tile, gr, g, et, &misc->last_flag);
    };
    // ---- everything a chain does between two of its passes: transform of the finishing pass, (end of component), gather of
    //      the next pass, staging ----
    auto finish_a = [&](int chain, uint32_t par) {
      float* zrow = reinterpret_cast<float*>(zs_b + chain * zs_stride) + row * Dv;
      const long long tf = T4_CLK();
      float ls = chain ? lsumY : lsumX;
      transform(zrow, tab_s + (4 + chain) * kEpPad, bias_s + chain * bstride + 2 * H, ls, par);
      if (chain) lsumY = ls; else lsumX = ls;
      e_tr += T4_CLK() - tf;
      t2_epi_bar();                          // z2 visible to the row's other threads; this pass's b3 / z2 table are dead
      e_fin += T4_CLK() - tf;
    };
    // start = true: the chain's very first pass (nothing to finish, position already at it)
    auto finish_b = [&](int chain, bool start) {
      float* zrow = reinterpret_cast<float*>(zs_b + chain * zs_stride) + row * Dv;
      const long long tf = T4_CLK();
      T4Pos p = chain ? pY : pX;
      uint32_t ng = chain ? ngY : ngX;
      if (!start && p.k == K - 1) {
        comp_end(chain, p, zrow, chain ? lsumY : lsumX, part_s);
        if (chain) lsumY = 0.f; else lsumX = 0.f;
      }
      if ((int)ng < npass) {
        if (!start) t4_pos_next(a, chain, p);
        long long soff;
        stage_offsets(chain, p, ng, soff);
        if (p.k == 0) {                      // a component starts from x (every thread loads the columns it owns)
          load_x(p, zrow);
          t2_quad_bar(quad);
        }
        const long long tg = T4_CLK();
        t2_gather_z1(zrow, tab_s + (2 * chain + (ng & 1u)) * kEpPad, in_dim, k0p >> 3, g, row, A0_b, a.error_flag);
        ptx::fence_proxy_async_smem();
        ptx::tc_fence_before();
        t2_warp_arrive(&misc->a0r[chain], lane);
        e_ga += T4_CLK() - tg;
        stage(chain, ng, soff);
        ++ng;
      }
      if (chain) { pY = p; ngY = ng; } else { pX = p; ngX = ng; }
      e_fin += T4_CLK() - tf;
    };

    // ---- z1 tables of both chains' first passes ----
    if (npass > 0) {
      if (et < 2 * kEpPad) {
        const int chain = et >> 6, i = et & (kEpPad - 1);
        const T4Pos& p = chain ? pY : pX;
        const StepDesc* sd = a.steps + (p.c * K + p.k);
        ptx::cp_async16(tab_s + (2 * chain) * kEpPad + i, reinterpret_cast<const float4*>(a.fblob + __ldg(&sd->ep_off)) + i);
      }
      ptx::cp_async_wait_all();
      t2_epi_bar();
    }
    // ---- the slot loop.  ONE copy of every block for both chains, runtime chunk indices and no peeled prologue / epilogue:
    //      the fully unrolled form of this kernel was 300 KB of SASS, and at full occupancy its instruction fetches contended
    //      inside every GPC (per-CTA MMA issue time 2.07 M cycles on a 12-SM GPC vs 2.6 - 3.0 M on 18 / 20-SM GPCs).
    //      Slot -1 is chain 0's first gather, slot 0 also does chain 1's first gather (one A0 buffer), slot 2 npass only finishes
    //      chain 1's last pass. ----
    const int nslots = npass > 0 ? 2 * npass : -1;
#pragma unroll 1
    for (int s = -1; s <= nslots; ++s) {
      const bool real = s >= 0 && s < nslots;
      const int ch = s & 1;                                  // chain that starts a pass in this slot
      const int fin = ch ^ 1;                                // chain whose pass (slot s - 1) finishes / whose next pass is gathered
      const float* biasB = bias_s + ch * bstride;
      const float* biasA = bias_s + fin * bstride;
#pragma unroll 1
      for (int t = 0; t < 5; ++t) {
        const int j = (t == 0) ? NJ - 1 : t - 1;
        if (warp_e == 0) T4_TRACE(40 + 8 * t);
        if (t == 0 ? (s > 0) : real) e2_chunk(j, t == 0 ? biasA : biasB);
        if (warp_e == 0) T4_TRACE(41 + 8 * t);
        if (t == 0 && real) {
#pragma unroll 1
          for (int q = 0; q < NQ; ++q) { e1_chunk(q, biasB, (uint32_t)ch); if (warp_e == 0) T4_TRACE(44 + q); }
        }
        // Placement (event trace, tools/tc4_profile.py): the slot's first half (A's last chunk, B's layer-1 phase, B's chunk 0) is
        // epilogue bound, its second half (B's chunks 2 .. 4) tensor-pipe bound with ~3 k cycles of epilogue slack.  A's transform
        // follows B's chunk 0 directly (its tensor-memory read releases [448, 512) just before B's piece 0 wants it); A's
        // bookkeeping / x reload / gather / staging block (3 k) goes behind B's chunk 2, where it delays no packed piece.
        if (t == 1 && s > 0) finish_a(fin, (uint32_t)(s - 1) & 1u);
        if (t == 3) finish_b(fin, s <= 0);
        if (warp_e == 0) T4_TRACE(42 + 8 * t);
      }
      tq = T4_CLK();
      ptx::cp_async_wait_all();
      t2_epi_bar();                          // staged biases / tables visible before the next slot uses them
      e_bar += T4_CLK() - tq;
    }
    if (PROF && a.prof != nullptr && blockIdx.x == 0 && et == 0) {
      a.prof[8] = T4_CLK() - e_t0; a.prof[9] = e_l1f; a.prof[10] = e_l2f; a.prof[11] = e_l3f; a.prof[12] = e_fin; a.prof[13] = e_bar;
      a.prof[14] = e_e1; a.prof[15] = e_e2; a.prof[19] = e_tr; a.prof[20] = e_ga;
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

#undef T4_CLK
#undef T4_TRACE

inline cudaError_t tc4_configure() {
  cudaError_t e = cudaFuncSetAttribute(coupling_tc4_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc4_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc4_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc4_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  return e;
}

inline int tc4_launch(const CouplingArgs& a, const TcPlan& p, int grid, cudaStream_t st, int prof) {
  if (prof) {
    if (p.tanh_mode == 0) coupling_tc4_kernel<0, 1><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p);
    else                  coupling_tc4_kernel<1, 1><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p);
  } else {
    if (p.tanh_mode == 0) coupling_tc4_kernel<0, 0><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p);
    else                  coupling_tc4_kernel<1, 0><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p);
  }
  return 0;
}

}  // namespace gbnf
