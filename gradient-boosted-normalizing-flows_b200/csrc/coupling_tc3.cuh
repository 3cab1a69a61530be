// tcgen05 / TMEM / bulk-TMA coupling-stack kernel for hidden width 1024 (GBNF_GEMM_F16_TC*, Glow components,
// coupling_network_depth == 1): BASELINE configuration 5 (BSDS300 shape, models/glow.py:300-308 block
// Net(D//2 -> 1024 -> 1024 -> 2 (D - D//2)), models/layers.py:230-243).
//
// Why a CTA PAIR.  The layer-2 A operand of a 128-row tile (128 x 1024 fp16) is 256 KB = ALL of one SM's tensor memory, so
// the single-CTA layout of coupling_tc2.cuh (A1 + accumulators resident in TMEM) cannot hold it, and neither can shared memory
// next to a weight ring.  (Half tiles do not help: an M = 64 accumulator still spans all four lane quadrants, and a
// cta_group::2 M = 128 MMA wants its TMEM A operand duplicated across the lane halves -- tools/tc_probe7.cu and the CuTe
// tmem_frg layouts.)  Here a 2-CTA thread-block cluster owns the tile and SPLITS THE HIDDEN UNITS:
//
//   CTA p (p = cluster rank) computes hidden units [512 p, 512 p + 512) of layer 1 -> its K-half of layer 2's A operand
//   (A1_p, 256 TMEM columns), multiplies it with ITS K-half of W2 for ALL 1024 layer-2 outputs (partial sums), and owns the
//   layer-2 output chunks J with (J & 1) == p (128 columns each): partial sums of the chunks it does not own are shipped to
//   the peer's shared memory (st.shared::cluster + remote mbarrier arrive), the owner adds them to its own accumulator,
//   applies bias + tanh, packs fp16 pairs in place (= a K-piece of ITS half of the last layer's A operand) and accumulates
//   its partial last-layer product.  The two partial last-layer products (128 x <= 64 fp32) are exchanged the same way, both
//   CTAs apply the (identical) coupling transform to their own copy of the resident z tile, rank 0 writes the results.
//
//   TMEM (512 columns per CTA):  A1_p [0, 256) | slot A [256, 384): own layer-2 chunk (128 fp32 columns; its fp16 pairs are
//   packed in place into [256, 320), the vacated upper half [320, 384) then receives that piece's last-layer product, which
//   the epilogue adds into registers) | slots B0 [384, 448) and B1 [448, 512): the two shipped halves of the peer's chunk,
//   double buffered so that the second half does not wait for the first one's epilogue.  Layer-1 accumulators use slot A and
//   B0 + B1 before layer 2 starts.
//   weights: one linear stream per (step, CTA) in the order the MMA warp consumes it, cut into 16 KB ring stages
//   (pack_weight_tc3_kernel): W1 half | for chunk pair m = 0..3: two shipped halves [32 k-slabs][64 x 16] of chunk
//   2 m + 1 - p, then the own chunk 2 m + p [32 k-slabs][128 x 16] | last-layer pieces [8 k-slabs][Np3 x 16] per own chunk.
//
// Warp roles as in coupling_tc2.cuh: warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..17 = epilogue (four threads per row).
//
// RealNVP (RNVP = 1): a step is TWO coupling passes on the same z1, one per network, each with the schedule, exchange and weight
// stream of a Glow step (the image is laid out per (step, net, layer)).  The pass order needs no buffer for the shift (shared
// memory is nearly exhausted): forward s then t (z2 = BN(z2) * exp(s), then z2 += t), inverse t then s (z2 -= t, then
// z2 = BN^-1(z2 * exp(-s))).  A0 aliases the staging buffer, so the second pass gathers z1 again; only the pass of the s network
// applies the BatchNorm tables (t3_net).  The per-pass code is one copy with the network as a runtime index.
#pragma once
#include "coupling_tc2.cuh"

namespace gbnf {

constexpr int kT3Threads = 576;
constexpr int kT3EpiThreads = 512;
constexpr int kT3H = 1024;                   // hidden width this kernel is built for
constexpr int kT3HH = 512;                   // hidden units (= layer-2 K range) per CTA
constexpr int kT3MaxStages = 8;
constexpr uint32_t kT3StageBytes = 16384;    // 4 k-slabs of [128 x 16] or 8 k-slabs of [64 x 16]
constexpr uint32_t kT3XBytes = 65536;        // exchange buffer: 128 rows x 128 columns fp32, written by the peer CTA
constexpr int kT3BiasFloats = 512 + 512 + 64; // b1 (own half) | b2 (own chunks) | b3
// TMEM columns
constexpr uint32_t kT3SlotA = 256, kT3SlotB0 = 384, kT3SlotB1 = 448, kT3L3Tmp = 320;

struct Tc3Misc {
  uint64_t full[kT3MaxStages];
  uint64_t empty[kT3MaxStages];
  uint64_t a0r;       // epilogue -> MMA : A0 written, TMEM of the previous pass drained                 (16 arrivals)
  uint64_t a1r[4];    // epilogue -> MMA : A1 k-quarter q packed, its layer-1 accumulator drained        (16 arrivals)
  uint64_t l1f[4];    // MMA -> epilogue : layer-1 chunk q accumulated                                   (commit)
  uint64_t l2own;     // MMA -> epilogue : own layer-2 chunk accumulated in slot A                       (commit)
  uint64_t l2ship[2]; // MMA -> epilogue : shipped half chunk y accumulated in slot B y                  (commit)
  uint64_t sbr[2];    // epilogue -> MMA : slot B y read out                                             (16 arrivals)
  uint64_t l3r;       // epilogue -> MMA : last-layer piece product read out of slot A's upper half      (16 arrivals)
  uint64_t sr;        // epilogue -> MMA : A2 piece packed in slot A                                     (16 arrivals)
  uint64_t l3f;       // MMA -> epilogue : last-layer product of ONE own chunk's piece complete          (commit)
  uint64_t xfull;     // PEER epilogue -> epilogue : both halves of a chunk's partial sums are in my exchange buffer (armed by me with expect_tx; the peer's two bulk copies complete it)
  uint64_t x3full;    // PEER epilogue -> epilogue : the peer's partial last-layer product is in my exchange buffer (armed by me; one bulk copy of the peer completes it)
  uint64_t xfree;     // PEER epilogue -> epilogue : the peer has consumed what I last wrote into ITS exchange buffer (16 remote arrivals, relaxed)
  uint32_t tmem_base;
  uint32_t last_flag;
  int meta[2][8];     // per step (double buffered): in_dim, out_dim, Kp of layer 1, Np of the last layer
  float coef[kMaxComponents];
};
constexpr uint32_t kT3MiscBytes = 1536;
static_assert(sizeof(Tc3Misc) <= kT3MiscBytes, "misc region too small");

inline bool tc3_eligible(const ModelDims& md, const std::vector<StepDesc>& steps) {
  if (md.nlayers != 3 || md.h != kT3H || md.D > kTcMaxD) return false;
  if (md.kind == GBNF_KIND_GLOW ? (md.nnets != 1 || md.act == GBNF_ACT_MIXED) : md.nnets != 2) return false;
  for (const StepDesc& s : steps)
    for (int n = 0; n < md.nnets; ++n)
      if (s.layer[n][0].Kp > 32 || s.layer[n][2].Np > 64) return false;
  return true;
}

inline bool tc3_make_plan(const ModelDims& md, const std::vector<StepDesc>& steps, TcPlan* p) {
  int k0p = 16, out_max = 1;
  for (const StepDesc& s : steps) { k0p = std::max(k0p, s.layer[0][0].Kp); out_max = std::max(out_max, s.out_dim); }
  auto al = [](uint32_t v) { return (v + 127u) & ~127u; };
  p->K0p = k0p; p->out_max = out_max;
  uint32_t o = 0;
  p->off_zs = o;   o = al(o + kTcRows * md.Dv * 4);
  p->off_a1 = o;   o = al(o + kT3XBytes);                 // here: the exchange buffer the PEER writes
  p->off_sh = o;                                          // here: staging buffer of one shipped half chunk (source of the bulk copy)
  p->off_a0 = o;   o = al(o + kT3XBytes / 2);             // A0 (<= 8 KB, live from the gather to the last layer-1 MMA) and the per-row
                                                          // partial sums at the end of a component ALIAS the staging buffer (live during
                                                          // layer 2 and the exchange of the partial last-layer products)
  p->off_misc = o; o = al(o + kT3MiscBytes);
  p->off_bias = o; o = al(o + 2 * kT3BiasFloats * 4);
  p->off_tab = o;  o = al(o + 2 * 2 * kEpPad * 16);
  p->off_w3 = o;
  p->off_ring = o;
  const uint32_t limit = 227 * 1024;
  p->nst = std::min<int>(kT3MaxStages, (limit - o) / kT3StageBytes);
  p->smem_bytes = o + (size_t)p->nst * kT3StageBytes;
  p->tmem_cols = 512;
  return p->nst >= 4;
}

// ---- the fixed per-pass op order of CTA `p`, walked identically by its producer, MMA issuer and epilogue ----------------
//   OWN  (J)      : layer-2 chunk J (128 columns, (J & 1) == p) -> slot A; 8 ring stages
//   SHIP (J, hh)  : half hh of chunk J (64 columns, owned by the peer) -> slot B; 4 ring stages
//   L3   (m)      : last-layer piece of own chunk number m (J = 2 m + p), issued one op group later so that the epilogue has
//                   had time to pack it; 1 ring stage
enum { T3_OP_OWN = 0, T3_OP_SHIP, T3_OP_L3 };
// SHIP FIRST: in chunk pair m both CTAs first produce what the PEER is waiting for (the shipped chunk 2 m + 1 - p), then their
// own chunk 2 m + p, whose epilogue (peer's partial sums + tanh + pack) runs while the MMA warp is already busy with the next
// pair's shipped halves; the own chunk's last-layer piece follows those.  (Own-first order chained the two CTAs: own(J) waited
// for the peer's ship(J), which the peer only started after ITS own(J - 1), ... -- 8 serial hops per pass, measured 99 k cycles.)
template <class F>
__device__ __forceinline__ void t3_schedule(int p, F&& f) {
  // NOT unrolled: one copy of the per-pair code.  The fully unrolled kernel was 308 KB of SASS and lost a quarter of its
  // throughput to instruction fetch at full occupancy (DESIGN 4.1f).
#pragma unroll 1
  for (int m = 0; m < 4; ++m) {
    f(T3_OP_SHIP, 2 * m + 1 - p, 0);
    f(T3_OP_SHIP, 2 * m + 1 - p, 1);
    if (m > 0) f(T3_OP_L3, m - 1, 0);
    f(T3_OP_OWN, 2 * m + p, 0);
  }
  f(T3_OP_L3, 3, 0);
}

// Network of pass i (0, 1) of a step: Glow has one pass (net 0); RealNVP runs net 1 (s) first forward, net 0 (t) first inverse.
template <int RNVP, int INV>
__device__ __forceinline__ int t3_net(int i) { return RNVP ? (INV ? i : 1 - i) : 0; }

template <int ACT, int TANH_MODE>
__device__ __forceinline__ void t3_act_pack32_add(const uint32_t (&r)[32], const float4* __restrict__ xb, const float* __restrict__ bias,
                                                  uint32_t* p, int* status) {
  // own accumulator + the peer's partial sums (exchange buffer, float4 (c4 * 128 + row)) + bias -> activation -> fp16 pairs
  float v[32];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 o = xb[q * kTcRows];
    const float4 b = *reinterpret_cast<const float4*>(bias + 4 * q);
    v[4 * q + 0] = (__uint_as_float(r[4 * q + 0]) + o.x) + b.x;
    v[4 * q + 1] = (__uint_as_float(r[4 * q + 1]) + o.y) + b.y;
    v[4 * q + 2] = (__uint_as_float(r[4 * q + 2]) + o.z) + b.z;
    v[4 * q + 3] = (__uint_as_float(r[4 * q + 3]) + o.w) + b.w;
  }
  if (ACT == 2) {
    float mx = 0.f;
#pragma unroll
    for (int q = 0; q < 32; ++q) mx = fmax_nan(mx, v[q]);
    if (!(mx <= 65504.f)) *reinterpret_cast<volatile int*>(status + 2) = 1;
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    tc_act4<ACT, TANH_MODE>(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    p[2 * q] = pack_half2(v[4 * q], v[4 * q + 1]);
    p[2 * q + 1] = pack_half2(v[4 * q + 2], v[4 * q + 3]);
  }
}

// PROF = 1: per-role cycle counters of CTA 0 (rank 0 of pair 0) in a.prof (gbnf_get_profile): [0] MMA warp total, [1] wait ring,
// [2] wait a0r + a1r, [3] wait slot B, [4] wait packed piece, [5] passes; [8] epilogue (thread 0) total, [9] wait l1f, [10] wait l2own,
// [11] wait xfull, [12] wait l2ship, [13] wait xfree, [14] wait l3f, [15] wait x3full, [19] gather, [20] layer-1 epilogues,
// [21] own epilogues, [22] ship epilogues, [23] transform + end-of-pass barrier; [16] producer total, [17] wait empty.
// INV: 1 = inverse direction (sampling), the contract of coupling_tc2_kernel's INV: a.x = z in the flow's output column order,
// ONE component (c0), steps walked from the last to the first by all three roles (the ring and barrier phases stay in step);
// the gather and the coupling epilogue use the INVERSE gather-order tables; writes a.z_out = x and a.ldj_out = log-det of the
// inverse map.  The exchange, the TMEM plan, the barriers and the weight image are those of the forward.
// RNVP: 1 = RealNVP components (two passes per step, see the header), 0 = Glow.
#define T3_CLK() (PROF ? clock64() : 0LL)
template <int TANH_MODE, int PROF = 0, int INV = 0, int RNVP = 0>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kT3Threads, 1) coupling_tc3_kernel(CouplingArgs a, TcPlan plan) {
  constexpr int kPasses = RNVP ? 2 : 1;              // coupling passes per step
  extern __shared__ __align__(1024) unsigned char smem[];
  asm volatile(".reg .pred t3_p_full;" ::);
  const ModelDims& md = a.md;
  const int D = md.D, Dv = md.Dv;
  float* zs = reinterpret_cast<float*>(smem + plan.off_zs);
  unsigned char* A0 = smem + plan.off_a0;
  float4* xb = reinterpret_cast<float4*>(smem + plan.off_a1);          // exchange buffer (written by the peer)
  float4* stg = reinterpret_cast<float4*>(smem + plan.off_sh);         // what I ship next (read by my bulk copy)
  float* bias_s = reinterpret_cast<float*>(smem + plan.off_bias);
  float4* tab_s = reinterpret_cast<float4*>(smem + plan.off_tab);
  Tc3Misc* misc = reinterpret_cast<Tc3Misc*>(smem + plan.off_misc);
  unsigned char* ring = smem + plan.off_ring;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nst = plan.nst;
  const int p = (int)ptx::cluster_ctarank();         // which half of the hidden units this CTA owns
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    for (int i = 0; i < nst; ++i) { ptx::mbar_init(&misc->full[i], 1); ptx::mbar_init(&misc->empty[i], 1); }
    ptx::mbar_init(&misc->a0r, 16);
    for (int i = 0; i < 4; ++i) { ptx::mbar_init(&misc->a1r[i], 16); ptx::mbar_init(&misc->l1f[i], 1); }
    ptx::mbar_init(&misc->l2own, 1); ptx::mbar_init(&misc->l2ship[0], 1); ptx::mbar_init(&misc->l2ship[1], 1);
    ptx::mbar_init(&misc->sbr[0], 16); ptx::mbar_init(&misc->sbr[1], 16); ptx::mbar_init(&misc->sr, 16); ptx::mbar_init(&misc->l3f, 1);
    ptx::mbar_init(&misc->l3r, 16);
    ptx::mbar_init(&misc->xfull, 1); ptx::mbar_init(&misc->x3full, 1); ptx::mbar_init(&misc->xfree, 16);
    ptx::fence_mbar_init();
    ptx::mbar_arrive_expect_tx(&misc->xfull, kT3XBytes);     // armed for the first chunk the peer ships (two 32 KB bulk copies)
    if (a.G_ll != nullptr) mixture_coefficients(a.rho, a.n_mix, a.skip_c, a.mix_mode, misc->coef);
  }
  if (warp == 1) ptx::tmem_alloc(&misc->tmem_base, 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();                           // the peer's barriers are initialised before anybody arrives on them
  ptx::tc_fence_after();
  const uint32_t tbase = misc->tmem_base;
  const __half* wb = reinterpret_cast<const __half*>(a.wblob);

  if (warp == 0) {
    // ===================================== TMA producer =====================================================
    uint32_t par = 0;
    int slot = 0;
    const long long p_t0 = T3_CLK();
    long long p_wait = 0;
    auto push = [&](const __half* src, uint32_t bytes) {
      const long long tw = T3_CLK();
      t2_wait(&misc->empty[slot], par ^ 1u, a.error_flag, 10, lane);
      p_wait += T3_CLK() - tw;
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(&misc->full[slot], bytes);
        ptx::tma_bulk_g2s(ring + (size_t)slot * kT3StageBytes, src, bytes, &misc->full[slot]);
      }
      __syncwarp();
      if (++slot == nst) { slot = 0; par ^= 1u; }
    };
    for (int u = pair; u < a.num_units; u += npairs) {
      const int cb = a.c0 + (u % a.split) * a.comps_per_unit, ce = min(a.c1, cb + a.comps_per_unit);
      for (int c = cb; c < ce; ++c)
        for (int pi = 0; pi < md.K * kPasses; ++pi) {
          const int kk = RNVP ? pi >> 1 : pi, net = t3_net<RNVP, INV>(pi & 1);
          const int k = INV ? md.K - 1 - kk : kk;
          const StepDesc* sd = a.steps + (c * md.K + k);
          const int kp0 = __ldg(&sd->layer[net][0].Kp);
          const int np3 = __ldg(&sd->layer[net][2].Np);
          const __half* w1 = wb + __ldg(&sd->layer[net][0].w_off) + (size_t)p * kT3HH * kp0;
          const __half* w2 = wb + __ldg(&sd->layer[net][1].w_off) + (size_t)p * kT3H * kT3HH;
          const __half* w3 = wb + __ldg(&sd->layer[net][2].w_off) + (size_t)p * np3 * kT3HH;
          // The packed weights of this configuration (184 MB at cfg5) do not fit in L2 and every CTA pair reaches a step at about
          // the same time, so without help each ring stage's first touch is an HBM miss that ALL pairs wait for: pull the stream
          // into L2 well ahead of the ring (256 KB within the pass, the head of the next pass at the start of this one).
          constexpr uint32_t kAhead = 262144;
          if (ptx::elect_one()) {
            const bool same = RNVP && (pi & 1) == 0;     // the step's second pass is next
            const int nn = t3_net<RNVP, INV>(same ? 1 : 0);
            const StepDesc* sn = same ? sd : (kk + 1 < md.K) ? (INV ? sd - 1 : sd + 1)
                               : (c + 1 < ce) ? a.steps + (c + 1) * md.K + (INV ? md.K - 1 : 0) : nullptr;
            if (sn != nullptr) {
              const int kpn = __ldg(&sn->layer[nn][0].Kp), npn = __ldg(&sn->layer[nn][2].Np);
              ptx::prefetch_l2(wb + __ldg(&sn->layer[nn][0].w_off) + (size_t)p * kT3HH * kpn, (uint32_t)(kT3HH * kpn * 2));
              ptx::prefetch_l2(wb + __ldg(&sn->layer[nn][1].w_off) + (size_t)p * kT3H * kT3HH, kAhead);
              ptx::prefetch_l2(wb + __ldg(&sn->layer[nn][2].w_off) + (size_t)p * npn * kT3HH, (uint32_t)(npn * kT3HH * 2));
            }
          }
          __syncwarp();
          uint32_t w2_pos = 0;                                  // bytes of my W2 stream pushed so far
          auto push_w2 = [&](const __half* src) {
            if (w2_pos + kAhead < (uint32_t)(kT3H * kT3HH * 2) && ptx::elect_one())
              ptx::prefetch_l2(reinterpret_cast<const unsigned char*>(w2) + w2_pos + kAhead, kT3StageBytes);
            w2_pos += kT3StageBytes;
            push(src, kT3StageBytes);
          };
          for (int j = 0; j < (kp0 >> 4); ++j) push(w1 + (size_t)j * 8192, kT3StageBytes);     // W1 half: (Kp0 / 16) x 16 KB
          t3_schedule(p, [&](int op, int x, int y) {
            if (op == T3_OP_OWN) {
              const __half* base = w2 + (size_t)(2 * (x >> 1) + 1) * 65536;       // pair m = x >> 1: [shipped block][own block]
              for (int t = 0; t < 8; ++t) push_w2(base + (size_t)t * 8192);
            } else if (op == T3_OP_SHIP) {
              const __half* base = w2 + (size_t)(2 * (x >> 1)) * 65536 + (size_t)y * 32768;
              for (int t = 0; t < 4; ++t) push_w2(base + (size_t)t * 8192);
            } else {
              push(w3 + (size_t)x * 8 * np3 * 16, (uint32_t)(8 * np3) * 32u);
            }
          });
        }
    }
    if (PROF && a.prof != nullptr && blockIdx.x == 0 && lane == 0) { a.prof[16] = T3_CLK() - p_t0; a.prof[17] = p_wait; }
  } else if (warp == 1) {
    // ===================================== MMA issuer =======================================================
    uint32_t units = 0;
    uint32_t n_sbr[2] = {0, 0}, n_sr = 0, n_l3r = 0;  // waits done so far on the slot-B / packed-piece / piece-read barriers
    int nslot = 0, slot = 0;
    uint32_t npar = 0;
    const long long m_t0 = T3_CLK();
    long long m_wf = 0, m_wa = 0, m_wb = 0, m_ws = 0, tw;
    const uint64_t a0_desc = ptx::make_smem_desc(ptx::smem_u32(A0));
    const uint64_t ring_desc = ptx::make_smem_desc(ptx::smem_u32(ring));
    const uint32_t idesc_128 = ptx::make_idesc_f16(128, 128);
    const uint32_t idesc_64 = ptx::make_idesc_f16(128, 64);
    // readiness of the NEXT ring stage is tested before the current stage's MMAs are issued and consumed afterwards
    // (an mbarrier test costs 100-160 cycles on this warp, see coupling_tc2.cuh)
    auto test_full = [&](uint64_t* bar, uint32_t par) {
      asm volatile("mbarrier.test_wait.parity.shared::cta.b64 t3_p_full, [%0], %1;" ::"r"(ptx::smem_u32(bar)), "r"(par) : "memory");
    };
    test_full(&misc->full[0], 0u);
    auto acquire = [&]() -> uint64_t {
      slot = nslot;
      uint32_t full_ok;
      asm volatile("selp.u32 %0, 1, 0, t3_p_full;" : "=r"(full_ok));
      tw = T3_CLK();
      if (!full_ok) ptx::mbar_wait(&misc->full[slot], npar, a.error_flag, 21);
      m_wf += T3_CLK() - tw;
      ptx::tc_fence_after();
      if (++nslot == nst) { nslot = 0; npar ^= 1u; }
      test_full(&misc->full[nslot], npar);
      return ring_desc + (uint64_t)((uint32_t)slot * (kT3StageBytes >> 4));
    };
    auto wait_epi = [&](uint64_t* bar, uint32_t par, int code) {
      ptx::mbar_wait(bar, par, a.error_flag, code);
      ptx::tc_fence_after();
    };
    for (int u = pair; u < a.num_units; u += npairs) {
      const int cb = a.c0 + (u % a.split) * a.comps_per_unit, ce = min(a.c1, cb + a.comps_per_unit);
      for (int c = cb; c < ce; ++c)
        for (int pi = 0; pi < md.K * kPasses; ++pi, ++units) {
          const int kk = RNVP ? pi >> 1 : pi, net = t3_net<RNVP, INV>(pi & 1);
          const int k = INV ? md.K - 1 - kk : kk;
          const StepDesc* sd = a.steps + (c * md.K + k);
          const int k0s = __ldg(&sd->layer[net][0].Kp) >> 4;
          const int np3 = __ldg(&sd->layer[net][2].Np);
          const uint32_t idesc_o = ptx::make_idesc_f16(128, np3);
          const uint32_t b3_step = (uint32_t)np3 * 2u;
          const uint32_t upar = units & 1u;
          // ---- layer 1: the W1 half sits in k0s held ring stages; chunk q -> slot A (even q) / slot B + last (odd q) ----
          uint64_t l1_desc[2];
          int l1_slot[2];
          for (int j = 0; j < k0s; ++j) { l1_desc[j] = acquire(); l1_slot[j] = slot; }
          tw = T3_CLK();
          wait_epi(&misc->a0r, upar, 20);
          m_wa += T3_CLK() - tw;
#pragma unroll 1
          for (int q = 0; q < 4; ++q) {
            tw = T3_CLK();
            if (q >= 2) wait_epi(&misc->a1r[q - 2], upar, 22);                    // its accumulator slot has been read out
            m_wa += T3_CLK() - tw;
            if (ptx::elect_one()) {
              const uint32_t d = tbase + ((q & 1) ? kT3SlotB0 : kT3SlotA);
              // chunk q = k0s k-slabs of [128 x 16] at byte q * k0s * 4096 of the W1 half image (16 KB per held stage)
              const uint32_t byte0 = (uint32_t)(q * k0s) * 4096u;
              const uint64_t bq = l1_desc[byte0 >> 14] + (uint64_t)((byte0 & 16383u) >> 4);
              for (int i = 0; i < k0s; ++i)
                ptx::umma_f16(d, a0_desc + (uint64_t)(i * 256), bq + (uint64_t)(i * 256), idesc_128, i > 0 ? 1u : 0u);
              ptx::umma_commit(&misc->l1f[q]);
              if (q == 3) for (int j = 0; j < k0s; ++j) ptx::umma_commit(&misc->empty[l1_slot[j]]);
            }
            __syncwarp();
          }
          tw = T3_CLK();
          wait_epi(&misc->a1r[2], upar, 22);
          wait_epi(&misc->a1r[3], upar, 22);          // all of A1_p exists, slots A and B are free
          m_wa += T3_CLK() - tw;
          // ---- layer 2 (partial sums over my K half) and my partial last-layer product ----
          t3_schedule(p, [&](int op, int x, int y) {
            if (op == T3_OP_OWN) {
              if ((x >> 1) > 0) {                    // the previous piece's last-layer product has been read out of slot A
                tw = T3_CLK();
                wait_epi(&misc->l3r, n_l3r & 1u, 26);
                m_ws += T3_CLK() - tw;
                ++n_l3r;
              }
              for (int t = 0; t < 8; ++t) {
                const uint64_t bd = acquire();
                const int cur = slot;
                if (ptx::elect_one()) {
                  const uint32_t d = tbase + kT3SlotA;
#pragma unroll
                  for (int i = 0; i < 4; ++i)
                    ptx::umma_f16_ts(d, tbase + 8u * (uint32_t)(4 * t + i), bd + (uint64_t)(i * 256), idesc_128, (t > 0 || i > 0) ? 1u : 0u);
                  ptx::umma_commit(&misc->empty[cur]);
                  if (t == 7) ptx::umma_commit(&misc->l2own);
                }
                __syncwarp();
              }
            } else if (op == T3_OP_SHIP) {
              tw = T3_CLK();
              wait_epi(&misc->sbr[y], (n_sbr[y] & 1u) ^ 1u, 25);                  // slot B y read out (passes the first time)
              m_wb += T3_CLK() - tw;
              ++n_sbr[y];
              for (int t = 0; t < 4; ++t) {
                const uint64_t bd = acquire();
                const int cur = slot;
                if (ptx::elect_one()) {
                  const uint32_t d = tbase + (y ? kT3SlotB1 : kT3SlotB0);
#pragma unroll
                  for (int i = 0; i < 8; ++i)
                    ptx::umma_f16_ts(d, tbase + 8u * (uint32_t)(8 * t + i), bd + (uint64_t)(i * 128), idesc_64, (t > 0 || i > 0) ? 1u : 0u);
                  ptx::umma_commit(&misc->empty[cur]);
                  if (t == 3) ptx::umma_commit(&misc->l2ship[y]);
                }
                __syncwarp();
              }
            } else {
              // last-layer piece of own chunk number x: A2 packed in slot A [0, 64) x its k-slabs of W3 -> last-layer accumulator
              const uint64_t bd = acquire();
              const int cur = slot;
              tw = T3_CLK();
              wait_epi(&misc->sr, n_sr & 1u, 23);
              m_ws += T3_CLK() - tw;
              ++n_sr;
              if (ptx::elect_one()) {
                const uint32_t at = tbase + kT3SlotA, d = tbase + kT3L3Tmp;       // fresh product per piece, summed by the epilogue
                for (int i = 0; i < 8; ++i)
                  ptx::umma_f16_ts(d, at + 8u * (uint32_t)i, bd + (uint64_t)((uint32_t)i * b3_step), idesc_o, i > 0 ? 1u : 0u);
                ptx::umma_commit(&misc->empty[cur]);
                ptx::umma_commit(&misc->l3f);
              }
              __syncwarp();
            }
          });
        }
    }
    if (PROF && a.prof != nullptr && blockIdx.x == 0 && lane == 0) {
      a.prof[0] = T3_CLK() - m_t0; a.prof[1] = m_wf; a.prof[2] = m_wa; a.prof[3] = m_wb; a.prof[4] = m_ws; a.prof[5] = units;
    }
  } else {
    // ===================================== epilogue / elementwise warps =====================================
    const int et = threadIdx.x - 64;
    const int warp_e = et >> 5;
    const int quad = warp & 3;
    const int g = warp_e >> 2;
    const int row = quad * 32 + lane;
    float* zrow = zs + row * Dv;
    const uint32_t lane_base = tbase + ((uint32_t)(quad * 32) << 16);
    const int dq = (D + 3) >> 2;
    const int h0col = min(D, g * dq), h1col = min(D, (g + 1) * dq);
    uint32_t units = 0;
    uint32_t n_own = 0, n_ship[2] = {0, 0}, n_xfree = 0, n_l3f = 0;   // waits done so far on l2own / xfull, l2ship, xfree, l3f
    const long long e_t0 = T3_CLK();
    long long e_l1f = 0, e_own = 0, e_xfull = 0, e_ship = 0, e_xfree = 0, e_l3f = 0, e_x3 = 0, e_g = 0, e_c1 = 0, e_c2 = 0, e_c3 = 0, e_c4 = 0, tq;
    float* const part = reinterpret_cast<float*>(A0);
    const uint32_t peer = (uint32_t)(p ^ 1);
    const uint32_t xb_peer = ptx::mapa(ptx::smem_u32(xb), peer);                 // the PEER's exchange buffer
    const uint32_t xfull_peer = ptx::mapa(ptx::smem_u32(&misc->xfull), peer);
    const uint32_t x3full_peer = ptx::mapa(ptx::smem_u32(&misc->x3full), peer);
    const uint32_t xfree_peer = ptx::mapa(ptx::smem_u32(&misc->xfree), peer);
    // EVERY lane arrives (release at cluster scope orders that lane's own DSMEM stores / exchange-buffer loads before the
    // arrival): a cluster-scope fence per lane followed by one elected arrival stalled every warp on MEMBAR for thousands of
    // cycles per hand-off (ncu: 24 % of the warp samples)
    // xfree only says "my loads from the exchange buffer are done": no writes to publish, so one RELAXED arrival per warp, issued
    // after the arithmetic that consumed the loaded values (a release arrival per lane cost ~1 k cycles per hand-off)
    auto remote_arrive = [&](uint32_t bar_cluster_addr) {
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_remote_relaxed(bar_cluster_addr);
    };
    // staging of one pass's constants: biases of network `net` (b1 own half | b2 own chunks | b3), gather-order tables, scalars
    auto stage_pass = [&](const StepDesc* sd, int net, int buf) {
      float* bdst = bias_s + buf * kT3BiasFloats;
      const float* b1 = a.fblob + __ldg(&sd->layer[net][0].b_off) + p * kT3HH;
      const float* b2 = a.fblob + __ldg(&sd->layer[net][1].b_off);
      const float* b3 = a.fblob + __ldg(&sd->layer[net][2].b_off);
      if (et < 128) ptx::cp_async16(bdst + 4 * et, b1 + 4 * et);
      else if (et < 256) { const int i = et - 128; const int m = i >> 5, w = i & 31; ptx::cp_async16(bdst + 512 + 128 * m + 4 * w, b2 + 128 * (2 * m + p) + 4 * w); }
      else if (et < 272) ptx::cp_async16(bdst + 1024 + 4 * (et - 256), b3 + 4 * (et - 256));
      else if (et >= 384) {
        const int i = et - 384;
        ptx::cp_async16(tab_s + buf * (2 * kEpPad) + i, reinterpret_cast<const float4*>(a.fblob + __ldg(&sd->ep_off)) + (INV ? 2 * kEpPad : 0) + i);
      }
      if (et == 300) {
        int* m = misc->meta[buf];
        m[0] = __ldg(&sd->in_dim); m[1] = __ldg(&sd->out_dim); m[2] = __ldg(&sd->layer[net][0].Kp); m[3] = __ldg(&sd->layer[net][2].Np);
      }
    };
    if (pair < a.num_units) {
      const int cb0 = a.c0 + (pair % a.split) * a.comps_per_unit;
      stage_pass(a.steps + cb0 * md.K + (INV ? md.K - 1 : 0), t3_net<RNVP, INV>(0), 0);
    }
    for (int u = pair; u < a.num_units; u += npairs) {
      const int tile = u / a.split, cs = u - tile * a.split;
      const int cb = a.c0 + cs * a.comps_per_unit, ce = min(a.c1, cb + a.comps_per_unit);
      const long long row0 = (long long)tile * kTcRows;
      const long long gr = row0 + row;
      for (int c = cb; c < ce; ++c) {
        const CompDesc* cdp = a.comps + c;
        const float2 cconst = __ldg(reinterpret_cast<const float2*>(a.fblob + a.cc_off) + c);
        const long long base_off = (md.base == GBNF_BASE_STD_NORMAL) ? 0LL : __ldg(&cdp->base_off);
        const float ldj_const = cconst.x, base_const = cconst.y;
        t2_epi_bar();                                // previous component's readers are done with zs / part
        {                                            // x tile (L2-resident after the first component) -> this thread's share of zs
          // INV: z arrives in the flow's OUTPUT column order, logical column j lives at physical column sigma[j]
          const int* sig = INV ? a.iblob + __ldg(&cdp->sigma_off) : nullptr;
          const long long gbase = row0 * D;
          const long long glimit = a.B * (long long)D;
          const int total = kTcRows * D;
          for (int i0 = et; i0 < total; i0 += 8 * kT3EpiThreads) {
            float v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const int i = i0 + q * kT3EpiThreads;
              v[q] = (i < total && gbase + i < glimit) ? __ldg(a.x + gbase + i) : 0.f;
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const int i = i0 + q * kT3EpiThreads;
              if (i < total) { const int r = i / D, j = i - r * D; zs[r * Dv + (INV ? __ldg(sig + j) : j)] = v[q]; }
            }
          }
          if (g == 0) for (int q = D; q < Dv; ++q) zrow[q] = 0.f;
        }
        ptx::cp_async_wait_all();
        t2_epi_bar();
        float lsum = 0.f;
        for (int pi = 0; pi < md.K * kPasses; ++pi, ++units) {
          const int kk = RNVP ? pi >> 1 : pi, net = t3_net<RNVP, INV>(pi & 1);
          const int k = INV ? md.K - 1 - kk : kk;
          const StepDesc* sd = a.steps + (c * md.K + k);
          const int buf = units & 1u;
          const int* meta = misc->meta[buf];
          const int in_dim = meta[0], out_dim = meta[1], np3 = meta[3];
          const float4* tab1 = tab_s + buf * (2 * kEpPad);
          const float4* tab2 = tab1 + kEpPad;
          const float* bias_c = bias_s + buf * kT3BiasFloats;
          const uint32_t upar = units & 1u;
          const int kfirst = INV ? md.K - 1 : 0;
          const bool same = RNVP && (pi & 1) == 0;     // the step's second pass is next
          const StepDesc* sd_next = same ? sd : (kk + 1 < md.K) ? (INV ? sd - 1 : sd + 1)
                                    : (c + 1 < ce) ? a.steps + (c + 1) * md.K + kfirst
                                    : (u + npairs < a.num_units) ? a.steps + (a.c0 + ((u + npairs) % a.split) * a.comps_per_unit) * md.K + kfirst
                                                                 : nullptr;
          // mixed RealNVP networks: t = ReLU, s = tanh (as in coupling_tc2.cuh)
          const int act_kind = (md.act == GBNF_ACT_RELU || (RNVP && md.act == GBNF_ACT_MIXED && net == 0)) ? 2 : 1;
          // ---- ActNorm / eval-BatchNorm affine fused into the gather of z1 -> A0 (both CTAs build the same image); the RealNVP
          //      t pass feeds z1 as the s pass of the step leaves it (forward) or finds it (inverse) ----
          tq = T3_CLK();
          if (RNVP && net == 0) t2_gather_z1<0, 1>(zrow, tab1, in_dim, meta[2] >> 3, g, row, A0, a.error_flag);
          else                  t2_gather_z1<INV>(zrow, tab1, in_dim, meta[2] >> 3, g, row, A0, a.error_flag);
          ptx::fence_proxy_async_smem();
          ptx::tc_fence_before();
          t2_warp_arrive(&misc->a0r, lane);
          if (et == 0) ptx::mbar_arrive_expect_tx(&misc->x3full, (uint32_t)np3 * 512u);   // this pass's partial last-layer product of the peer
          e_g += T3_CLK() - tq;
          // ---- layer 1: my 512 hidden units, chunk q -> bias + act -> fp16 pairs -> A1 quarter q ----
#pragma unroll 1
          for (int q = 0; q < 4; ++q) {
            tq = T3_CLK();
            t2_wait(&misc->l1f[q], upar, a.error_flag, 30, lane);
            e_l1f += T3_CLK() - tq;
            tq = T3_CLK();
            ptx::tc_fence_after();
            uint32_t pk[16];
            {
              uint32_t r[32];
              ptx::tmem_ld32(lane_base + ((q & 1) ? kT3SlotB0 : kT3SlotA) + (uint32_t)g * 32u, r);
              ptx::tmem_ld_wait();
              if (act_kind == 1) t2_act_pack<1, TANH_MODE>(r, bias_c + q * 128 + g * 32, pk, a.error_flag);
              else               t2_act_pack<2, TANH_MODE>(r, bias_c + q * 128 + g * 32, pk, a.error_flag);
            }
            ptx::tmem_st16(lane_base + (uint32_t)q * 64u + (uint32_t)g * 16u, pk);
            ptx::tmem_st_wait();
            ptx::tc_fence_before();
            t2_warp_arrive(&misc->a1r[q], lane);
            e_c1 += T3_CLK() - tq;
          }
          // the next pass's constants (other buffer: its last readers finished a pass ago)
          if (sd_next != nullptr) stage_pass(sd_next, t3_net<RNVP, INV>(same ? 1 : 0), buf ^ 1);
          // ---- layer 2: per chunk pair m -- [read out the previous own chunk's last-layer product] -> the two shipped halves
          //      (their MMAs ran under the previous own epilogue) -> my own chunk ----
          const int c0 = g * 16;
          float acc3[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) acc3[i] = 0.f;
          auto l3read = [&](int mm) {
            tq = T3_CLK();
            t2_wait(&misc->l3f, n_l3f & 1u, a.error_flag, 32, lane);
            ++n_l3f;
            e_l3f += T3_CLK() - tq;
            ptx::tc_fence_after();
            if (c0 < np3) {
              uint32_t r3[16];
              ptx::tmem_ld16(lane_base + kT3L3Tmp + (uint32_t)c0, r3);
              ptx::tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 16; ++i) acc3[i] += __uint_as_float(r3[i]);
            }
            ptx::tc_fence_before();
            if (mm < 3) t2_warp_arrive(&misc->l3r, lane);      // slot A may take the next own chunk
          };
#pragma unroll 1
          for (int m = 0; m < 4; ++m) {
            if (m > 0) l3read(m - 1);
#pragma unroll
            for (int y = 0; y < 2; ++y) {
              tq = T3_CLK();
              t2_wait(&misc->l2ship[y], n_ship[y] & 1u, a.error_flag, 34, lane);
              e_ship += T3_CLK() - tq;
              tq = T3_CLK();
              ++n_ship[y];
              ptx::tc_fence_after();
              uint32_t r[16];
              ptx::tmem_ld16(lane_base + (y ? kT3SlotB1 : kT3SlotB0) + (uint32_t)g * 16u, r);
              ptx::tmem_ld_wait();
              ptx::tc_fence_before();
              t2_warp_arrive(&misc->sbr[y], lane);   // slot B y may be overwritten by the next pair's half
              // The half chunk goes to the peer as ONE 32 KB bulk copy out of a local staging buffer (DSMEM stores from 512
              // threads ran at ~10 B/clk and kept the epilogue warps busy for 3.4 k cycles per half; the copy engine moves
              // ~20 B/clk on its own).  Staging layout = destination layout: float4 (c4 * 128 + row), c4 = column / 4.
              if (et == 0) ptx::bulk_wait_read0();   // my previous copy has read the staging buffer
              t2_epi_bar();
#pragma unroll
              for (int i = 0; i < 4; ++i)
                stg[(4 * g + i) * kTcRows + row] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]),
                                                               __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3]));
              ptx::fence_proxy_async_smem();
              t2_epi_bar();
              if (et == 0) {
                if (y == 0) {                        // the peer has consumed the previous chunk I wrote into its buffer
                  const long long tx = T3_CLK();
                  ptx::mbar_wait_cluster(&misc->xfree, (n_xfree & 1u) ^ 1u, a.error_flag, 35);
                  e_xfree += T3_CLK() - tx;
                }
                ptx::bulk_s2c(xb_peer + (uint32_t)y * (kT3XBytes / 2), stg, kT3XBytes / 2, xfull_peer);
                ptx::bulk_commit();
              }
              if (y == 0) ++n_xfree;
              e_c3 += T3_CLK() - tq;
            }
            {
              tq = T3_CLK();
              t2_wait(&misc->l2own, n_own & 1u, a.error_flag, 31, lane);
              e_own += T3_CLK() - tq;
              ptx::tc_fence_after();
              tq = T3_CLK();
              ptx::mbar_wait_cluster(&misc->xfull, n_own & 1u, a.error_flag, 33);   // the peer's partial sums of this chunk have landed
              __syncwarp();
              e_xfull += T3_CLK() - tq;
              tq = T3_CLK();
              ++n_own;
              uint32_t pk[16];
              {
                uint32_t r[32];
                ptx::tmem_ld32(lane_base + kT3SlotA + (uint32_t)g * 32u, r);
                ptx::tmem_ld_wait();
                if (act_kind == 1) t3_act_pack32_add<1, TANH_MODE>(r, xb + (g * 8) * kTcRows + row, bias_c + 512 + 128 * m + g * 32, pk, a.error_flag);
                else               t3_act_pack32_add<2, TANH_MODE>(r, xb + (g * 8) * kTcRows + row, bias_c + 512 + 128 * m + g * 32, pk, a.error_flag);
              }
              t2_quad_bar(quad);                     // all four threads of the row have read their columns of slot A
              ptx::tmem_st16(lane_base + kT3SlotA + (uint32_t)g * 16u, pk);
              ptx::tmem_st_wait();
              ptx::tc_fence_before();
              t2_warp_arrive(&misc->sr, lane);
              if (et == 0) ptx::mbar_arrive_expect_tx(&misc->xfull, kT3XBytes);   // arm the next chunk's phase (all waiters have
                                                                                  // passed: the peer ships only after 16 xfree arrivals)
              remote_arrive(xfree_peer);             // my exchange buffer may be overwritten
              e_c2 += T3_CLK() - tq;
            }
          }
          // ---- last layer: my partial product = the four pieces summed in registers; exchange the partial products, then the
          //      coupling transform on this thread's 16-column slice ----
          l3read(3);
          if (et == 0) ptx::bulk_wait_read0();
          t2_epi_bar();
          if (c0 < np3) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
              stg[(4 * g + i) * kTcRows + row] = make_float4(acc3[4 * i], acc3[4 * i + 1], acc3[4 * i + 2], acc3[4 * i + 3]);
          }
          ptx::fence_proxy_async_smem();
          t2_epi_bar();
          if (et == 0) {
            tq = T3_CLK();
            ptx::mbar_wait_cluster(&misc->xfree, (n_xfree & 1u) ^ 1u, a.error_flag, 36);
            e_xfree += T3_CLK() - tq;
            ptx::bulk_s2c(xb_peer, stg, (uint32_t)np3 * 512u, x3full_peer);       // [np3 / 4][128 rows] float4
            ptx::bulk_commit();
          }
          ++n_xfree;
          tq = T3_CLK();
          ptx::mbar_wait_cluster(&misc->x3full, upar, a.error_flag, 37);
          __syncwarp();
          e_x3 += T3_CLK() - tq;
          tq = T3_CLK();
          if (c0 < np3) {
            float acc[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 o = xb[(4 * g + i) * kTcRows + row];
              acc[4 * i + 0] = acc3[4 * i + 0] + o.x;      // a + b == b + a: both CTAs get the same bits
              acc[4 * i + 1] = acc3[4 * i + 1] + o.y;
              acc[4 * i + 2] = acc3[4 * i + 2] + o.z;
              acc[4 * i + 3] = acc3[4 * i + 3] + o.w;
            }
            const float* bias = bias_c + 1024;
            if (!RNVP && md.coupling == GBNF_COUPLING_AFFINE) {
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
                const float shift = acc[2 * jj] + b.x;
                const float raw = acc[2 * jj + 1] + b.y;
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
                  if (RNVP) {                                                       // transformations.py:575-577
                    const float v = acc[half * 8 + jj] + bias[j];
                    if (net == 0) {                                                 // t_net: shift
                      z[jj] = INV ? z[jj] - v : z[jj] + v;
                    } else if (INV) {                                               // s_net: scale, then eval-BatchNorm inverse
                      const float y = z[jj] * __expf(-v);
                      z[jj] = (y + t[jj].x) * t[jj].y + t[jj].z;
                      lsum -= (j < out_dim) ? v : 0.f;
                    } else {                                                        // eval-BatchNorm, then s_net: scale
                      const float zn = (z[jj] + t[jj].x) * t[jj].y + t[jj].z;
                      z[jj] = zn * __expf(v);
                      lsum += (j < out_dim) ? v : 0.f;
                    }
                  } else if (INV) {
                    z[jj] = ((z[jj] - (acc[half * 8 + jj] + bias[j])) + t[jj].x) * t[jj].y + t[jj].z;   // glow.py:350, then ActNorm reverse
                  } else {
                    const float zn = (z[jj] + t[jj].x) * t[jj].y + t[jj].z;
                    z[jj] = zn + (acc[half * 8 + jj] + bias[j]);                      // additive coupling, glow.py:328-329
                  }
                }
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) if (c0 + half * 8 + jj < out_dim) zrow[__float_as_int(t[jj].w)] = z[jj];
              }
            }
          }
          remote_arrive(xfree_peer);                 // I have read the peer's partial product out of my exchange buffer
          ptx::cp_async_wait_all();
          if (et == 0) ptx::bulk_wait_read0();       // my copy has read the staging buffer, which the next gather (A0) overwrites
          t2_epi_bar();                              // z2 updates, staged constants of the next pass
          e_c4 += T3_CLK() - tq;
        }
        // ---- component log-density for this row (both CTAs hold the same z; rank 0 writes) ----
        t2_component_logq(a, zrow, lsum, part, row, g, quad, h0col, h1col, Dv, base_off, INV ? -ldj_const : ldj_const, base_const,
                          misc->coef, c, tile, p == 0);
        if (p == 0 && a.z_out != nullptr && gr < a.B) {
          if (INV) {   // physical == logical column order at the flow's input
            for (int j = h0col; j < h1col; ++j) a.z_out[gr * D + j] = zrow[j];
          } else {
            const int* sig = a.iblob + __ldg(&cdp->sigma_off);
            for (int j = h0col; j < h1col; ++j) a.z_out[gr * D + j] = zrow[__ldg(sig + j)];
          }
        }
      }
      if (a.G_ll != nullptr && p == 0) t2_tile_logsumexp(a, tile, gr, g, et, &misc->last_flag);
    }
    if (et == 0) ptx::bulk_wait0();                  // my last bulk copy into the peer has completed
    if (PROF && a.prof != nullptr && blockIdx.x == 0 && et == 0) {
      a.prof[8] = T3_CLK() - e_t0; a.prof[9] = e_l1f; a.prof[10] = e_own; a.prof[11] = e_xfull; a.prof[12] = e_ship; a.prof[13] = e_xfree;
      a.prof[14] = e_l3f; a.prof[15] = e_x3; a.prof[19] = e_g; a.prof[20] = e_c1; a.prof[21] = e_c2; a.prof[22] = e_c3; a.prof[23] = e_c4;
    }
    ptx::tc_fence_before();
  }
  __syncthreads();
  ptx::cluster_sync_all();       // the peer may still be writing into my shared memory / arriving on my barriers until here
  if (warp == 1) {
    __syncwarp();
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tbase, 512);
  }
}

#undef T3_CLK
inline cudaError_t tc3_configure() {
  cudaError_t e = cudaFuncSetAttribute(coupling_tc3_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc3_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc3_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc3_kernel<0, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc3_kernel<1, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc3_kernel<0, 0, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc3_kernel<1, 0, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc3_kernel<0, 0, 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc3_kernel<1, 0, 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  return e;
}

// How many CTA pairs the device can keep resident at once (GPCs with an odd number of usable SMs strand one SM each): a
// persistent grid larger than this would run its last clusters as a second wave.
inline int tc3_max_pairs(const TcPlan& p, int num_sms) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * (num_sms / 2)), 1, 1);
  cfg.blockDim = dim3(kT3Threads, 1, 1);
  cfg.dynamicSmemBytes = p.smem_bytes;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, coupling_tc3_kernel<0>, &cfg) != cudaSuccess || n <= 0) { cudaGetLastError(); n = num_sms / 2; }
  return std::min(n, num_sms / 2);
}

// grid = 2 x (CTA pairs): the cluster dimension is a compile-time attribute of the kernel.  The cycle-counter build exists for
// Glow only: a profiling RealNVP handle runs the production kernel.
inline int tc3_launch(const CouplingArgs& a, const TcPlan& p, int pairs, cudaStream_t st, int prof = 0) {
  if (a.md.nnets == 2) {
    if (p.tanh_mode == 0) coupling_tc3_kernel<0, 0, 0, 1><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p);
    else                  coupling_tc3_kernel<1, 0, 0, 1><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p);
    return 0;
  }
  if (prof) { coupling_tc3_kernel<0, 1><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p); return 0; }
  if (p.tanh_mode == 0) coupling_tc3_kernel<0><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p);
  else                  coupling_tc3_kernel<1><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p);
  return 0;
}

inline int tc3_launch_inverse(const CouplingArgs& a, const TcPlan& p, int pairs, cudaStream_t st) {
  if (a.md.nnets == 2) {
    if (p.tanh_mode == 0) coupling_tc3_kernel<0, 0, 1, 1><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p);
    else                  coupling_tc3_kernel<1, 0, 1, 1><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p);
    return 0;
  }
  if (p.tanh_mode == 0) coupling_tc3_kernel<0, 0, 1><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p);
  else                  coupling_tc3_kernel<1, 0, 1><<<2 * pairs, kT3Threads, p.smem_bytes, st>>>(a, p);
  return 0;
}

// ---- weight image of the pair kernel (see the header comment): element i of a layer's image -> (n, k) of nn.Linear.weight ----
__global__ void pack_weight_tc3_kernel(const float* __restrict__ W, const float* __restrict__ b, LayerDesc ld, int layer,
                                       __half* __restrict__ wblob, float* __restrict__ fblob, int* overflow) {
  const long long total = (long long)ld.Kp * ld.Np;
  __half* dst = wblob + ld.w_off;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long half_elems = total / 2;
    const int p = (int)(i / half_elems);
    long long r = i % half_elems;
    int n, k;
    if (layer == 0) {            // [chunk q][k-slab][128 x 16]; n = hidden unit, k = input feature
      const int per_chunk = 128 * ld.Kp;
      const int q = (int)(r / per_chunk), rr0 = (int)(r % per_chunk);
      const int slab = rr0 / 2048, rr = rr0 % 2048;
      n = kT3HH * p + 128 * q + (rr / 128) * 8 + (rr % 64) / 8;
      k = 16 * slab + ((rr % 128) / 64) * 8 + rr % 8;
    } else if (layer == 1) {     // [J][own: [32 slabs][128 x 16] | shipped: [2 halves][32 slabs][64 x 16]]; k in my half
      // blocks in the order CTA p consumes them: pair m = [shipped chunk 2 m + 1 - p][own chunk 2 m + p]
      const int blk = (int)(r / 65536), rr0 = (int)(r % 65536);
      const int J = (blk & 1) ? 2 * (blk >> 1) + p : 2 * (blk >> 1) + 1 - p;
      if ((J & 1) == p) {
        const int slab = rr0 / 2048, rr = rr0 % 2048;
        n = 128 * J + (rr / 128) * 8 + (rr % 64) / 8;
        k = kT3HH * p + 16 * slab + ((rr % 128) / 64) * 8 + rr % 8;
      } else {
        const int hh = rr0 / 32768, r2 = rr0 % 32768;
        const int slab = r2 / 1024, rr = r2 % 1024;
        n = 128 * J + 64 * hh + (rr / 128) * 8 + (rr % 64) / 8;
        k = kT3HH * p + 16 * slab + ((rr % 128) / 64) * 8 + rr % 8;
      }
    } else {                     // [own chunk m][8 slabs][Np x 16]; k = hidden unit of layer 2 in own chunk J = 2 m + p
      const int per_piece = 128 * ld.Np;
      const int m = (int)(r / per_piece), rr0 = (int)(r % per_piece);
      const int slab = rr0 / (16 * ld.Np), rr = rr0 % (16 * ld.Np);
      n = (rr / 128) * 8 + (rr % 64) / 8;
      k = 128 * (2 * m + p) + 16 * slab + ((rr % 128) / 64) * 8 + rr % 8;
    }
    const float v = (k < ld.K_in && n < ld.N_out) ? W[(long long)n * ld.K_in + k] : 0.f;
    const __half hv = __float2half_rn(v);
    if (__hisinf(hv) || __hisnan(hv)) *overflow = 1;
    dst[i] = hv;
  }
  if (blockIdx.x == 0)
    for (int n = threadIdx.x; n < ld.Np; n += blockDim.x) fblob[ld.b_off + n] = (n < ld.N_out) ? b[n] : 0.f;
}

}  // namespace gbnf
