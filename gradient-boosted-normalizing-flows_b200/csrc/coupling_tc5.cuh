// Interleaved s / t kernel for RealNVP components of hidden width 256 with tanh networks (BASELINE configurations 1 and 2),
// forward direction.
//
// A RealNVP step evaluates TWO independent MLPs on the same input z1 -- the shift network t and the log-scale network s
// (models/transformations.py:560-579, models/realnvp.py:35-76) -- and coupling_tc2_kernel runs them one after the other, each as a
// strictly serial chain layer 1 -> tanh -> layer 2 -> tanh -> last layer.  These configurations are MUFU bound (4 h tanh per row
// and step: 8.2 k cycles per 128-row step against 6.0 k of GEMM at the measured peak rate), and in a serial chain neither the
// MUFU nor the tensor pipe is busy while the other works: 20 k cycles per step.  At h = 256 BOTH networks fit in tensor memory
// side by side, so this kernel interleaves them: while the epilogue warps activate a chunk of one network, the tensor pipe
// multiplies the next chunk of the other.
//
//   TMEM (512 columns): A1_t [0, 128) | A1_s [128, 256) | slot_t [256, 384) | slot_s [384, 512)
//     layer 1, chunk q (N = 128) of network n -> slot_n; epilogue: bias + tanh -> fp16 pairs -> A1_n quarter q
//     layer 2, chunk j (N = 128, K = 256 from A1_n) -> slot_n; epilogue: bias + tanh -> fp16 pairs packed IN PLACE (slot_n[0, 64) =
//       k-piece j of the last layer's A operand); that piece's last-layer product goes to the vacated slot_n[64, 64 + Np3) and is
//       summed in registers by the epilogue (two pieces per network)
//   op order of both the MMA issuer and the epilogue: L1(t,0) L1(s,0) L1(t,1) L1(s,1) L2(t,0) L2(s,0) L3(t,0) L3(s,0) L2(t,1) L2(s,1)
//   L3(t,1) L3(s,1); then the coupling z2' = t + z2 exp(s) with the eval-BatchNorm affine of the gather-order tables, log-det += sum s.
//   One gather of z1 feeds both networks (one A0).  Weight image, tables and work units are coupling_tc2_kernel's (same handle).
#pragma once
#include "coupling_tc2.cuh"

namespace gbnf {

struct Tc5Misc {
  uint64_t full[kT2MaxStages];
  uint64_t empty[kT2MaxStages];
  uint64_t a0r;          // epilogue -> MMA : A0 gathered                                                       (16 arrivals)
  uint64_t a1r[2];       // epilogue -> MMA : network n: layer-1 chunk packed into A1_n, slot_n drained          (16 arrivals)
  uint64_t sr[2];        // epilogue -> MMA : network n: last-layer A piece packed in slot_n                      (16 arrivals)
  uint64_t l3r[2];       // epilogue -> MMA : network n: last-layer piece product read, slot_n free               (16 arrivals)
  uint64_t l1f[2];       // MMA -> epilogue : network n: a layer-1 chunk accumulated                              (commit)
  uint64_t l2f[2];       // MMA -> epilogue : network n: a layer-2 chunk accumulated                              (commit)
  uint64_t l3f[2];       // MMA -> epilogue : network n: a last-layer piece product complete                      (commit)
  uint64_t w3full[2];    // producer -> MMA : network n's last-layer weights of this pass landed
  uint64_t w3empty[2];   // MMA -> producer : ... may be overwritten
  uint32_t tmem_base;
  uint32_t last_flag;
  float coef[kMaxComponents];
};
static_assert(sizeof(Tc5Misc) <= kT2MiscBytes, "misc region too small");

inline bool tc5_eligible(const ModelDims& md, const std::vector<StepDesc>& steps) {
  if (!tc2_eligible(md, steps) || steps.empty()) return false;
  if (md.h != 256 || md.nnets != 2 || md.kind != GBNF_KIND_REALNVP || md.act != GBNF_ACT_TANH) return false;
  const StepDesc& s0 = steps[0];
  for (const StepDesc& s : steps)
    for (int n = 0; n < 2; ++n)
      if (s.layer[n][0].Kp != s0.layer[0][0].Kp || s.layer[n][2].Np != s0.layer[0][2].Np) return false;
  return s0.layer[0][0].Kp <= 32 && s0.layer[0][2].Np <= 64;
}

__host__ __device__ inline uint32_t t5_bias_floats(int np3) { return 2u * (512u + (uint32_t)np3); }   // b1 b2 b3 of t, then of s

inline bool tc5_make_plan(const ModelDims& md, const std::vector<StepDesc>& steps, TcPlan* p) {
  const int k0p = steps[0].layer[0][0].Kp, np3 = steps[0].layer[0][2].Np;
  auto al = [](uint32_t v) { return (v + 127u) & ~127u; };
  int out_max = 1;
  for (const StepDesc& s : steps) out_max = std::max(out_max, s.out_dim);
  p->K0p = k0p; p->out_max = out_max;
  uint32_t o = 0;
  p->off_zs = o;   o = al(o + kTcRows * md.Dv * 4);
  p->off_a0 = o;   o = al(o + (k0p / 16) * 4096);
  p->off_a1 = o;   o = al(o + 6 * kTcRows * 4);                   // per-row partial sums at a component's end
  p->off_sh = o;   o = al(o + kTcRows * md.D * 4);                 // the untransformed x tile of the unit (every component restarts from it)
  p->off_misc = o; o = al(o + kT2MiscBytes);
  p->off_bias = o; o = al(o + 2 * t5_bias_floats(np3) * 4);       // this pass | next pass
  p->off_tab = o;  o = al(o + 2 * 2 * kEpPad * 16);               // z1 | z2 tables of this step and of the next
  p->off_w3 = o;   o = al(o + 2 * 16 * (uint32_t)np3 * 32u);      // last-layer weights of t | s (all 16 k-slabs of [np3 x 16])
  p->off_ring = o;
  const uint32_t limit = 227 * 1024;
  if (o + 4 * kT2StageBytes > limit) return false;
  p->nst = std::min<int>(6, (limit - o) / kT2StageBytes);
  p->smem_bytes = o + (size_t)p->nst * kT2StageBytes;
  p->tmem_cols = 512;
  return true;
}

constexpr uint32_t kT5A1 = 0u, kT5Slot = 256u, kT5L3Tmp = 64u;    // A1_n = 128 n, slot_n = 256 + 128 n, piece product at slot_n + 64

template <int TANH_MODE>
__global__ void __launch_bounds__(kT2Threads, 1) coupling_tc5_kernel(CouplingArgs a, TcPlan plan) {
  extern __shared__ __align__(1024) unsigned char smem[];
  asm volatile(".reg .pred t5_p_full;" ::);
  const ModelDims& md = a.md;
  const int D = md.D, Dv = md.Dv, K = md.K;
  float* const zs = reinterpret_cast<float*>(smem + plan.off_zs);
  unsigned char* const A0 = smem + plan.off_a0;
  float* const part_s = reinterpret_cast<float*>(smem + plan.off_a1);
  float* const xs = reinterpret_cast<float*>(smem + plan.off_sh);
  float* const bias_s = reinterpret_cast<float*>(smem + plan.off_bias);
  float4* const tab_s = reinterpret_cast<float4*>(smem + plan.off_tab);
  Tc5Misc* const misc = reinterpret_cast<Tc5Misc*>(smem + plan.off_misc);
  unsigned char* const ring = smem + plan.off_ring;
  unsigned char* const w3buf = smem + plan.off_w3;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nst = plan.nst;
  const int k0p = __ldg(&a.steps[a.c0 * md.K].layer[0][0].Kp), np3 = __ldg(&a.steps[a.c0 * md.K].layer[0][2].Np);
  const int k0s = k0p >> 4;
  const uint32_t w3_bytes = 16u * (uint32_t)np3 * 32u;          // one network's last layer
  const uint32_t bfl = t5_bias_floats(np3);

  if (threadIdx.x == 0) {
    for (int i = 0; i < nst; ++i) { ptx::mbar_init(&misc->full[i], 1); ptx::mbar_init(&misc->empty[i], 1); }
    ptx::mbar_init(&misc->a0r, 16);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&misc->a1r[i], 16); ptx::mbar_init(&misc->sr[i], 16); ptx::mbar_init(&misc->l3r[i], 16);
      ptx::mbar_init(&misc->l1f[i], 1); ptx::mbar_init(&misc->l2f[i], 1); ptx::mbar_init(&misc->l3f[i], 1);
      ptx::mbar_init(&misc->w3full[i], 1); ptx::mbar_init(&misc->w3empty[i], 1);
    }
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
    uint32_t par = 0, npass = 0;
    int slot = 0;
    auto push = [&](const __half* src, uint32_t bytes) {
      t2_wait(&misc->empty[slot], par ^ 1u, a.error_flag, 10, lane);
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(&misc->full[slot], bytes);
        ptx::tma_bulk_g2s(ring + (size_t)slot * kT2StageBytes, src, bytes, &misc->full[slot]);
      }
      __syncwarp();
      if (++slot == nst) { slot = 0; par ^= 1u; }
    };
    for (int u = blockIdx.x; u < a.num_units; u += gridDim.x) {
      const int cb = a.c0 + (u % a.split) * a.comps_per_unit, ce = min(a.c1, cb + a.comps_per_unit);
      for (int c = cb; c < ce; ++c)
#pragma unroll 1
        for (int k = 0; k < K; ++k, ++npass) {
          const StepDesc* sd = a.steps + (c * K + k);
          const __half* w1[2]; const __half* w2[2]; const __half* w3[2];
#pragma unroll
          for (int n = 0; n < 2; ++n) {
            w1[n] = wb + __ldg(&sd->layer[n][0].w_off); w2[n] = wb + __ldg(&sd->layer[n][1].w_off); w3[n] = wb + __ldg(&sd->layer[n][2].w_off);
          }
#pragma unroll
          for (int n = 0; n < 2; ++n) push(w1[n], (uint32_t)(2 * k0s) * 4096u);          // W1 of both layer-1 chunks
#pragma unroll
          for (int n = 0; n < 2; ++n) {                                                   // last-layer weights: own buffers
            t2_wait(&misc->w3empty[n], (npass & 1u) ^ 1u, a.error_flag, 11, lane);
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(&misc->w3full[n], w3_bytes);
              ptx::tma_bulk_g2s(w3buf + (size_t)n * w3_bytes, w3[n], w3_bytes, &misc->w3full[n]);
            }
            __syncwarp();
          }
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int n = 0; n < 2; ++n) {
              const __half* base = w2[n] + (size_t)(128 * j) * 16 * 16;                   // chunk j: [16 k-slabs][128 x 16]
              push(base, 32768u);
              push(base + (size_t)8 * 2048, 32768u);
            }
        }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer =======================================================
    int nslot = 0, slot = 0;
    uint32_t npar = 0, npass = 0;
    uint32_t ph_a1 = 0, ph_sr = 0, ph_l3r = 0;           // phase bits per network
    const uint64_t a0_desc = ptx::make_smem_desc(ptx::smem_u32(A0));
    const uint64_t ring_desc = ptx::make_smem_desc(ptx::smem_u32(ring));
    const uint64_t w3_desc = ptx::make_smem_desc(ptx::smem_u32(w3buf));
    const uint32_t idesc_128 = ptx::make_idesc_f16(128, 128);
    const uint32_t idesc_o = ptx::make_idesc_f16(128, np3);
    const uint32_t b3_step = (uint32_t)np3 * 2u;
    auto test_full = [&](uint64_t* bar, uint32_t par) {
      asm volatile("mbarrier.test_wait.parity.shared::cta.b64 t5_p_full, [%0], %1;" ::"r"(ptx::smem_u32(bar)), "r"(par) : "memory");
    };
    test_full(&misc->full[0], 0u);
    auto acquire = [&]() -> uint64_t {
      slot = nslot;
      uint32_t full_ok;
      asm volatile("selp.u32 %0, 1, 0, t5_p_full;" : "=r"(full_ok));
      if (!full_ok) ptx::mbar_wait(&misc->full[slot], npar, a.error_flag, 21);
      ptx::tc_fence_after();
      if (++nslot == nst) { nslot = 0; npar ^= 1u; }
      test_full(&misc->full[nslot], npar);
      return ring_desc + (uint64_t)((uint32_t)slot * (kT2StageBytes >> 4));
    };
    auto wait_bit = [&](uint64_t* bar, uint32_t& bits, int n, int code) {
      ptx::mbar_wait(bar, (bits >> n) & 1u, a.error_flag, code);
      bits ^= 1u << n;
      ptx::tc_fence_after();
    };
    for (int u = blockIdx.x; u < a.num_units; u += gridDim.x) {
      const int cb = a.c0 + (u % a.split) * a.comps_per_unit, ce = min(a.c1, cb + a.comps_per_unit);
      for (int c = cb; c < ce; ++c)
#pragma unroll 1
        for (int k = 0; k < K; ++k, ++npass) {
          uint64_t l1_desc[2];
          int l1_slot[2];
          l1_desc[0] = acquire(); l1_slot[0] = slot;
          l1_desc[1] = acquire(); l1_slot[1] = slot;
          ptx::mbar_wait(&misc->a0r, npass & 1u, a.error_flag, 20);
          ptx::tc_fence_after();
          // ---- layer 1: chunk q of network n -> slot_n (drained by the epilogue of the previous chunk / of the previous pass) ----
#pragma unroll
          for (int q = 0; q < 2; ++q)
#pragma unroll
            for (int n = 0; n < 2; ++n) {
              if (q == 0) { if (npass > 0) wait_bit(&misc->l3r[n], ph_l3r, n, 26); }     // last piece product of the previous pass read
              else wait_bit(&misc->a1r[n], ph_a1, n, 22);                                 // chunk 0 packed, slot_n drained
              if (ptx::elect_one()) {
                const uint32_t d = tbase + kT5Slot + 128u * n;
                const uint64_t bq = l1_desc[n] + (uint64_t)(q * k0s * 256);
                for (int i = 0; i < k0s; ++i)
                  ptx::umma_f16(d, a0_desc + (uint64_t)(i * 256), bq + (uint64_t)(i * 256), idesc_128, i > 0 ? 1u : 0u);
                ptx::umma_commit(&misc->l1f[n]);
                if (q == 1) ptx::umma_commit(&misc->empty[l1_slot[n]]);
              }
              __syncwarp();
            }
          // ---- layer 2 chunk j and the last-layer piece j of both networks ----
#pragma unroll
          for (int j = 0; j < 2; ++j) {
#pragma unroll
            for (int n = 0; n < 2; ++n) {
              if (j == 0) wait_bit(&misc->a1r[n], ph_a1, n, 22);                          // A1_n complete, slot_n drained
              else wait_bit(&misc->l3r[n], ph_l3r, n, 26);                                // piece 0's product read: slot_n free
#pragma unroll
              for (int y = 0; y < 2; ++y) {
                const uint64_t bd = acquire();
                const int cur = slot;
                if (ptx::elect_one()) {
                  const uint32_t d = tbase + kT5Slot + 128u * n, at = tbase + kT5A1 + 128u * n + 64u * y;
#pragma unroll
                  for (int i = 0; i < 8; ++i) ptx::umma_f16_ts(d, at + 8u * i, bd + (uint64_t)(i * 256), idesc_128, (y > 0 || i > 0) ? 1u : 0u);
                  ptx::umma_commit(&misc->empty[cur]);
                  if (y == 1) ptx::umma_commit(&misc->l2f[n]);
                }
                __syncwarp();
              }
            }
#pragma unroll
            for (int n = 0; n < 2; ++n) {
              wait_bit(&misc->sr[n], ph_sr, n, 23);                                       // piece packed in slot_n[0, 64)
              if (j == 0) { ptx::mbar_wait(&misc->w3full[n], npass & 1u, a.error_flag, 24); ptx::tc_fence_after(); }
              if (ptx::elect_one()) {
                const uint32_t at = tbase + kT5Slot + 128u * n, d = at + kT5L3Tmp;
                const uint64_t bd = w3_desc + (uint64_t)((uint32_t)n * (w3_bytes >> 4)) + (uint64_t)((uint32_t)(8 * j) * b3_step);
                for (int i = 0; i < 8; ++i)
                  ptx::umma_f16_ts(d, at + 8u * i, bd + (uint64_t)((uint32_t)i * b3_step), idesc_o, i > 0 ? 1u : 0u);
                ptx::umma_commit(&misc->l3f[n]);
                if (j == 1) ptx::umma_commit(&misc->w3empty[n]);
              }
              __syncwarp();
            }
          }
        }
    }
  } else {
    // ===================================== epilogue / elementwise warps =====================================
    const int et = threadIdx.x - 64;
    const int warp_e = et >> 5;
    const int quad = warp & 3;
    const int g = warp_e >> 2;
    const int row = quad * 32 + lane;
    float* const zrow = zs + row * Dv;
    const uint32_t lane_base = tbase + ((uint32_t)(quad * 32) << 16);
    const int dq = (D + 3) >> 2;
    const int h0col = min(D, g * dq), h1col = min(D, (g + 1) * dq);
    const int c0 = g * 16;
    uint32_t npass = 0, ph_l1f = 0, ph_l2f = 0, ph_l3f = 0;

    // staging for a pass: biases of both networks (contiguous in fblob: b1 b2 b3 of t, then of s) and the step's two tables
    auto stage = [&](const StepDesc* sd, uint32_t buf) {
      const float* bsrc = a.fblob + __ldg(&sd->layer[0][0].b_off);
      for (int i = et; i < (int)(bfl >> 2); i += kT2EpiThreads) ptx::cp_async16(bias_s + buf * bfl + 4 * i, bsrc + 4 * i);
      if (et >= kT2EpiThreads - 2 * kEpPad) {
        const int i = et - (kT2EpiThreads - 2 * kEpPad);
        ptx::cp_async16(tab_s + buf * (2 * kEpPad) + i, reinterpret_cast<const float4*>(a.fblob + __ldg(&sd->ep_off)) + i);
      }
    };
    if (blockIdx.x < a.num_units) {
      const int cb0 = a.c0 + ((int)blockIdx.x % a.split) * a.comps_per_unit;
      stage(a.steps + cb0 * K, 0u);
    }
    for (int u = blockIdx.x; u < a.num_units; u += gridDim.x) {
      const int tile = u / a.split, cs = u - tile * a.split;
      const int cb = a.c0 + cs * a.comps_per_unit, ce = min(a.c1, cb + a.comps_per_unit);
      const long long gr = (long long)tile * kTcRows + row;
      for (int c = cb; c < ce; ++c) {
        const CompDesc* cdp = a.comps + c;
        const float2 cconst = __ldg(reinterpret_cast<const float2*>(a.fblob + a.cc_off) + c);
        const long long base_off = (md.base == GBNF_BASE_STD_NORMAL) ? 0LL : __ldg(&cdp->base_off);
        // ---- x tile: fetched from HBM once per unit (coalesced, 8 loads in flight per thread) and kept in shared memory; every
        //      component restarts from it (with K = 1 a component is one step: a global reload per component cost 2 %) ----
        if (c == cb) {
          t2_load_x_tile(xs, a, D, (long long)tile * kTcRows, et);
          t2_epi_bar();
        }
        for (int pc = h0col; pc < h1col; ++pc) zrow[pc] = xs[row * D + pc];
        if (g == 0) for (int pc = D; pc < Dv; ++pc) zrow[pc] = 0.f;
        ptx::cp_async_wait_all();
        t2_epi_bar();
        float lsum = 0.f;
#pragma unroll 1
        for (int k = 0; k < K; ++k, ++npass) {
          const StepDesc* sd = a.steps + (c * K + k);
          const uint32_t buf = npass & 1u;
          const float* bias_c = bias_s + buf * bfl;                           // [b1_t b2_t b3_t | b1_s b2_s b3_s]
          const float4* tab1 = tab_s + buf * (2 * kEpPad);
          const float4* tab2 = tab1 + kEpPad;
          const int in_dim = __ldg(&sd->in_dim), out_dim = __ldg(&sd->out_dim);
          const StepDesc* sd_next = (k + 1 < K) ? sd + 1
                                    : (c + 1 < ce) ? a.steps + (c + 1) * K
                                    : (u + (int)gridDim.x < a.num_units) ? a.steps + (a.c0 + ((u + (int)gridDim.x) % a.split) * a.comps_per_unit) * K
                                    : nullptr;
          // ---- eval-BatchNorm affine fused into the gather of z1 -> A0 (one A0 feeds both networks) ----
          // The same code as t2_gather_z1, kept inline on purpose: called through the helper, the compiler keeps the table
          // pointer live across the pass and reschedules this MUFU-bound kernel, which measured 1.5 % slower on cfg1 / cfg2
          // (NVIDIA B200, 1000 W power limit).
          {
            const int nch = k0p >> 3;
            for (int chn = g; chn < nch; chn += 4) {
              float4 t[8];
              float v[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) t[e] = tab1[chn * 8 + e];
#pragma unroll
              for (int e = 0; e < 8; ++e) v[e] = zrow[__float_as_int(t[e].w)];
#pragma unroll
              for (int e = 0; e < 8; ++e) v[e] = (v[e] + t[e].x) * t[e].y + t[e].z;
#pragma unroll
              for (int e = 0; e < 8; ++e) if (chn * 8 + e < in_dim) zrow[__float_as_int(t[e].w)] = v[e];
#pragma unroll
              for (int e = 0; e < 8; ++e) v[e] = (chn * 8 + e < in_dim) ? v[e] : 0.f;
              {
                const float mx = fmax_nan(fmax_nan(fmax_nan(fabsf(v[0]), fabsf(v[1])), fmax_nan(fabsf(v[2]), fabsf(v[3]))),
                                          fmax_nan(fmax_nan(fabsf(v[4]), fabsf(v[5])), fmax_nan(fabsf(v[6]), fabsf(v[7]))));
                if (!(mx <= 65504.f)) *reinterpret_cast<volatile int*>(a.error_flag + 2) = 1;
              }
              st_shared_v4(A0 + a_chunk_off(row, chn * 8), pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]),
                           pack_half2(v[6], v[7]));
            }
          }
          ptx::fence_proxy_async_smem();
          ptx::tc_fence_before();
          t2_warp_arrive(&misc->a0r, lane);
          if (sd_next != nullptr) stage(sd_next, buf ^ 1u);                   // next pass's biases / tables, off the critical path
          // ---- layer 1: both chunks of both networks ----
#pragma unroll 1
          for (int q = 0; q < 2; ++q)
#pragma unroll 1
            for (int n = 0; n < 2; ++n) {
              t2_wait(&misc->l1f[n], (ph_l1f >> n) & 1u, a.error_flag, 30, lane);
              ph_l1f ^= 1u << n;
              ptx::tc_fence_after();
              uint32_t pk[16];
              {
                uint32_t r[32];
                ptx::tmem_ld32(lane_base + kT5Slot + 128u * n + (uint32_t)g * 32u, r);
                ptx::tmem_ld_wait();
                t2_act_pack<1, TANH_MODE>(r, bias_c + n * (512 + np3) + q * 128 + g * 32, pk, a.error_flag);
              }
              ptx::tmem_st16(lane_base + kT5A1 + 128u * n + 64u * q + (uint32_t)g * 16u, pk);
              ptx::tmem_st_wait();
              ptx::tc_fence_before();
              t2_warp_arrive(&misc->a1r[n], lane);
            }
          // ---- layer 2 chunk j + the last-layer piece j of both networks; piece products summed in registers ----
          float acc3[2][16];
#pragma unroll
          for (int n = 0; n < 2; ++n)
#pragma unroll
            for (int i = 0; i < 16; ++i) acc3[n][i] = 0.f;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
#pragma unroll 1
            for (int n = 0; n < 2; ++n) {
              t2_wait(&misc->l2f[n], (ph_l2f >> n) & 1u, a.error_flag, 31, lane);
              ph_l2f ^= 1u << n;
              ptx::tc_fence_after();
              const uint32_t sc = lane_base + kT5Slot + 128u * n;
              uint32_t pk[16];
              {
                uint32_t r[32];
                ptx::tmem_ld32(sc + (uint32_t)g * 32u, r);
                ptx::tmem_ld_wait();
                t2_act_pack<1, TANH_MODE>(r, bias_c + n * (512 + np3) + 256 + j * 128 + g * 32, pk, a.error_flag);
              }
              t2_quad_bar(quad);
              ptx::tmem_st16(sc + (uint32_t)g * 16u, pk);
              ptx::tmem_st_wait();
              ptx::tc_fence_before();
              t2_warp_arrive(&misc->sr[n], lane);
            }
#pragma unroll
            for (int n = 0; n < 2; ++n) {
              t2_wait(&misc->l3f[n], (ph_l3f >> n) & 1u, a.error_flag, 32, lane);
              ph_l3f ^= 1u << n;
              ptx::tc_fence_after();
              if (c0 < np3) {
                uint32_t r3[16];
                ptx::tmem_ld16(lane_base + kT5Slot + 128u * n + kT5L3Tmp + (uint32_t)c0, r3);
                ptx::tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) acc3[n][i] += __uint_as_float(r3[i]);
              }
              ptx::tc_fence_before();
              t2_warp_arrive(&misc->l3r[n], lane);
            }
          }
          // ---- coupling transform (transformations.py:575-577) on this thread's 16-column slice ----
          if (c0 < np3) {
            const float* b3t = bias_c + 512;
            const float* b3s = bias_c + (512 + np3) + 512;
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
                const float shift = acc3[0][half * 8 + jj] + b3t[j];
                const float sc = acc3[1][half * 8 + jj] + b3s[j];
                const float zn = (z[jj] + t[jj].x) * t[jj].y + t[jj].z;
                z[jj] = shift + zn * __expf(sc);
                lsum += (j < out_dim) ? sc : 0.f;
              }
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) if (c0 + half * 8 + jj < out_dim) zrow[__float_as_int(t[jj].w)] = z[jj];
            }
          }
          ptx::cp_async_wait_all();
          t2_epi_bar();
        }
        // ---- component log-density for this row ----
        t2_component_logq(a, zrow, lsum, part_s, row, g, quad, h0col, h1col, Dv, base_off, cconst.x, cconst.y, misc->coef, c, tile,
                          true);
        if (a.z_out != nullptr && gr < a.B) {
          const int* sig = a.iblob + __ldg(&cdp->sigma_off);
          for (int j = h0col; j < h1col; ++j) a.z_out[gr * D + j] = zrow[__ldg(sig + j)];
        }
        t2_epi_bar();                                  // partial sums / z rows are dead before the next component overwrites them
      }
      if (a.G_ll != nullptr) t2_tile_logsumexp(a, tile, gr, g, et, &misc->last_flag);
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

inline cudaError_t tc5_configure() {
  cudaError_t e = cudaFuncSetAttribute(coupling_tc5_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(coupling_tc5_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  return e;
}

inline int tc5_launch(const CouplingArgs& a, const TcPlan& p, int grid, cudaStream_t st) {
  if (p.tanh_mode == 0) coupling_tc5_kernel<0><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p);
  else                  coupling_tc5_kernel<1><<<grid, kT2Threads, p.smem_bytes, st>>>(a, p);
  return 0;
}

}  // namespace gbnf
