// tcgen05 / TMEM / bulk-TMA coupling-stack kernel (GBNF_GEMM_F16_TC*).
//
// One persistent CTA per SM owns a 128-row tile and walks components x coupling steps x MLP layers with the rows
// resident on chip:
//   z            fp32 [128][Dv]      shared memory, never permuted physically (gather indices resolved at pack time)
//   A0           fp16 [128][K0p]     shared, UMMA canonical K-major no-swizzle image of z1 (layer-0 A operand)
//   A1           fp16 [128][h]       shared, same layout; activations of the hidden layers, rewritten in place
//   accumulators fp32 [128][<=512]   TMEM (tcgen05.mma D), read back by the epilogue warps with tcgen05.ld
//   weights      fp16 k-slabs        streamed L2 -> shared by bulk TMA (cp.async.bulk + mbarrier complete_tx) through a
//                                    ring of 16 KB stages; every CTA walks the components in the same order so the
//                                    packed blob stays L2-resident
// Warp roles: warp 0 = TMA producer (one lane), warp 1 = MMA issuer (one lane; owns the TMEM allocation),
// warps 2..9 = 8 epilogue warps (two threads per row, splitting the columns): bias + activation + fp16 repack of the
// hidden layers, the coupling transform, log-det, base density and the online logsumexp over components.
// Nothing but x (in) and log q / G_ll (out) touches HBM.
#pragma once
#include <string>
#include <vector>
#include "common.cuh"
#include "tc_ptx.cuh"

namespace gbnf {

constexpr int kTcThreads = 320;          // 2 control warps + 8 epilogue warps
constexpr int kTcEpiThreads = 256;
constexpr int kTcRows = 128;
constexpr uint32_t kTcStageBytes = 16384;
constexpr int kTcMaxStages = 8;
constexpr int kTcMaxD = 64;

struct TcPlan {
  int nst = 0;                 // ring stages
  int K0p = 0;                 // padded layer-0 K (max over steps)
  int out_max = 0;
  int tanh_mode = 1;           // 0: MUFU.TANH (tanh.approx.f32), 1: 1 - 2/(1+2^(2x log2 e)) via ex2.approx + rcp.approx
  uint32_t off_zs = 0, off_a0 = 0, off_a1 = 0, off_ring = 0, off_sh = 0, off_misc = 0, off_bias = 0, off_tab = 0, off_w3 = 0;
  size_t smem_bytes = 0;
  int tmem_cols = 512;
};

// misc region layout (bytes from off_misc)
struct TcMisc {
  uint64_t full[kTcMaxStages];
  uint64_t empty[kTcMaxStages];
  uint64_t acc_full;
  uint64_t a_ready;
  uint32_t tmem_base;
  uint32_t pad_;
  float coef[kMaxComponents];
  float part[kTcRows];
};

constexpr uint32_t kTcMiscBytes = 5120;   // >= sizeof(TcMisc), sizeof(Tc2Misc)
static_assert(sizeof(TcMisc) <= kTcMiscBytes, "misc region too small");

inline bool tc_make_plan(const ModelDims& md, const std::vector<StepDesc>& steps, TcPlan* p, std::string* why) {
  if (md.h % 64 != 0 || md.h > 512) {
    *why = "hidden width must be <= 512, or <= 1024 with coupling_network_depth 1 and D <= 64 (use GBNF_GEMM_FP32 otherwise)";
    return false;
  }
  if (md.D > kTcMaxD) { *why = "D must be <= 64"; return false; }
  int k0p = 16, out_max = 1;
  for (const StepDesc& s : steps) {
    k0p = std::max(k0p, s.layer[0][0].Kp);
    out_max = std::max(out_max, s.out_dim);
    for (int n = 0; n < md.nnets; ++n)
      for (int l = 0; l < md.nlayers; ++l)
        if (s.layer[n][l].Np > 512) { *why = "layer wider than 512 columns"; return false; }
  }
  auto al = [](uint32_t v) { return (v + 127u) & ~127u; };
  p->K0p = k0p; p->out_max = out_max;
  uint32_t o = 0;
  p->off_zs = o;   o = al(o + kTcRows * md.Dv * 4);
  p->off_a0 = o;   o = al(o + (k0p / 16) * 4096);
  p->off_a1 = o;   o = al(o + (md.h / 16) * 4096);
  p->off_sh = o;   o = al(o + (md.nnets == 2 ? kTcRows * out_max * 4 : 0));
  p->off_misc = o; o = al(o + kTcMiscBytes);
  p->off_ring = o;
  const uint32_t limit = 227 * 1024;
  if (o + 2 * kTcStageBytes > limit) { *why = "shared memory budget exceeded"; return false; }
  p->nst = std::min<int>(kTcMaxStages, (limit - o) / kTcStageBytes);
  p->smem_bytes = o + (size_t)p->nst * kTcStageBytes;
  p->tmem_cols = 512;
  return true;
}

// ---- activation / transcendental helpers -------------------------------------------------------------------
template <int TANH_MODE>
__device__ __forceinline__ float tc_tanh(float v) {
  if (TANH_MODE == 0) {
    float r;
    asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
  } else {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(v * 2.8853900817779268f));   // e^(2v)
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
  }
}
template <int ACT, int TANH_MODE>   // ACT: 1 tanh, 2 relu
__device__ __forceinline__ float tc_act(float v) {
  return ACT == 1 ? tc_tanh<TANH_MODE>(v) : fmaxf(v, 0.f);
}
// NaN-propagating maximum (fmaxf returns the non-NaN operand): used by the "finite in fp16" checks
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float fmin_nan(float a, float b) {
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
// Four activations of one row at once.  The accurate tanh costs two MUFU operations per value (ex2 + rcp), and the MUFU pipe
// (16 / clk / SM) is what bounds the accurate mode: one reciprocal serves four values (1 / (a0 a1 a2 a3), then the partial
// products give each 1 / a_i back) -> 1.25 MUFU + 2.5 FMA-pipe operations per value instead of 2 + 1.  a_i = e^(2 v_i) + 1 with
// 2 v_i capped at 20 (tanh(10) rounds to 1 in fp32), so the product of four stays below 5.5e34; NaN passes the cap (min.NaN)
// and poisons only values of the same row; v = -inf gives a = 1 -> -1.  Error: 3 ulp on 1 / a_i -> < 4e-7 absolute on tanh.
template <int ACT, int TANH_MODE>
__device__ __forceinline__ void tc_act4(float& v0, float& v1, float& v2, float& v3) {
  if (ACT == 1 && TANH_MODE != 0) {
    const float c = 2.8853900817779268f, cap = 28.853900817779268f;
    float e0, e1, e2, e3, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fmin_nan(v0 * c, cap)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fmin_nan(v1 * c, cap)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2) : "f"(fmin_nan(v2 * c, cap)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e3) : "f"(fmin_nan(v3 * c, cap)));
    const float a0 = e0 + 1.0f, a1 = e1 + 1.0f, a2 = e2 + 1.0f, a3 = e3 + 1.0f;
    const float p01 = a0 * a1, p23 = a2 * a3;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p01 * p23));
    const float rm = -2.0f * r, r01 = rm * p23, r23 = rm * p01;          // -2 / (a0 a1), -2 / (a2 a3)
    v0 = fmaf(r01, a1, 1.0f);
    v1 = fmaf(r01, a0, 1.0f);
    v2 = fmaf(r23, a3, 1.0f);
    v3 = fmaf(r23, a2, 1.0f);
  } else {
    v0 = tc_act<ACT, TANH_MODE>(v0);
    v1 = tc_act<ACT, TANH_MODE>(v1);
    v2 = tc_act<ACT, TANH_MODE>(v2);
    v3 = tc_act<ACT, TANH_MODE>(v3);
  }
}
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void st_shared_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(ptx::smem_u32(p)), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// byte offset of the 16-byte k-chunk holding elements [k8, k8+8) of `row` in a canonical K-major A image
__device__ __forceinline__ uint32_t a_chunk_off(int row, int k8) {
  return (uint32_t)((k8 >> 4) * 4096 + (row >> 3) * 256 + ((k8 >> 3) & 1) * 128 + (row & 7) * 16);
}

// hidden layer epilogue: TMEM accumulator -> +bias -> act -> fp16 -> A1 (this thread's half of the columns)
template <int ACT, int TANH_MODE>
__device__ __forceinline__ void tc_hidden_epilogue(uint32_t tbase, int quad, int row, int hsel, int Np,
                                                   const float* __restrict__ bias, unsigned char* A1, int* status) {
  const int half = Np >> 1;
  const uint32_t lane_base = tbase + ((uint32_t)(quad * 32) << 16);
  for (int c0 = hsel * half; c0 < (hsel + 1) * half; c0 += 32) {
    uint32_t r[32];
    ptx::tmem_ld32(lane_base + (uint32_t)c0, r);
    ptx::tmem_ld_wait();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + c0 + 8 * q));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + c0 + 8 * q + 4));
      float v0 = __uint_as_float(r[8 * q + 0]) + b0.x, v1 = __uint_as_float(r[8 * q + 1]) + b0.y;
      float v2 = __uint_as_float(r[8 * q + 2]) + b0.z, v3 = __uint_as_float(r[8 * q + 3]) + b0.w;
      float v4 = __uint_as_float(r[8 * q + 4]) + b1.x, v5 = __uint_as_float(r[8 * q + 5]) + b1.y;
      float v6 = __uint_as_float(r[8 * q + 6]) + b1.z, v7 = __uint_as_float(r[8 * q + 7]) + b1.w;
      tc_act4<ACT, TANH_MODE>(v0, v1, v2, v3);
      tc_act4<ACT, TANH_MODE>(v4, v5, v6, v7);
      if (ACT == 2 && !(fmax_nan(fmax_nan(fmax_nan(v0, v1), fmax_nan(v2, v3)), fmax_nan(fmax_nan(v4, v5), fmax_nan(v6, v7))) <= 65504.f))
        *reinterpret_cast<volatile int*>(status + 2) = 1;                           // ReLU activation not finite in fp16
      st_shared_v4(A1 + a_chunk_off(row, c0 + 8 * q), pack_half2(v0, v1), pack_half2(v2, v3), pack_half2(v4, v5),
                   pack_half2(v6, v7));
    }
  }
}

template <int TANH_MODE>
__global__ void __launch_bounds__(kTcThreads, 1) coupling_tc_kernel(CouplingArgs a, TcPlan plan) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const ModelDims& md = a.md;
  const int D = md.D, Dv = md.Dv;
  float* zs = reinterpret_cast<float*>(smem + plan.off_zs);
  unsigned char* A0 = smem + plan.off_a0;
  unsigned char* A1 = smem + plan.off_a1;
  float* sh = reinterpret_cast<float*>(smem + plan.off_sh);
  TcMisc* misc = reinterpret_cast<TcMisc*>(smem + plan.off_misc);
  unsigned char* ring = smem + plan.off_ring;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nst = plan.nst;

  if (threadIdx.x == 0) {
    for (int i = 0; i < nst; ++i) { ptx::mbar_init(&misc->full[i], 1); ptx::mbar_init(&misc->empty[i], 1); }
    ptx::mbar_init(&misc->acc_full, 1);
    ptx::mbar_init(&misc->a_ready, kTcEpiThreads);
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
    if (lane == 0) {
      uint32_t sidx = 0;
      const long long p_t0 = clock64();
      long long p_wait = 0;
      for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x)
        for (int c = a.c0; c < a.c1; ++c)
          for (int k = 0; k < md.K; ++k) {
            const StepDesc& sd = a.steps[c * md.K + k];
            for (int net = 0; net < md.nnets; ++net)
              for (int l = 0; l < md.nlayers; ++l) {
                const LayerDesc& L = sd.layer[net][l];
                const uint32_t slab_bytes = (uint32_t)L.Np * 32u;
                const int nslabs = L.Kp >> 4;
                const int sps = min(nslabs, max(1, (int)(kTcStageBytes / slab_bytes)));
                for (int s0 = 0; s0 < nslabs; s0 += sps, ++sidx) {
                  const int n = min(sps, nslabs - s0);
                  const int slot = sidx % nst;
                  const uint32_t par = (sidx / nst) & 1u;
                  const long long tw = clock64();
                  ptx::mbar_wait(&misc->empty[slot], par ^ 1u, a.error_flag, 10);
                  p_wait += clock64() - tw;
                  const uint32_t bytes = (uint32_t)n * slab_bytes;
                  ptx::mbar_arrive_expect_tx(&misc->full[slot], bytes);
                  ptx::tma_bulk_g2s(ring + (size_t)slot * kTcStageBytes, wb + L.w_off + (long long)s0 * L.Np * 16, bytes,
                                    &misc->full[slot]);
                }
              }
          }
      if (a.prof != nullptr && blockIdx.x == 0) { a.prof[16] = clock64() - p_t0; a.prof[17] = p_wait; a.prof[18] = sidx; }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer =======================================================
    if (lane == 0) {
      uint32_t sidx = 0, lcount = 0;
      const long long m_t0 = clock64();
      long long m_wa = 0, m_wf = 0;
      const uint32_t a0_addr = ptx::smem_u32(A0), a1_addr = ptx::smem_u32(A1), ring_addr = ptx::smem_u32(ring);
      for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x)
        for (int c = a.c0; c < a.c1; ++c)
          for (int k = 0; k < md.K; ++k) {
            const StepDesc& sd = a.steps[c * md.K + k];
            for (int net = 0; net < md.nnets; ++net)
              for (int l = 0; l < md.nlayers; ++l, ++lcount) {
                const LayerDesc& L = sd.layer[net][l];
                const uint32_t slab_bytes = (uint32_t)L.Np * 32u;
                const int nslabs = L.Kp >> 4;
                const int sps = min(nslabs, max(1, (int)(kTcStageBytes / slab_bytes)));
                const uint32_t a_addr = (l == 0) ? a0_addr : a1_addr;
                long long tw = clock64();
                ptx::mbar_wait(&misc->a_ready, lcount & 1u, a.error_flag, 20);   // A operand written, TMEM drained
                m_wa += clock64() - tw;
                ptx::tc_fence_after();
                for (int s0 = 0; s0 < nslabs; s0 += sps, ++sidx) {
                  const int n = min(sps, nslabs - s0);
                  const int slot = sidx % nst;
                  const uint32_t par = (sidx / nst) & 1u;
                  tw = clock64();
                  ptx::mbar_wait(&misc->full[slot], par, a.error_flag, 21);
                  m_wf += clock64() - tw;
                  ptx::tc_fence_after();
                  const uint32_t stage_addr = ring_addr + (uint32_t)slot * kTcStageBytes;
                  for (int i = 0; i < n; ++i) {
                    const int kidx = s0 + i;
                    const uint64_t adesc = ptx::make_smem_desc(a_addr + (uint32_t)kidx * 4096u);
                    for (int n0 = 0; n0 < L.Np; n0 += 256) {
                      const int nc = min(256, L.Np - n0);
                      const uint64_t bdesc = ptx::make_smem_desc(stage_addr + (uint32_t)i * slab_bytes + (uint32_t)n0 * 32u);
                      ptx::umma_f16(tbase + (uint32_t)n0, adesc, bdesc, ptx::make_idesc_f16(128, nc), kidx > 0 ? 1u : 0u);
                    }
                  }
                  ptx::umma_commit(&misc->empty[slot]);          // ring slot reusable once these MMAs retire
                }
                ptx::umma_commit(&misc->acc_full);               // accumulator of this layer complete
              }
          }
      if (a.prof != nullptr && blockIdx.x == 0) {
        a.prof[0] = clock64() - m_t0; a.prof[1] = m_wa; a.prof[2] = m_wf; a.prof[3] = lcount;
      }
    }
  } else {
    // ===================================== epilogue / elementwise warps =====================================
    const int et = threadIdx.x - 64;
    const int warp_e = et >> 5;
    const int quad = warp & 3;             // TMEM lane quadrant this warp may access
    const int hsel = warp_e >> 2;          // which half of the columns
    const int row = quad * 32 + lane;
    const int h0col = hsel == 0 ? 0 : (D + 1) / 2, h1col = hsel == 0 ? (D + 1) / 2 : D;   // column split for elementwise passes
    uint32_t lcount = 0;
    const long long e_t0 = clock64();
    long long e_wacc = 0, e_hid = 0, e_last = 0, e_pro = 0, e_tmp;
    for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x) {
      const long long row0 = (long long)tile * kTcRows;
      const long long gr = row0 + row;
      OnlineLse lse; lse.init();
      for (int c = a.c0; c < a.c1; ++c) {
        // ---- load the x tile (coalesced over the flat tile) ----
        e_tmp = clock64();
        epi_bar();                                   // previous component's readers are done with zs
        for (int i = et; i < kTcRows * D; i += kTcEpiThreads) {
          const int r = i / D, j = i - r * D;
          const long long g = row0 + r;
          zs[r * Dv + j] = (g < a.B) ? __ldg(a.x + g * D + j) : 0.f;
        }
        epi_bar();
        e_pro += clock64() - e_tmp;
        float ldj = 0.f;
        for (int k = 0; k < md.K; ++k) {
          e_tmp = clock64();
          const StepDesc& sd = a.steps[c * md.K + k];
          const float* add = a.fblob + sd.vec_off;
          const float* mul = add + Dv;
          const float* off = mul + Dv;
          const int* idx1 = a.iblob + sd.idx_off;
          const int* idx2 = idx1 + sd.in_dim;
          // ---- ActNorm / eval-BatchNorm affine on this thread's half of its row ----
          if (sd.has_affine) {
            for (int p = h0col; p < h1col; ++p) zs[row * Dv + p] = (zs[row * Dv + p] + __ldg(add + p)) * __ldg(mul + p) + __ldg(off + p);
            epi_bar();
          }
          // ---- gather z1 -> A0 (fp16, canonical layout), zero padded to K0p ----
          {
            const int K0p = sd.layer[0][0].Kp;
            const int nch = K0p >> 3;                // 8-element chunks
            for (int ch = hsel; ch < nch; ch += 2) {
              float v[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int j = ch * 8 + e;
                v[e] = (j < sd.in_dim) ? zs[row * Dv + __ldg(idx1 + j)] : 0.f;
                if (!(fabsf(v[e]) <= 65504.f)) *reinterpret_cast<volatile int*>(a.error_flag + 2) = 1;   // not finite in fp16
              }
              st_shared_v4(A0 + a_chunk_off(row, ch * 8), pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]),
                           pack_half2(v[6], v[7]));
            }
          }
          e_pro += clock64() - e_tmp;
          for (int net = 0; net < md.nnets; ++net) {
            const int act_kind = (md.act == GBNF_ACT_TANH) ? 1 : (md.act == GBNF_ACT_RELU) ? 2 : (net == 0 ? 2 : 1);
            for (int l = 0; l < md.nlayers; ++l, ++lcount) {
              const LayerDesc& L = sd.layer[net][l];
              // hand the A operand (and the drained TMEM) to the MMA warp
              ptx::fence_proxy_async_smem();
              ptx::tc_fence_before();
              ptx::mbar_arrive(&misc->a_ready);
              e_tmp = clock64();
              ptx::mbar_wait(&misc->acc_full, lcount & 1u, a.error_flag, 30);
              e_wacc += clock64() - e_tmp;
              ptx::tc_fence_after();
              e_tmp = clock64();
              const float* bias = a.fblob + L.b_off;
              if (l < md.nlayers - 1) {
                if (act_kind == 1) tc_hidden_epilogue<1, TANH_MODE>(tbase, quad, row, hsel, L.Np, bias, A1, a.error_flag);
                else               tc_hidden_epilogue<2, TANH_MODE>(tbase, quad, row, hsel, L.Np, bias, A1, a.error_flag);
                e_hid += clock64() - e_tmp;
              } else {
                // ---- last layer: coupling transform on this thread's 32-column slice ----
                float lsum = 0.f;
                const int c0 = hsel * 32;
                if (c0 < L.Np) {
                  uint32_t r[32];
                  ptx::tmem_ld32(tbase + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, r);
                  ptx::tmem_ld_wait();
                  if (md.kind == GBNF_KIND_GLOW && md.coupling == GBNF_COUPLING_AFFINE) {
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) {
                      const int j = hsel * 16 + jj;
                      if (j < sd.out_dim) {
                        const float shift = __uint_as_float(r[2 * jj]) + __ldg(bias + 2 * j);
                        const float raw = __uint_as_float(r[2 * jj + 1]) + __ldg(bias + 2 * j + 1);
                        const float s = 1.0f / (1.0f + __expf(-(raw + 2.0f)));        // sigmoid(raw + 2), glow.py:333
                        float* zp = zs + row * Dv + __ldg(idx2 + j);
                        *zp = (*zp + shift) * s;
                        lsum += __logf(s);                                             // glow.py:338
                      }
                    }
                  } else if (md.kind == GBNF_KIND_GLOW) {
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) {
                      const int j = c0 + jj;
                      if (j < sd.out_dim) zs[row * Dv + __ldg(idx2 + j)] += __uint_as_float(r[jj]) + __ldg(bias + j);
                    }
                  } else if (net == 0) {                                               // RealNVP t_net: keep the shift
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) {
                      const int j = c0 + jj;
                      if (j < sd.out_dim) sh[row * plan.out_max + j] = __uint_as_float(r[jj]) + __ldg(bias + j);
                    }
                  } else {                                                             // RealNVP s_net: transform
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) {
                      const int j = c0 + jj;
                      if (j < sd.out_dim) {
                        const float sc = __uint_as_float(r[jj]) + __ldg(bias + j);
                        float* zp = zs + row * Dv + __ldg(idx2 + j);
                        *zp = sh[row * plan.out_max + j] + *zp * __expf(sc);           // transformations.py:575
                        lsum += sc;                                                    // transformations.py:577
                      }
                    }
                  }
                }
                if (net == md.nnets - 1) {
                  if (hsel == 1) misc->part[row] = lsum;
                  epi_bar();                       // z2 updates + partial log-dets visible to the row's other thread
                  if (hsel == 0) ldj += lsum + misc->part[row];
                  epi_bar();                       // part[] may be rewritten
                }
                e_last += clock64() - e_tmp;
              }
            }
          }
        }
        // ---- component log-density for this row ----
        const CompDesc& cd = a.comps[c];
        const float* bm = a.fblob + cd.base_off;
        const float* bi = bm + Dv;
        float q = 0.f;
        for (int p = h0col; p < h1col; ++p) { const float d = zs[row * Dv + p] - __ldg(bm + p); q = fmaf(d * d, __ldg(bi + p), q); }
        if (hsel == 1) misc->part[row] = q;
        epi_bar();
        if (hsel == 0) {
          q += misc->part[row];
          const float ldj_tot = ldj + __ldg(a.fblob + cd.const_off);
          const float lq = (__ldg(bm + 2 * Dv) - q) + ldj_tot;
          if (gr < a.B) {
            if (a.logq) a.logq[gr * a.ld_logq + (c - a.c0)] = lq;
            if (a.ldj_out) a.ldj_out[gr] = ldj_tot;
          }
          if (a.G_ll != nullptr && c < a.n_mix) lse.add(misc->coef[c] + lq);
        }
        if (a.z_out != nullptr && gr < a.B) {
          const int* sig = a.iblob + cd.sigma_off;
          for (int j = h0col; j < h1col; ++j) a.z_out[gr * D + j] = zs[row * Dv + __ldg(sig + j)];
        }
      }
      if (a.G_ll != nullptr && hsel == 0 && gr < a.B) a.G_ll[gr] = lse.value();
    }
    if (a.prof != nullptr && blockIdx.x == 0 && et == 0) {
      a.prof[8] = clock64() - e_t0; a.prof[9] = e_wacc; a.prof[10] = e_hid; a.prof[11] = e_last; a.prof[12] = e_pro;
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

inline cudaError_t tc_configure(const TcPlan&) {
  // per-function attribute shared by every handle in the process: always the device maximum
  cudaError_t e = cudaFuncSetAttribute(coupling_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(coupling_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

inline int tc_launch(const CouplingArgs& a, const TcPlan& p, int grid, cudaStream_t st) {
  if (p.tanh_mode == 0) coupling_tc_kernel<0><<<grid, kTcThreads, p.smem_bytes, st>>>(a, p);
  else                  coupling_tc_kernel<1><<<grid, kTcThreads, p.smem_bytes, st>>>(a, p);
  return 0;
}

}  // namespace gbnf
