// fp32 CUDA-core coupling-stack kernel (GBNF_GEMM_FP32): reference-class numerics, used as the exact mode and as
// the on-device cross-check of the tensor-core path.  One CTA owns R resident rows and walks components x steps;
// activations never leave shared memory, weights stream from L2 in [32 x 64] fp32 tiles via cp.async.
#pragma once
#include "common.cuh"

namespace gbnf {

constexpr int kF32Threads = 256;
constexpr int kF32KT = 32;   // k-tile
constexpr int kF32NT = 64;   // n-tile

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

template <int ACT>
__device__ __forceinline__ float apply_act(float v) {
  if (ACT == 1) return tanhf(v);
  if (ACT == 2) return fmaxf(v, 0.f);
  return v;
}

// out[r][n] = act( sum_k in[r][k] * Wt[k][n] + bias[n] )  for r < R, n < Np.   in/out: shared, row stride ld.
// 256 threads as 16 (rows) x 16 (cols); each thread owns TM = R/16 rows x 4 columns of a 64-column chunk.
// IN_RELU: the input is read through max(., 0) (pre-activation residual blocks); ACCUM: out += result (the block's skip; out != in).
template <int R, int ACT, bool IN_RELU = false, bool ACCUM = false>
__device__ void gemm_layer_fp32(const float* __restrict__ in, float* __restrict__ out, int ld,
                                const float* __restrict__ Wt, const float* __restrict__ bias, int Kp, int Np,
                                float* __restrict__ Ws /* [2][32][64] */) {
  constexpr int TM = R / 16;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int nk = Kp / kF32KT;
  for (int n0 = 0; n0 < Np; n0 += kF32NT) {
    float acc[TM][4];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    // tile (kt): Wt[kt*32 .. +32][n0 .. n0+64]  -> Ws[buf][32][64]; 512 x 16B chunks, 2 per thread
    auto issue = [&](int kt, int buf) {
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        int chunk = tid + q * kF32Threads;          // 0..511
        int kr = chunk >> 4, nc = (chunk & 15) * 4;
        cp_async16(Ws + (buf * kF32KT + kr) * kF32NT + nc, Wt + (long long)(kt * kF32KT + kr) * Np + n0 + nc);
      }
      cp_async_commit();
    };
    issue(0, 0);
    for (int kt = 0; kt < nk; ++kt) {
      const int buf = kt & 1;
      if (kt + 1 < nk) { issue(kt + 1, buf ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
      __syncthreads();
      const float* wsb = Ws + buf * kF32KT * kF32NT;
#pragma unroll
      for (int kk = 0; kk < kF32KT; kk += 4) {
        float4 a[TM];
#pragma unroll
        for (int i = 0; i < TM; ++i) {
          a[i] = *reinterpret_cast<const float4*>(in + (ty * TM + i) * ld + kt * kF32KT + kk);
          if (IN_RELU) { a[i].x = fmaxf(a[i].x, 0.f); a[i].y = fmaxf(a[i].y, 0.f); a[i].z = fmaxf(a[i].z, 0.f); a[i].w = fmaxf(a[i].w, 0.f); }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 b = *reinterpret_cast<const float4*>(wsb + (kk + q) * kF32NT + tx * 4);
#pragma unroll
          for (int i = 0; i < TM; ++i) {
            const float av = q == 0 ? a[i].x : q == 1 ? a[i].y : q == 2 ? a[i].z : a[i].w;
            acc[i][0] = fmaf(av, b.x, acc[i][0]);
            acc[i][1] = fmaf(av, b.y, acc[i][1]);
            acc[i][2] = fmaf(av, b.z, acc[i][2]);
            acc[i][3] = fmaf(av, b.w, acc[i][3]);
          }
        }
      }
      __syncthreads();
    }
    const float4 bv = *reinterpret_cast<const float4*>(bias + n0 + tx * 4);
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      float4 o;
      o.x = apply_act<ACT>(acc[i][0] + bv.x);
      o.y = apply_act<ACT>(acc[i][1] + bv.y);
      o.z = apply_act<ACT>(acc[i][2] + bv.z);
      o.w = apply_act<ACT>(acc[i][3] + bv.w);
      if (ACCUM) {
        const float4 p = *reinterpret_cast<const float4*>(out + (ty * TM + i) * ld + n0 + tx * 4);
        o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
      }
      *reinterpret_cast<float4*>(out + (ty * TM + i) * ld + n0 + tx * 4) = o;
    }
  }
  __syncthreads();
}

// Dense D x D step (InvertibleConv1x1 on feature vectors, models/layers.py:781-796): zs[:, 0:D] <- zs[:, 0:D] . M through the
// activation buffers; M = Wt[Kp][Np] in the GEMM layout with the lazy permutation folded in at pack time (pack_meta_kernel).
template <int R>
__device__ void dense_step_fp32(float* zs, int Dv, int D, const float* M, const float* zero_bias, int Kp, int Np,
                                float* act0, float* act1, int ld, float* Ws) {
  for (int i = threadIdx.x; i < R * Kp; i += blockDim.x) {
    int r = i / Kp, j = i % Kp;
    act0[r * ld + j] = (j < D) ? zs[r * Dv + j] : 0.f;
  }
  __syncthreads();
  gemm_layer_fp32<R, 0>(act0, act1, ld, M, zero_bias, Kp, Np, Ws);
  for (int i = threadIdx.x; i < R * D; i += blockDim.x) {
    int r = i / D, j = i % D;
    zs[r * Dv + j] = act1[r * ld + j];
  }
  __syncthreads();
}

template <int R>
__device__ void run_net_fp32(const StepDesc& sd, int net, int act_kind, int nlayers, const CouplingArgs& a,
                             float* act0, float* act1, int ld, float* Ws) {
  // layer 0: act0 -> act1 ; hidden layers ping-pong ; result of the last layer is left in `act1`
  const float* wb = reinterpret_cast<const float*>(a.wblob);
  if (act_kind == 3) {
    // ResidualNet (models/layers.py:246-301): t = initial(x); per block t += second(relu(first(relu(t)))); out = final(t).
    // t lives in act1 (updated in place by the accumulating GEMM), the block's hidden activation in act0.
    const LayerDesc& L0 = sd.layer[net][0];
    gemm_layer_fp32<R, 0>(act0, act1, ld, wb + L0.w_off, a.fblob + L0.b_off, L0.Kp, L0.Np, Ws);
    for (int l = 1; l + 1 < nlayers; l += 2) {
      const LayerDesc& La = sd.layer[net][l];
      const LayerDesc& Lb = sd.layer[net][l + 1];
      gemm_layer_fp32<R, 2, true>(act1, act0, ld, wb + La.w_off, a.fblob + La.b_off, La.Kp, La.Np, Ws);
      gemm_layer_fp32<R, 0, false, true>(act0, act1, ld, wb + Lb.w_off, a.fblob + Lb.b_off, Lb.Kp, Lb.Np, Ws);
    }
    const LayerDesc& Lf = sd.layer[net][nlayers - 1];
    gemm_layer_fp32<R, 0>(act1, act0, ld, wb + Lf.w_off, a.fblob + Lf.b_off, Lf.Kp, Lf.Np, Ws);
    for (int i = threadIdx.x; i < R * Lf.Np; i += blockDim.x) {
      int r = i / Lf.Np, n = i % Lf.Np;
      act1[r * ld + n] = act0[r * ld + n];
    }
    __syncthreads();
    return;
  }
  float* src = act0;
  float* dst = act1;
  for (int l = 0; l < nlayers; ++l) {
    const LayerDesc& L = sd.layer[net][l];
    const bool last = (l == nlayers - 1);
    if (last)               gemm_layer_fp32<R, 0>(src, dst, ld, wb + L.w_off, a.fblob + L.b_off, L.Kp, L.Np, Ws);
    else if (act_kind == 1) gemm_layer_fp32<R, 1>(src, dst, ld, wb + L.w_off, a.fblob + L.b_off, L.Kp, L.Np, Ws);
    else                    gemm_layer_fp32<R, 2>(src, dst, ld, wb + L.w_off, a.fblob + L.b_off, L.Kp, L.Np, Ws);
    float* t = src; src = dst; dst = t;
  }
  // after the loop `src` holds the output; make sure it is act1 (copy if the layer count left it in act0)
  if (src != act1) {
    const LayerDesc& L = sd.layer[net][nlayers - 1];
    for (int i = threadIdx.x; i < R * L.Np; i += blockDim.x) {
      int r = i / L.Np, n = i % L.Np;
      act1[r * ld + n] = act0[r * ld + n];
    }
    __syncthreads();
  }
}

// Dynamic smem: zs[R][Dv] | act0[R][ld] | act1[R][ld] | Ws[2][32][64] | sh[R][out_max] | coef[C] | rowacc[R][4]
template <int R>
__global__ void __launch_bounds__(kF32Threads, 1) coupling_fp32_kernel(CouplingArgs a, int ld, int out_max) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ModelDims& md = a.md;
  const int D = md.D, Dv = md.Dv;
  float* zs = reinterpret_cast<float*>(smem_raw);
  float* act0 = zs + ((R * Dv + 3) & ~3);
  float* act1 = act0 + R * ld;
  float* Ws = act1 + R * ld;
  float* sh = Ws + 2 * kF32KT * kF32NT;
  float* coef = sh + R * out_max;
  float* ldj = coef + kMaxComponents;   // [R]
  float* lse_m = ldj + R;               // [R]
  float* lse_s = lse_m + R;             // [R]
  const int tid = threadIdx.x;

  if (a.G_ll != nullptr) {
    if (tid == 0) mixture_coefficients(a.rho, a.n_mix, a.skip_c, a.mix_mode, coef);
    __syncthreads();
  }

  for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x) {
    const long long row0 = (long long)tile * R;
    if (tid < R) { lse_m[tid] = -INFINITY; lse_s[tid] = 0.f; }
    for (int c = a.c0; c < a.c1; ++c) {
      // load x tile (coalesced over the flat tile) into zs
      for (int i = tid; i < R * D; i += kF32Threads) {
        int r = i / D, j = i % D;
        long long gr = row0 + r;
        zs[r * Dv + j] = (gr < a.B) ? a.x[gr * D + j] : 0.f;
      }
      if (tid < R) ldj[tid] = 0.f;
      __syncthreads();
      for (int k = 0; k < md.K; ++k) {
        const StepDesc& sd = a.steps[c * md.K + k];
        const float* add = a.fblob + sd.vec_off;
        const float* mul = add + Dv;
        const float* off = mul + Dv;
        const int* idx1 = a.iblob + sd.idx_off;
        const int* idx2 = idx1 + sd.in_dim;
        if (sd.has_affine) {
          for (int i = tid; i < R * D; i += kF32Threads) {
            int r = i / D, p = i % D;
            zs[r * Dv + p] = (zs[r * Dv + p] + add[p]) * mul[p] + off[p];
          }
          __syncthreads();
        }
        if (sd.has_invconv)
          dense_step_fp32<R>(zs, Dv, D, reinterpret_cast<const float*>(a.wblob) + sd.icw_off, a.fblob + sd.icb_off, sd.ic_Kp, sd.ic_Np,
                             act0, act1, ld, Ws);
        const int Kp0 = sd.layer[0][0].Kp;
        for (int net = 0; net < md.nnets; ++net) {
          for (int i = tid; i < R * Kp0; i += kF32Threads) {
            int r = i / Kp0, j = i % Kp0;
            act0[r * ld + j] = (j < sd.in_dim) ? zs[r * Dv + idx1[j]] : 0.f;
          }
          __syncthreads();
          int act_kind = (md.act == GBNF_ACT_TANH) ? 1 : (md.act == GBNF_ACT_RELU) ? 2 : (md.act == GBNF_ACT_RESIDUAL) ? 3 : (net == 0 ? 2 : 1);
          run_net_fp32<R>(sd, net, act_kind, md.nlayers, a, act0, act1, ld, Ws);
          if (md.nnets == 2 && net == 0) {   // keep t_net output (shift) while s_net runs
            for (int i = tid; i < R * sd.out_dim; i += kF32Threads) {
              int r = i / sd.out_dim, j = i % sd.out_dim;
              sh[r * out_max + j] = act1[r * ld + j];
            }
            __syncthreads();
          }
        }
        // coupling transform, one thread per row (deterministic log-det summation order)
        if (tid < R) {
          const int r = tid;
          float l = ldj[r];
          if (md.kind == GBNF_KIND_GLOW) {
            if (md.coupling == GBNF_COUPLING_AFFINE) {
              for (int j = 0; j < sd.out_dim; ++j) {
                float shift = act1[r * ld + 2 * j], raw = act1[r * ld + 2 * j + 1];
                float s = 1.f / (1.f + expf(-(raw + 2.f)));            // torch.sigmoid(scale + 2.)  glow.py:333
                float* zp = zs + r * Dv + idx2[j];
                *zp = (*zp + shift) * s;
                l += logf(s);                                          // torch.log(scale)           glow.py:338
              }
            } else {
              for (int j = 0; j < sd.out_dim; ++j) zs[r * Dv + idx2[j]] += act1[r * ld + j];
            }
          } else {
            for (int j = 0; j < sd.out_dim; ++j) {
              float shift = sh[r * out_max + j], sc = act1[r * ld + j];
              float* zp = zs + r * Dv + idx2[j];
              *zp = shift + *zp * expf(sc);                            // transformations.py:575
              l += sc;                                                 // transformations.py:577
            }
          }
          ldj[r] = l;
        }
        __syncthreads();
      }
      // component log-density for the resident rows
      if (tid < R) {
        const int r = tid;
        const long long gr = row0 + r;
        const CompDesc& cd = a.comps[c];
        const float* bm = a.fblob + cd.base_off;
        const float* bi = bm + Dv;
        float q = 0.f;
        for (int p = 0; p < D; ++p) { float d = zs[r * Dv + p] - bm[p]; q = fmaf(d * d, bi[p], q); }
        const float ldj_tot = ldj[r] + a.fblob[cd.const_off];
        const float lq = (bm[2 * Dv] - q) + ldj_tot;
        if (gr < a.B) {
          if (a.logq) a.logq[gr * a.ld_logq + (c - a.c0)] = lq;
          if (a.ldj_out) a.ldj_out[gr] = ldj_tot;
          if (a.z_out) {
            const int* sig = a.iblob + cd.sigma_off;
            for (int j = 0; j < D; ++j) a.z_out[gr * D + j] = zs[r * Dv + sig[j]];
          }
        }
        if (a.G_ll != nullptr && c < a.n_mix) {
          OnlineLse o; o.m = lse_m[r]; o.s = lse_s[r];
          o.add(coef[c] + lq);
          lse_m[r] = o.m; lse_s[r] = o.s;
        }
      }
      __syncthreads();
    }
    if (a.G_ll != nullptr && tid < R) {
      const long long gr = row0 + tid;
      OnlineLse o; o.m = lse_m[tid]; o.s = lse_s[tid];
      if (gr < a.B) a.G_ll[gr] = o.value();
    }
    __syncthreads();
  }
}

// ---- inverse direction (sampling): x = f_c^{-1}(z) for the component of each work unit -----------------------------------------
// Exact inverse of the forward kernel above, step by step in reverse order: coupling^-1 (the MLPs see z1, which the forward
// step left untouched), then ActNorm^-1 / eval-BatchNorm^-1 on all columns.  Upstream: FlowStep.decode models/glow.py:344-366,
// RealNVPFlow.decode models/realnvp.py:97-113 (whose flip pairing is not an inverse of encode, SURVEY 7 -- this one is).
// a.x = z [B, D] (logical column order), a.z_out = x [B, D], a.ldj_out = log-det of the inverse map (= -forward log-det); work
// units from `ut` (one component and up to R rows each, common.cuh).
template <int R>
__global__ void __launch_bounds__(kF32Threads, 1) coupling_fp32_inverse_kernel(CouplingArgs a, int ld, int out_max, UnitTable ut) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ModelDims& md = a.md;
  const int D = md.D, Dv = md.Dv;
  float* zs = reinterpret_cast<float*>(smem_raw);
  float* act0 = zs + ((R * Dv + 3) & ~3);
  float* act1 = act0 + R * ld;
  float* Ws = act1 + R * ld;
  float* sh = Ws + 2 * kF32KT * kF32NT;
  float* coef = sh + R * out_max;
  float* ldj = coef + kMaxComponents;   // [R]
  const int tid = threadIdx.x;
  const int num_units = min(a.num_units, __ldg(ut.count));
  for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
    const int4 un = __ldg(ut.unit + u);
    const int c = un.x;
    const long long row0 = un.y, row_end = row0 + un.z;
    const CompDesc& cd = a.comps[c];
    const int* sig = a.iblob + cd.sigma_off;
    // z arrives in the flow's OUTPUT column order: logical column j lives at physical column sigma[j]
    for (int i = tid; i < R * D; i += kF32Threads) {
      int r = i / D, j = i % D;
      long long gr = row0 + r;
      zs[r * Dv + sig[j]] = (gr < row_end) ? a.x[gr * D + j] : 0.f;
    }
    if (tid < R) ldj[tid] = 0.f;
    __syncthreads();
    for (int k = md.K - 1; k >= 0; --k) {
      const StepDesc& sd = a.steps[c * md.K + k];
      const float* add = a.fblob + sd.vec_off;
      const float* mul = add + Dv;
      const float* off = mul + Dv;
      const int* idx1 = a.iblob + sd.idx_off;
      const int* idx2 = idx1 + sd.in_dim;
      const int Kp0 = sd.layer[0][0].Kp;
      for (int net = 0; net < md.nnets; ++net) {
        for (int i = tid; i < R * Kp0; i += kF32Threads) {
          int r = i / Kp0, j = i % Kp0;
          act0[r * ld + j] = (j < sd.in_dim) ? zs[r * Dv + idx1[j]] : 0.f;
        }
        __syncthreads();
        int act_kind = (md.act == GBNF_ACT_TANH) ? 1 : (md.act == GBNF_ACT_RELU) ? 2 : (md.act == GBNF_ACT_RESIDUAL) ? 3 : (net == 0 ? 2 : 1);
        run_net_fp32<R>(sd, net, act_kind, md.nlayers, a, act0, act1, ld, Ws);
        if (md.nnets == 2 && net == 0) {
          for (int i = tid; i < R * sd.out_dim; i += kF32Threads) {
            int r = i / sd.out_dim, j = i % sd.out_dim;
            sh[r * out_max + j] = act1[r * ld + j];
          }
          __syncthreads();
        }
      }
      if (tid < R) {
        const int r = tid;
        float l = ldj[r];
        if (md.kind == GBNF_KIND_GLOW) {
          if (md.coupling == GBNF_COUPLING_AFFINE) {
            for (int j = 0; j < sd.out_dim; ++j) {
              float shift = act1[r * ld + 2 * j], raw = act1[r * ld + 2 * j + 1];
              float s = 1.f / (1.f + expf(-(raw + 2.f)));
              float* zp = zs + r * Dv + idx2[j];
              *zp = *zp / s - shift;                                   // glow.py:354-356
              l -= logf(s);                                            // glow.py:357
            }
          } else {
            for (int j = 0; j < sd.out_dim; ++j) zs[r * Dv + idx2[j]] -= act1[r * ld + j];   // glow.py:350
          }
        } else {
          for (int j = 0; j < sd.out_dim; ++j) {
            float shift = sh[r * out_max + j], sc = act1[r * ld + j];
            float* zp = zs + r * Dv + idx2[j];
            *zp = (*zp - shift) * expf(-sc);                           // inverse of transformations.py:575
            l -= sc;
          }
        }
        ldj[r] = l;
      }
      __syncthreads();
      if (sd.has_invconv)                                              // W^-1 (layers.py:772-776), back to the pre-step column layout
        dense_step_fp32<R>(zs, Dv, D, reinterpret_cast<const float*>(a.wblob) + sd.icwinv_off, a.fblob + sd.icb_off, sd.ic_Kp, sd.ic_Np,
                           act0, act1, ld, Ws);
      if (sd.has_affine) {                                             // ActNorm reverse (layers.py:505-518) / BatchNorm^-1
        for (int i = tid; i < R * D; i += kF32Threads) {
          int r = i / D, p = i % D;
          zs[r * Dv + p] = (zs[r * Dv + p] - off[p]) / mul[p] - add[p];
        }
        __syncthreads();
      }
    }
    for (int i = tid; i < R * D; i += kF32Threads) {
      int r = i / D, p = i % D;
      long long gr = row0 + r;
      if (gr < row_end && a.z_out) a.z_out[gr * D + p] = zs[r * Dv + p];   // physical == logical at the flow's input
    }
    if (tid < R && a.ldj_out && row0 + tid < row_end) a.ldj_out[row0 + tid] = ldj[tid] - a.fblob[cd.const_off];
    __syncthreads();
  }
}

}  // namespace gbnf
