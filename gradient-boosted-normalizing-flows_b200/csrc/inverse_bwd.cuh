// Backward of the INVERSE map x = f_c^{-1}(z) (sampling with gradients: BoostedFlow.rsample, gbnf_*_inverse_backward): gradients
// of any loss L(x, ldj_inv) with respect to every parameter of the components that drew rows, and to z.  Same recompute-in-kernel
// scheme, envelope and shared-memory history as the training backward (train_bwd.cuh), walked in the other direction:
//
//   phase A  inv_bwd_rows_kernel   one CTA per work unit of <= 16 rows of ONE component (rows sorted by component on the device
//            for a mixture): the inverse sweep k = K-1 .. 0 in shared memory (keeps every step's input and coupling-network
//            outputs; z1 passes through, so the networks see the same input as in the forward direction), then the backward sweep
//            k = 0 .. K-1: ActNorm^-1 (or the RealNVP split), coupling^-1, the data-gradient GEMMs.  Leaves the hidden activations
//            and d pre-activations in the L2 scratch at each row's sorted position, accumulates the ActNorm gradients.
//   phase B  inv_wgrad_kernel      train_wgrad_kernel's tiles, one job per (component, step, network, layer), over that
//            component's contiguous range of sorted rows, read on the device (no host synchronisation); deterministic.
//
// Chain rule per step (u = the coupling-order vector after coupling^-1, y = the step's inverse input, [y1 | y2]):
//   Glow affine   u2 = y2 / s - shift, s = sigmoid(raw + 2), ldj -= sum log s:
//                 d y2 = d u2 / s, d shift = -d u2, d s = -d u2 y2 / s^2 - dldj / s, d raw = d s s (1 - s)
//   Glow additive u2 = y2 - net: d y2 = d u2, d net = -d u2
//   Glow          x[perm[j]] = u[j] e^-logs[perm[j]] - bias[perm[j]], ldj -= sum logs:
//                 d u = d x e^-logs, d bias = -sum d x, d logs = -sum d x (x + bias) - sum dldj
//   RealNVP       u2 = (y2 - t) e^-s, ldj -= sum s: d y2 = d u2 e^-s, d t = -d u2 e^-s, d s = -d u2 u2 - dldj
//   every coupling: d y1 = d u1 + the networks' input gradient (z1 passes through AND feeds them).
#pragma once
#include "train_bwd.cuh"

namespace gbnf {

struct InvBwdArgs {
  const float* z; long long B;                 // [B, D] in the caller's row order
  const float* dx; const float* dldj;          // upstream gradients dL/dx [B, D], dL/dldj_inv [B]
  const long long* perm;                       // sorted position -> caller row (NULL: the identity)
  const int4* units; const int* n_units;       // {component slot, first sorted position, rows}; the count lives on the device
  const TrainStep* steps; int K;               // [component slots][K]; scratch pointers indexed by sorted position
  int D, hp, act, coupling, kind, nnets;
  int nlayers;                                 // Linear layers per coupling network: depth + 2
  int ld;                                      // row stride of the shared activation buffers
  const float* zeros;                          // >= 1024 zero floats (bias of the data-gradient GEMMs)
  float* dz;                                   // optional dL/dz [B, D]
};

// Dynamic shared memory: exactly train_bwd_smem_bytes (zh[(K+1)][R][D] | oh[K][nnets][R][64] | 3 x [R][ld] | Ws | 2 x [R][D]),
// so that one bound (fused_backward_smem_bytes in boosted_flow.py) routes both backward kernels.
__global__ void __launch_bounds__(kF32Threads, 1) inv_bwd_rows_kernel(InvBwdArgs a) {
  if ((int)blockIdx.x >= *a.n_units) return;
  const int4 unit = a.units[blockIdx.x];
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int R = kTrR;
  const int D = a.D, K = a.K, L = a.nlayers, ld = a.ld, hD0 = a.D / 2;
  const bool glow = a.kind == GBNF_KIND_GLOW;
  float* zh = reinterpret_cast<float*>(smem_raw);
  float* oh = zh + (((K + 1) * R * D + 3) & ~3);
  float* act0 = oh + K * a.nnets * R * 64;
  float* act1 = act0 + R * ld;
  float* act2 = act1 + R * ld;
  float* Ws = act2 + R * ld;
  float* dzb = Ws + 2 * kF32KT * kF32NT;
  float* tmp = dzb + ((R * D + 3) & ~3);
  const int tid = threadIdx.x;
  const TrainStep* cs = a.steps + (long long)unit.x * K;
  const long long p0 = unit.y;                 // sorted position of the unit's first row (the scratch row)
  const int nrow = unit.z;
  const int hp = a.hp;
  auto row_of = [&](int r) { return a.perm ? a.perm[p0 + r] : p0 + r; };
  auto act_of = [&](int net) { return (a.act == GBNF_ACT_TANH) ? 1 : (a.act == GBNF_ACT_RELU) ? 2 : (net == 0 ? 2 : 1); };   // mixed: t ReLU, s tanh

  // ---------------- inverse sweep: zh[k + 1] (step k's inverse input, coupling order) -> zh[k] (its output, input order) -------
  for (int i = tid; i < R * D; i += kF32Threads) {
    const int r = i / D, j = i - r * D;
    zh[K * R * D + i] = (r < nrow) ? a.z[row_of(r) * D + j] : 0.f;
  }
  __syncthreads();
  for (int k = K - 1; k >= 0; --k) {
    const TrainStep& s = cs[k];
    const int h0 = s.in_dim;
    const float* y = zh + (k + 1) * R * D;
    float* xo = zh + k * R * D;
    for (int net = 0; net < a.nnets; ++net) {
      for (int i = tid; i < R * s.Kp[0]; i += kF32Threads) {
        const int r = i / s.Kp[0], j = i - r * s.Kp[0];
        const float v = (j < h0) ? y[r * D + j] : 0.f;
        act0[r * ld + j] = v;
        if (net == 0 && r < nrow) s.z1[(p0 + r) * s.Kp[0] + j] = v;
      }
      __syncthreads();
      const int ak = act_of(net);
      float* in = act0;
      float* out = act1;
      for (int l = 0; l < L - 1; ++l) {
        train_gemm<R>(ak, in, out, ld, s.Wt[net][l], s.b[net][l], s.Kp[l], s.Np[l], Ws);
        for (int i = tid; i < R * hp; i += kF32Threads) {
          const int r = i / hp, j = i - r * hp;
          if (r < nrow) s.hid[net][l][(p0 + r) * hp + j] = out[r * ld + j];
        }
        in = out;
        out = (out == act1) ? act2 : act1;
      }
      train_gemm<R>(0, in, act0, ld, s.Wt[net][L - 1], s.b[net][L - 1], s.Kp[L - 1], s.Np[L - 1], Ws);
      for (int i = tid; i < R * 64; i += kF32Threads) oh[((k * a.nnets + net) * R + (i >> 6)) * 64 + (i & 63)] = act0[(i >> 6) * ld + (i & 63)];
      __syncthreads();
    }
    const float* o0 = oh + k * a.nnets * R * 64;
    const float* o1 = o0 + R * 64;                               // s-network output: read for RealNVP only
    for (int i = tid; i < R * D; i += kF32Threads) {
      const int r = i / D, j = i - r * D;
      float v = y[i];
      if (j >= h0) {
        const int jj = j - h0;
        if (!glow) {
          v = (v - o0[r * 64 + jj]) * expf(-o1[r * 64 + jj]);
        } else if (a.coupling == GBNF_COUPLING_AFFINE) {
          const float shift = o0[r * 64 + 2 * jj], raw = o0[r * 64 + 2 * jj + 1];
          const float sg = 1.f / (1.f + expf(-(raw + 2.f)));
          v = v / sg - shift;
        } else {
          v = v - o0[r * 64 + jj];
        }
      }
      const int pj = train_src_col(s, a.kind, j, hD0);
      xo[r * D + pj] = glow ? v * expf(-s.an_logs[pj]) - s.an_bias[pj] : v;
    }
    __syncthreads();
  }
  // ---------------- backward sweep: dzb = dL/d(step k's output) -> dL/d(its inverse input) ------------------------------------
  for (int i = tid; i < R * D; i += kF32Threads) {
    const int r = i / D;
    dzb[i] = (r < nrow) ? a.dx[row_of(r) * D + (i - r * D)] : 0.f;
  }
  __syncthreads();
  for (int k = 0; k < K; ++k) {
    const TrainStep& s = cs[k];
    const int h0 = s.in_dim, h1d = s.out_dim;
    const float* y = zh + (k + 1) * R * D;
    const float* xk = zh + k * R * D;
    const float* o0 = oh + k * a.nnets * R * 64;
    const float* o1 = o0 + R * 64;
    // ActNorm^-1 (Glow) or the split (RealNVP) backward: d u in coupling order -> tmp
    for (int j = tid; j < D; j += kF32Threads) {
      const int pj = train_src_col(s, a.kind, j, hD0);
      if (glow) {
        const float e = expf(-s.an_logs[pj]), bias = s.an_bias[pj];
        float gl = 0.f, gb = 0.f;
        for (int r = 0; r < R; ++r) {
          const float g = dzb[r * D + pj];
          tmp[r * D + j] = g * e;
          gb -= g;
          gl -= g * (xk[r * D + pj] + bias);
        }
        if (s.g_logs != nullptr) {
          float dl = 0.f;
          for (int r = 0; r < nrow; ++r) dl += a.dldj[row_of(r)];
          atomicAdd(s.g_logs + pj, gl - dl);
          atomicAdd(s.g_bias + pj, gb);
        }
      } else {
        for (int r = 0; r < R; ++r) tmp[r * D + j] = dzb[r * D + pj];
      }
    }
    __syncthreads();
    for (int net = a.nnets - 1; net >= 0; --net) {
      // coupling^-1 backward -> d out of this network in act0; after the LAST network (net 0) tmp[:, h0:] = d y2
      const int NpL = s.Np[L - 1];
      for (int i = tid; i < R * NpL; i += kF32Threads) act0[(i / NpL) * ld + (i % NpL)] = 0.f;
      __syncthreads();
      for (int i = tid; i < R * h1d; i += kF32Threads) {
        const int r = i / h1d, jj = i - r * h1d;
        const float g2 = tmp[r * D + h0 + jj];
        const float dldj = (r < nrow) ? a.dldj[row_of(r)] : 0.f;
        const float y2 = y[r * D + h0 + jj];
        if (!glow) {
          const float e = expf(-o1[r * 64 + jj]);
          if (net == 1) act0[r * ld + jj] = -g2 * ((y2 - o0[r * 64 + jj]) * e) - dldj;   // d s
          else { act0[r * ld + jj] = -g2 * e; tmp[r * D + h0 + jj] = g2 * e; }          // d t ; d y2
        } else if (a.coupling == GBNF_COUPLING_AFFINE) {
          const float raw = o0[r * 64 + 2 * jj + 1];
          const float sg = 1.f / (1.f + expf(-(raw + 2.f)));
          const float dsg = -g2 * y2 / (sg * sg) - dldj / sg;
          act0[r * ld + 2 * jj] = -g2;                                      // d shift
          act0[r * ld + 2 * jj + 1] = dsg * sg * (1.f - sg);                // d raw
          tmp[r * D + h0 + jj] = g2 / sg;                                   // d y2
        } else {
          act0[r * ld + jj] = -g2;                                          // d net ; d y2 = d u2 unchanged
        }
      }
      __syncthreads();
      for (int i = tid; i < R * NpL; i += kF32Threads) {
        const int r = i / NpL, j = i - r * NpL;
        if (r < nrow) s.dpre[net][L - 1][(p0 + r) * NpL + j] = act0[r * ld + j];
      }
      const int ak = act_of(net);
      float* din = act0;
      float* dout = act1;
      for (int l = L - 1; l > 0; --l) {
        gemm_layer_fp32<R, 0>(din, dout, ld, s.Wn[net][l], a.zeros, s.NKp[l], s.KNp[l], Ws);
        for (int i = tid; i < R * hp; i += kF32Threads) {
          const int r = i / hp, j = i - r * hp;
          const float hv = (r < nrow) ? s.hid[net][l - 1][(p0 + r) * hp + j] : 0.f;
          const float d = dout[r * ld + j] * (ak == 2 ? act_grad_from_output<2>(hv) : act_grad_from_output<1>(hv));
          dout[r * ld + j] = d;
          if (r < nrow) s.dpre[net][l - 1][(p0 + r) * hp + j] = d;
        }
        __syncthreads();
        din = dout;
        dout = (dout == act1) ? act2 : act1;
      }
      gemm_layer_fp32<R, 0>(din, act0, ld, s.Wn[net][0], a.zeros, s.NKp[0], s.KNp[0], Ws);      // d y1 through the network
      for (int i = tid; i < R * h0; i += kF32Threads) {
        const int r = i / h0, j = i - r * h0;
        tmp[r * D + j] += act0[r * ld + j];
      }
      __syncthreads();
    }
    float* t = dzb; dzb = tmp; tmp = t;                          // the step's inverse input is the next step's output
  }
  if (a.dz != nullptr)
    for (int i = tid; i < R * D; i += kF32Threads) {
      const int r = i / D;
      if (r < nrow) a.dz[row_of(r) * D + (i - r * D)] = dzb[i];
    }
}

// ---- phase B: the weight-gradient tiles of train_wgrad_kernel over one component's range of sorted rows -------------------------
// One 64 x 64 tile t of a job's dW / db: train_wgrad_kernel's tile summed over rows [rb, re) in chunks of 32 from rb (a job covers
// one component's range of sorted rows).  A copy rather than a change of train_wgrad_kernel, whose code stays as it was.
__device__ __forceinline__ void wgrad_tile(const WgradJob& job, int t, long long rb, long long re) {
  __shared__ float sd[32][65];       // dact chunk [rows][n]
  __shared__ float si[32][65];       // input chunk [rows][k]
  const int n0 = (t / job.tiles_k) * 64, k0 = (t % job.tiles_k) * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // thread owns n = n0 + ty * 4 + i, k = k0 + tx * 4 + q
  float acc[4][4] = {};
  float bacc[4] = {};
  for (long long r0 = rb; r0 < re; r0 += 32) {
    for (int i = threadIdx.x; i < 32 * 64; i += 256) {
      const int r = i >> 6, c = i & 63;
      const long long gr = r0 + r;
      sd[r][c] = (gr < re && n0 + c < job.ld_d) ? job.dact[gr * job.ld_d + n0 + c] : 0.f;
      si[r][c] = (gr < re && k0 + c < job.ld_i) ? job.in[gr * job.ld_i + k0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < 32; ++r) {
      float dv[4], iv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { dv[i] = sd[r][ty * 4 + i]; iv[i] = si[r][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        bacc[i] += dv[i];
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i][q] = fmaf(dv[i], iv[q], acc[i][q]);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + ty * 4 + i;
    if (n >= job.N) continue;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int k = k0 + tx * 4 + q;
      if (k < job.Kd) job.dW[(long long)n * job.Kd + k] = acc[i][q];
    }
    if (k0 == 0 && tx == 0) job.db[n] = bacc[i];
  }
}

struct RangedWgradJob {
  WgradJob w;
  const int* lo; const int* hi;      // rows [*lo, *hi) of the sorted order (device: the counting sort's bin starts); NULL: [0, B)
};

__global__ void __launch_bounds__(256) inv_wgrad_kernel(const RangedWgradJob* __restrict__ jobs, int njobs, long long B) {
  int j = 0;
  while (j + 1 < njobs && (int)blockIdx.x >= jobs[j + 1].w.tile0) ++j;
  const RangedWgradJob rj = jobs[j];
  wgrad_tile(rj.w, (int)blockIdx.x - rj.w.tile0, rj.lo ? *rj.lo : 0LL, rj.hi ? *rj.hi : B);
}

}  // namespace gbnf
