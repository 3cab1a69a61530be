// Backward of the component that is being TRAINED (SURVEY 8(f).1): gradients of any loss L(z, log_det_j) of one Glow
// component with respect to all of its parameters, for the training step of density_experiment.py:647-661 / :361-374
// (nll = mean(-(log N(z) + ldj)) on the resampled batch; loss.backward()).  Recompute-in-kernel: nothing is saved by the
// forward pass -- the fixed-component kernels serve it -- and this launch recomputes the activations it needs.
//
//   phase A  train_bwd_rows_kernel   one CTA per 16 rows, all K steps: forward sweep in shared memory (keeps every step's
//            input and coupling-network output), then the backward sweep from the last step to the first: coupling
//            transform, the L = depth + 2 data-gradient GEMMs (d act = d out . W, nn.Linear layout) with the tanh / ReLU
//            derivative, permutation and ActNorm.  Leaves the depth + 1 hidden activations and the L "d pre-activation"
//            matrices of every step in an L2-resident scratch, accumulates the ActNorm gradients.
//   phase B  train_wgrad_kernel      dW[n][k] = sum_rows dact[r][n] * in[r][k] and db[n] = sum_rows dact[r][n] for every
//            (step, layer): 64 x 64 output tiles over ALL rows, written straight into the caller's gradient tensors
//            (deterministic: no atomics on the weight gradients).
// fp32 CUDA-core arithmetic throughout (reference-class numerics: the gate is 1e-4 on the gradients).
// Models, in the reference's own (logical) column order, coupling networks of every depth the library accepts (0 .. 4:
// Linear(in, h), depth x Linear(h, h), Linear(h, out), an activation after every layer but the last):
//   Glow step    = ActNorm1d -> Permute1d -> affine / additive coupling with ONE MLP (models/glow.py:317-342,
//                  models/layers.py:208-243,488-518,661-668);
//   RealNVP step = [z1 | z2] split (swapped when the step is flipped) -> z2' = t(z1) + z2 exp(s(z1)) with TWO MLPs, output
//                  [z1, z2'] (models/transformations.py:560-579, models/realnvp.py:35-76); steps WITHOUT BatchNorm only
//                  (train-mode BatchNorm couples the rows of a batch: those configurations train through autograd).
// Shared memory holds three activation rows whatever the depth (the hidden layers ping-pong between two of them; what phase B
// needs goes to the scratch), so the deepest component served at a given (kind, D, h) does not depend on the depth.
#pragma once
#include "coupling_fp32.cuh"

namespace gbnf {

constexpr int kTrR = 16;             // rows per CTA of phase A
constexpr size_t kTrMaxSmem = 227 * 1024;   // dynamic shared memory one block may use (sm_100)

struct TrainStep {                   // one coupling step of the component under training (device pointers)
  const float* an_bias; const float* an_logs; const long long* perm;       // Glow: raw reference tensors; RealNVP: null
  int flipped, in_dim, out_dim, pad_;                                      // RealNVP: (k + flip_init) odd; |z1|, |z2| of this step
  // per Linear layer l < L = depth + 2 of network net (0 = glow block / t, 1 = s)
  const float* Wt[2][GBNF_MAX_LAYERS];   // forward layout  Wt[Kp][Np]   (k-major, n contiguous, zero padded)
  const float* Wn[2][GBNF_MAX_LAYERS];   // backward layout Wn[NKp][KNp] (nn.Linear rows = n, k contiguous, zero padded)
  const float* b[2][GBNF_MAX_LAYERS];    // biases padded to Np
  int Kp[GBNF_MAX_LAYERS], Np[GBNF_MAX_LAYERS];     // forward padding (Kp % 32 == 0, Np % 64 == 0)
  int NKp[GBNF_MAX_LAYERS], KNp[GBNF_MAX_LAYERS];   // backward padding: rows (n) to a multiple of 32, columns (k) to a multiple of 64
  float* g_bias; float* g_logs;      // ActNorm gradients [D] (accumulated with atomics; zeroed by the host)
  // scratch (per step, [B][ld]) for phase B: the network input z1 [B][Kp[0]], the output of hidden layer l < L - 1
  // hid[net][l] [B][hp], and the d pre-activation of layer l dpre[net][l] ([B][hp]; the last layer [B][Np[L - 1]])
  float* z1; float* hid[2][GBNF_MAX_LAYERS - 1]; float* dpre[2][GBNF_MAX_LAYERS];
};

struct TrainArgs {
  const float* x; long long B;
  const float* dz; const float* dldj;          // upstream gradients dL/dz [B, D], dL/dldj [B]
  const TrainStep* steps; int K;
  int D, h, hp, act, coupling, kind, nnets;
  int nlayers;                                 // Linear layers per coupling network: depth + 2
  int ld;                                      // row stride of the shared activation buffers
  const float* zeros;                          // >= 1024 zero floats (bias of the data-gradient GEMMs)
  float* dx;                                   // optional dL/dx [B, D]
};

template <int ACT>
__device__ __forceinline__ float act_grad_from_output(float hval) {
  return ACT == 1 ? (1.f - hval * hval) : (hval > 0.f ? 1.f : 0.f);     // tanh' = 1 - tanh^2 ; relu' from its output
}

// column of the step's INPUT that feeds position j of the coupling order [z1 | z2]
__device__ __forceinline__ int train_src_col(const TrainStep& s, int kind, int j, int h0) {
  if (kind == GBNF_KIND_GLOW) return (int)s.perm[j];
  if (!s.flipped) return j;
  return (j < s.in_dim) ? h0 + j : j - s.in_dim;                 // flipped: z1 = x[:, h0:], z2 = x[:, :h0]
}
template <int R>
__device__ __forceinline__ void train_gemm(int act_kind, const float* in, float* out, int ld, const float* Wt, const float* b, int Kp, int Np,
                                           float* Ws) {
  if (act_kind == 2)      gemm_layer_fp32<R, 2>(in, out, ld, Wt, b, Kp, Np, Ws);
  else if (act_kind == 1) gemm_layer_fp32<R, 1>(in, out, ld, Wt, b, Kp, Np, Ws);
  else                    gemm_layer_fp32<R, 0>(in, out, ld, Wt, b, Kp, Np, Ws);
}

// Dynamic smem: zh[(K+1)][R][D] | oh[K][nnets][R][64] | act0[R][ld] | act1[R][ld] | act2[R][ld] | Ws[2][32][64] | dzb[R][D] | tmp[R][D]
// The history zh / oh grows with K: the deepest component that fits is the bound of the fused backward (gbnf.h lists a few).
// boosted_flow.py's fused_backward_smem_bytes() mirrors this count to route the shapes that do not fit to autograd.
inline size_t train_bwd_smem_bytes(int K, int D, int nnets, int ld) {
  return ((size_t)(((K + 1) * kTrR * D + 3) & ~3) + (size_t)K * nnets * kTrR * 64 + 3ull * kTrR * ld + 2ull * kF32KT * kF32NT +
          2ull * ((kTrR * D + 3) & ~3)) * sizeof(float);
}
__global__ void __launch_bounds__(kF32Threads, 1) train_bwd_rows_kernel(TrainArgs a) {
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
  const long long row0 = (long long)blockIdx.x * R;
  const int hp = a.hp;
  auto act_of = [&](int net) { return (a.act == GBNF_ACT_TANH) ? 1 : (a.act == GBNF_ACT_RELU) ? 2 : (net == 0 ? 2 : 1); };   // mixed: t ReLU, s tanh

  // ---------------- forward sweep ----------------
  for (int i = tid; i < R * D; i += kF32Threads) {
    const int r = i / D, j = i - r * D;
    const long long gr = row0 + r;
    zh[i] = (gr < a.B) ? a.x[gr * D + j] : 0.f;
  }
  __syncthreads();
  for (int k = 0; k < K; ++k) {
    const TrainStep& s = a.steps[k];
    const int h0 = s.in_dim;
    const float* zin = zh + k * R * D;
    float* zout = zh + (k + 1) * R * D;
    // coupling order [z1 | z2]: Glow yp[:, j] = (x[:, perm[j]] + bias) exp(logs) (layers.py:488-518, 661-668); RealNVP: the split
    for (int i = tid; i < R * D; i += kF32Threads) {
      const int r = i / D, j = i - r * D;
      const int pj = train_src_col(s, a.kind, j, hD0);
      tmp[i] = glow ? (zin[r * D + pj] + s.an_bias[pj]) * expf(s.an_logs[pj]) : zin[r * D + pj];
    }
    __syncthreads();
    for (int net = 0; net < a.nnets; ++net) {
      for (int i = tid; i < R * s.Kp[0]; i += kF32Threads) {
        const int r = i / s.Kp[0], j = i - r * s.Kp[0];
        const float v = (j < h0) ? tmp[r * D + j] : 0.f;
        act0[r * ld + j] = v;
        const long long gr = row0 + r;
        if (net == 0 && gr < a.B) s.z1[gr * s.Kp[0] + j] = v;
      }
      __syncthreads();
      const int ak = act_of(net);
      // act0 -> layer 0 -> act1; the hidden layers ping-pong between act1 and act2; the last layer writes act0
      float* in = act0;
      float* out = act1;
      for (int l = 0; l < L - 1; ++l) {
        train_gemm<R>(ak, in, out, ld, s.Wt[net][l], s.b[net][l], s.Kp[l], s.Np[l], Ws);
        for (int i = tid; i < R * hp; i += kF32Threads) {        // hidden activation for the backward sweep and for phase B
          const int r = i / hp, j = i - r * hp;
          const long long gr = row0 + r;
          if (gr < a.B) s.hid[net][l][gr * hp + j] = out[r * ld + j];
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
      float v = tmp[i];
      if (j >= h0) {
        const int jj = j - h0;
        if (!glow) {
          v = o0[r * 64 + jj] + v * expf(o1[r * 64 + jj]);                 // transformations.py:575
        } else if (a.coupling == GBNF_COUPLING_AFFINE) {
          const float shift = o0[r * 64 + 2 * jj], raw = o0[r * 64 + 2 * jj + 1];
          const float sg = 1.f / (1.f + expf(-(raw + 2.f)));            // glow.py:333
          v = (v + shift) * sg;                                           // glow.py:334-335
        } else {
          v = v + o0[r * 64 + jj];                                        // glow.py:328-329
        }
      }
      zout[i] = v;
    }
    __syncthreads();
  }
  // ---------------- backward sweep ----------------
  for (int i = tid; i < R * D; i += kF32Threads) {
    const int r = i / D;
    const long long gr = row0 + r;
    dzb[i] = (gr < a.B) ? a.dz[gr * D + (i - r * D)] : 0.f;
  }
  __syncthreads();
  for (int k = K - 1; k >= 0; --k) {
    const TrainStep& s = a.steps[k];
    const int h0 = s.in_dim, h1d = s.out_dim;
    const float* zin = zh + k * R * D;
    const float* o0 = oh + k * a.nnets * R * 64;
    const float* o1 = o0 + R * 64;                               // s-network output: read for RealNVP only
    for (int i = tid; i < R * D; i += kF32Threads) {             // recompute the coupling-order input of this step
      const int r = i / D, j = i - r * D;
      const int pj = train_src_col(s, a.kind, j, hD0);
      tmp[i] = glow ? (zin[r * D + pj] + s.an_bias[pj]) * expf(s.an_logs[pj]) : zin[r * D + pj];
    }
    __syncthreads();
    for (int net = a.nnets - 1; net >= 0; --net) {
      // coupling transform backward -> d out of this network in act0 [R][Np[L - 1]]; after the LAST network (net 0) dzb[:, h0:] = d z2
      const int NpL = s.Np[L - 1];
      for (int i = tid; i < R * NpL; i += kF32Threads) act0[(i / NpL) * ld + (i % NpL)] = 0.f;
      __syncthreads();
      for (int i = tid; i < R * h1d; i += kF32Threads) {
        const int r = i / h1d, jj = i - r * h1d;
        const long long gr = row0 + r;
        const float g2 = dzb[r * D + h0 + jj];
        const float dldj = (gr < a.B) ? a.dldj[gr] : 0.f;
        if (!glow) {
          const float e = expf(o1[r * 64 + jj]);
          if (net == 1) act0[r * ld + jj] = g2 * tmp[r * D + h0 + jj] * e + dldj;     // d scale: out = t + z2 e^s ; ldj += s
          else { act0[r * ld + jj] = g2; dzb[r * D + h0 + jj] = g2 * e; }             // d shift ; d z2
        } else if (a.coupling == GBNF_COUPLING_AFFINE) {
          const float shift = o0[r * 64 + 2 * jj], raw = o0[r * 64 + 2 * jj + 1];
          const float sg = 1.f / (1.f + expf(-(raw + 2.f)));
          const float y2 = tmp[r * D + h0 + jj];
          const float dsg = g2 * (y2 + shift) + dldj / sg;                  // out = (y2 + shift) sg ; ldj += log sg
          act0[r * ld + 2 * jj] = g2 * sg;                                  // d shift
          act0[r * ld + 2 * jj + 1] = dsg * sg * (1.f - sg);                // d raw
          dzb[r * D + h0 + jj] = g2 * sg;                                   // d y2
        } else {
          act0[r * ld + jj] = g2;                                           // out = y2 + net ; d y2 = g2 unchanged
        }
      }
      __syncthreads();
      for (int i = tid; i < R * NpL; i += kF32Threads) {
        const int r = i / NpL, j = i - r * NpL;
        const long long gr = row0 + r;
        if (gr < a.B) s.dpre[net][L - 1][gr * NpL + j] = act0[r * ld + j];
      }
      const int ak = act_of(net);
      // mirror of the forward sweep: d h_l = d_l . W_l (nn.Linear layout: rows n, columns k) into act1, act2, act1, ...,
      // times the activation derivative read from the stored h_l; d z1 = d_0 . W_0 ends in act0
      float* din = act0;
      float* dout = act1;
      for (int l = L - 1; l > 0; --l) {
        gemm_layer_fp32<R, 0>(din, dout, ld, s.Wn[net][l], a.zeros, s.NKp[l], s.KNp[l], Ws);
        for (int i = tid; i < R * hp; i += kF32Threads) {
          const int r = i / hp, j = i - r * hp;
          const long long gr = row0 + r;
          const float hv = (gr < a.B) ? s.hid[net][l - 1][gr * hp + j] : 0.f;
          const float d = dout[r * ld + j] * (ak == 2 ? act_grad_from_output<2>(hv) : act_grad_from_output<1>(hv));
          dout[r * ld + j] = d;
          if (gr < a.B) s.dpre[net][l - 1][gr * hp + j] = d;
        }
        __syncthreads();
        din = dout;
        dout = (dout == act1) ? act2 : act1;
      }
      gemm_layer_fp32<R, 0>(din, act0, ld, s.Wn[net][0], a.zeros, s.NKp[0], s.KNp[0], Ws);      // d z1 [R][KNp0] (first h0 columns valid)
      for (int i = tid; i < R * h0; i += kF32Threads) {
        const int r = i / h0, j = i - r * h0;
        dzb[r * D + j] += act0[r * ld + j];                                  // z1 passes through AND feeds the network(s)
      }
      __syncthreads();
    }
    // back to the step's input order: d x[:, src[j]] = d tmp[:, j]; Glow: y = (x + b) e^logs
    //   dx = dy e^logs ; d logs[p] += sum_r dy y + sum_r dldj ; d bias[p] += sum_r dy e^logs
    for (int j = tid; j < D; j += kF32Threads) {
      const int pj = train_src_col(s, a.kind, j, hD0);
      const float e = glow ? expf(s.an_logs[pj]) : 1.f;
      float gl = 0.f, gb = 0.f;
      for (int r = 0; r < R; ++r) {
        const float dy = dzb[r * D + j];
        gl += dy * tmp[r * D + j];
        gb += dy * e;
        act1[r * ld + pj] = dy * e;                                        // d x in input order (staged, then copied back)
      }
      if (glow) {
        float dl = 0.f;
        for (int r = 0; r < R; ++r) { const long long gr = row0 + r; if (gr < a.B) dl += a.dldj[gr]; }
        atomicAdd(s.g_logs + pj, gl + dl);                                 // ldj += sum_j logs_j (layers.py:512-516)
        atomicAdd(s.g_bias + pj, gb);
      }
    }
    __syncthreads();
    for (int i = tid; i < R * D; i += kF32Threads) { const int r = i / D, j = i - r * D; dzb[i] = act1[r * ld + j]; }
    __syncthreads();
  }
  if (a.dx != nullptr)
    for (int i = tid; i < R * D; i += kF32Threads) {
      const int r = i / D;
      const long long gr = row0 + r;
      if (gr < a.B) a.dx[gr * D + (i - r * D)] = dzb[i];
    }
}

// ---- phase B: weight and bias gradients ------------------------------------------------------------------------------------
struct WgradJob {
  const float* dact; int ld_d;       // [B][ld_d]  d pre-activation of the layer
  const float* in;   int ld_i;       // [B][ld_i]  input activation of the layer
  float* dW; float* db;              // nn.Linear layout [N][Kd] (unpadded), [N]
  int N, Kd;
  int tiles_n, tiles_k, tile0;       // this job's tiles are [tile0, tile0 + tiles_n * tiles_k)
};

__global__ void __launch_bounds__(256) train_wgrad_kernel(const WgradJob* __restrict__ jobs, int njobs, long long B) {
  __shared__ float sd[32][65];       // dact chunk [rows][n]
  __shared__ float si[32][65];       // input chunk [rows][k]
  int j = 0;
  while (j + 1 < njobs && (int)blockIdx.x >= jobs[j + 1].tile0) ++j;
  const WgradJob job = jobs[j];
  const int t = blockIdx.x - job.tile0;
  const int n0 = (t / job.tiles_k) * 64, k0 = (t % job.tiles_k) * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // thread owns n = n0 + ty * 4 + i, k = k0 + tx * 4 + q
  float acc[4][4] = {};
  float bacc[4] = {};
  for (long long r0 = 0; r0 < B; r0 += 32) {
    for (int i = threadIdx.x; i < 32 * 64; i += 256) {
      const int r = i >> 6, c = i & 63;
      const long long gr = r0 + r;
      sd[r][c] = (gr < B && n0 + c < job.ld_d) ? job.dact[gr * job.ld_d + n0 + c] : 0.f;
      si[r][c] = (gr < B && k0 + c < job.ld_i) ? job.in[gr * job.ld_i + k0 + c] : 0.f;
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

// fp32 copies of the trained component's weights in both layouts, ONE launch for all layers of all steps
struct TrainPackJob { const float* W; const float* b; float* Wt; float* Wn; float* bp; int N, Kd, Kp, Np, NKp, KNp; };
__global__ void __launch_bounds__(256) train_pack_kernel(const TrainPackJob* __restrict__ jobs) {
  const TrainPackJob j = jobs[blockIdx.y];
  const long long nt = (long long)j.Kp * j.Np, nn = (long long)j.NKp * j.KNp;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < nt + nn + j.Np; i += (long long)gridDim.x * 256) {
    if (i < nt) {
      const int k = (int)(i / j.Np), n = (int)(i % j.Np);
      j.Wt[i] = (k < j.Kd && n < j.N) ? j.W[(long long)n * j.Kd + k] : 0.f;
    } else if (i < nt + nn) {
      const long long q = i - nt;
      const int n = (int)(q / j.KNp), k = (int)(q % j.KNp);
      j.Wn[q] = (k < j.Kd && n < j.N) ? j.W[(long long)n * j.Kd + k] : 0.f;
    } else {
      const int n = (int)(i - nt - nn);
      j.bp[n] = (n < j.N) ? j.b[n] : 0.f;
    }
  }
}

}  // namespace gbnf
