// Mixture logsumexp, boosting weights, inverse-CDF resampling, row gather.  All HBM-bound streaming kernels:
// 128-bit loads where the row length allows it, warp-shuffle reductions, grids sized in multiples of the SM count.
#pragma once
#include "common.cuh"

namespace gbnf {

constexpr int kMixThreads = 256;

// rows of n <= 4 NV terms, 128-bit loads, two rows per iteration
template <int NV>
__device__ __forceinline__ float mixture_row_lse(const float4 (&v)[NV], int n, const float* coef) {
  float t[4 * NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) { t[4 * i] = v[i].x; t[4 * i + 1] = v[i].y; t[4 * i + 2] = v[i].z; t[4 * i + 3] = v[i].w; }
  float m = -INFINITY;
  bool has_nan = false;
#pragma unroll
  for (int c = 0; c < 4 * NV; ++c) { t[c] = (c < n) ? t[c] + coef[c] : -INFINITY; m = fmaxf(m, t[c]); has_nan |= (t[c] != t[c]); }
  float sum = 0.f;
#pragma unroll
  for (int c = 0; c < 4 * NV; ++c) sum += __expf(t[c] - m);                // exp(-inf) = 0 for skipped / padded terms
  // torch.logsumexp: a NaN term -> NaN (fmaxf drops it), +inf -> +inf, all terms -inf -> -inf
  if (has_nan) return __int_as_float(0x7fc00000);
  return (m == INFINITY || m == -INFINITY) ? m : m + __logf(sum);
}
// R rows in flight per thread (all their 128-bit loads are issued before the first logsumexp): the kernel is a pure stream,
// what it needs is bytes in flight
template <int NV, int R>
__device__ __forceinline__ void mixture_rows_small(const float* __restrict__ logq, long long B, int ld, int n, const float* coef,
                                                   float* __restrict__ G_ll, long long stride) {
  long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  for (; b + (R - 1) * stride < B; b += R * stride) {
    float4 v[R][NV];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int i = 0; i < NV; ++i) v[r][i] = __ldcs(reinterpret_cast<const float4*>(logq + (b + r * stride) * ld) + i);
#pragma unroll
    for (int r = 0; r < R; ++r) G_ll[b + r * stride] = mixture_row_lse<NV>(v[r], n, coef);
  }
  for (; b < B; b += stride) {
    float4 v0[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) v0[i] = __ldcs(reinterpret_cast<const float4*>(logq + b * ld) + i);
    G_ll[b] = mixture_row_lse<NV>(v0, n, coef);
  }
}

// ---- G_ll[b] = logsumexp_c(coef[c] + logq[b, c]) ---------------------------------------------------------
// One thread per row; a warp reads 32 consecutive rows = one contiguous span of 32*ld floats.  With ld % 4 == 0
// the row is fetched with 128-bit loads.
// With cv.world > 1 (component-parallel) logq is this rank's gather buffer: block 0 first publishes "my block is written"
// (the coupling launch before this one in the stream stored it into every rank's buffer), every block then waits until all
// ranks have published the current epoch.
// tstride > 0: logq is COMPONENT-major, element (b, c) at logq[c * tstride + b] (the component-parallel gather buffers: every
// rank's coupling kernel stores 128 consecutive rows of one component = 512 contiguous bytes per peer; with the row-major
// layout each row was a separate 4-byte NVLink write, which cost 2.3 ms per step on 8 GPUs).
__global__ void __launch_bounds__(kMixThreads) mixture_lse_kernel(const float* __restrict__ logq, long long B, int ld,
                                                                 int n, const float* __restrict__ rho, int skip_c,
                                                                 int mix_mode, float* __restrict__ G_ll, CommView cv, int* status,
                                                                 long long tstride = 0) {
  __shared__ float coef[kMaxComponents];
  __shared__ float rho_sum;
  if (cv.world > 1) {
    const int par = cv.epoch & 1u;
    if (blockIdx.x == 0 && threadIdx.x < cv.world) {
      __threadfence_system();
      *reinterpret_cast<volatile unsigned int*>(&cv.blk[threadIdx.x]->done_flag[par][cv.rank]) = cv.epoch;
    }
    if (threadIdx.x < cv.world) comm_wait_flag(&cv.blk[cv.rank]->done_flag[par][threadIdx.x], cv.epoch, status);
    __syncthreads();
    __threadfence_system();
  }
  if (threadIdx.x == 0) {
    if (mix_mode == GBNF_MIX_GEOMETRIC) {
      // utils/density_plotting.py:199-226: total += log_prob_c * rho_c over the components with rho_c != 0, then / sum(rho[0:n])
      float s = 0.f;
      for (int c = 0; c < n; ++c) { coef[c] = rho[c]; s += rho[c]; }
      rho_sum = s;
    } else {
      mixture_coefficients(rho, n, skip_c, mix_mode, coef);
    }
  }
  __syncthreads();
  const bool vec = (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(logq) & 15) == 0);
  const long long stride = (long long)gridDim.x * blockDim.x;
  if (tstride > 0) {          // component-major (logsumexp modes only): coalesced across the rows of a warp
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += stride) {
      if (n <= 16) {          // the same arithmetic as the row-major small path (exact max, then the sum)
        float4 v[4];
        float* t = reinterpret_cast<float*>(v);
#pragma unroll
        for (int c = 0; c < 16; ++c) t[c] = (c < n) ? __ldcs(logq + c * tstride + b) : 0.f;
        G_ll[b] = mixture_row_lse<4>(v, n, coef);
      } else {
        OnlineLse o; o.init();
        for (int c = 0; c < n; ++c) o.add(coef[c] + __ldcs(logq + c * tstride + b));
        G_ll[b] = o.value();
      }
    }
    return;
  }
  if (mix_mode == GBNF_MIX_GEOMETRIC) {
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += stride) {
      const float* row = logq + b * ld;
      float acc = 0.f;
      int c = 0;
      if (vec) {
        for (; c + 4 <= n; c += 4) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(row + c));
          // separate multiply and add, in component order: the reference's `total_prob += log_prob * rho[c]`
          if (coef[c] != 0.f) acc = __fadd_rn(acc, __fmul_rn(v.x, coef[c]));
          if (coef[c + 1] != 0.f) acc = __fadd_rn(acc, __fmul_rn(v.y, coef[c + 1]));
          if (coef[c + 2] != 0.f) acc = __fadd_rn(acc, __fmul_rn(v.z, coef[c + 2]));
          if (coef[c + 3] != 0.f) acc = __fadd_rn(acc, __fmul_rn(v.w, coef[c + 3]));
        }
      }
      for (; c < n; ++c) if (coef[c] != 0.f) acc = __fadd_rn(acc, __fmul_rn(__ldg(row + c), coef[c]));
      G_ll[b] = acc / rho_sum;
    }
    return;
  }
  if (vec && n <= 16) {
    // all terms of a row in registers: exact max, then one ex2 per term and one lg2 per row (MUFU); two rows in flight
    const int nv = (n + 3) >> 2;
    if (nv == 1) mixture_rows_small<1, 4>(logq, B, ld, n, coef, G_ll, stride);
    else if (nv == 2) mixture_rows_small<2, 4>(logq, B, ld, n, coef, G_ll, stride);
    else if (nv == 3) mixture_rows_small<3, 2>(logq, B, ld, n, coef, G_ll, stride);
    else mixture_rows_small<4, 2>(logq, B, ld, n, coef, G_ll, stride);
    return;
  }
  for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += stride) {
    const float* row = logq + b * ld;
    OnlineLse o; o.init();
    int c = 0;
    if (vec) {
      for (; c + 4 <= n; c += 4) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(row + c));
        o.add(coef[c] + v.x); o.add(coef[c + 1] + v.y); o.add(coef[c + 2] + v.z); o.add(coef[c + 3] + v.w);
      }
    }
    for (; c < n; ++c) o.add(coef[c] + __ldg(row + c));
    G_ll[b] = o.value();
  }
}

// ---- batch softmax statistics of u = -G_ll: (max, sum exp(u - max)) ----------------------------------------
// Block partials -> the last block to finish folds them (threadfence + atomic ticket), so one launch suffices.
struct MsPair { float m, s; };
__device__ __forceinline__ MsPair ms_merge(MsPair a, MsPair b) {
  if (b.m == -INFINITY) return a;
  if (a.m == -INFINITY) return b;
  MsPair r;
  r.m = fmaxf(a.m, b.m);
  r.s = a.s * expf(a.m - r.m) + b.s * expf(b.m - r.m);
  return r;
}
__device__ __forceinline__ MsPair ms_warp_reduce(MsPair v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    MsPair w;
    w.m = __shfl_xor_sync(0xffffffffu, v.m, o);
    w.s = __shfl_xor_sync(0xffffffffu, v.s, o);
    v = ms_merge(v, w);
  }
  return v;
}
__device__ inline MsPair ms_block_reduce(MsPair v, MsPair* sm /* [32] */) {
  v = ms_warp_reduce(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) sm[wid] = v;
  __syncthreads();
  MsPair r; r.m = -INFINITY; r.s = 0.f;
  if (wid == 0) {
    if (lane < (int)(blockDim.x >> 5)) r = sm[lane];
    r = ms_warp_reduce(r);
  }
  __syncthreads();
  return r;   // valid in warp 0
}

__global__ void __launch_bounds__(kMixThreads) softmax_stats_kernel(const float* __restrict__ G_ll, long long B,
                                                                   float* __restrict__ partial /* [grid][2] */,
                                                                   unsigned int* __restrict__ ticket,
                                                                   float* __restrict__ ms_out /* [2] */, CommView cv) {
  __shared__ MsPair sm[32];
  __shared__ bool is_last;
  // thread-local online (max, sum) over a strided slice, ONE sweep (G_ll is read from HBM once whatever its size): the
  // running sum is rescaled only when a 128-bit group raises the maximum, so exp() stays at ~one call per element
  MsPair v; v.m = -INFINITY; v.s = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const bool vec = (reinterpret_cast<uintptr_t>(G_ll) & 15) == 0;
  const long long B4 = vec ? (B >> 2) : 0;                                 // 128-bit body, scalar tail
  const float4* G4 = reinterpret_cast<const float4*>(G_ll);
  auto add4 = [&](const float4 g) {
    const float gm = -fminf(fminf(g.x, g.y), fminf(g.z, g.w));
    if (gm > v.m) { v.s = (v.m == -INFINITY) ? 0.f : v.s * expf(v.m - gm); v.m = gm; }
    if (v.m != -INFINITY) v.s += (expf(-g.x - v.m) + expf(-g.y - v.m)) + (expf(-g.z - v.m) + expf(-g.w - v.m));
  };
  long long i = i0;
  for (; i + 3 * stride < B4; i += 4 * stride) {                          // four 128-bit loads in flight per thread
    const float4 g0 = __ldg(G4 + i), g1 = __ldg(G4 + i + stride), g2 = __ldg(G4 + i + 2 * stride), g3 = __ldg(G4 + i + 3 * stride);
    add4(g0); add4(g1); add4(g2); add4(g3);
  }
  for (; i < B4; i += stride) add4(__ldg(G4 + i));
  for (long long j = 4 * B4 + i0; j < B; j += stride) {
    const float u = -__ldg(G_ll + j);
    if (u > v.m) { v.s = (v.m == -INFINITY) ? 0.f : v.s * expf(v.m - u); v.m = u; }
    if (v.m != -INFINITY) v.s += expf(u - v.m);
  }
  MsPair r = ms_block_reduce(v, sm);
  if (threadIdx.x == 0) {
    partial[2 * blockIdx.x] = r.m;
    partial[2 * blockIdx.x + 1] = r.s;
    __threadfence();
    unsigned int t = atomicAdd(ticket, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    MsPair w; w.m = -INFINITY; w.s = 0.f;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
      MsPair p; p.m = __ldcg(partial + 2 * i); p.s = __ldcg(partial + 2 * i + 1);
      w = ms_merge(w, p);
    }
    MsPair f = ms_block_reduce(w, sm);
    if (threadIdx.x == 0) { ms_out[0] = f.m; ms_out[1] = f.s; *ticket = 0u; }
    if (cv.world > 1) {   // publish this shard's (max, sum exp) into every rank's block
      __shared__ float pub[2];
      if (threadIdx.x == 0) { pub[0] = f.m; pub[1] = f.s; }
      __syncthreads();
      if (threadIdx.x < cv.world) {
        CommBlock* b = cv.blk[threadIdx.x];
        const int par = cv.epoch & 1u;
        b->ms[par][cv.rank][0] = pub[0];
        b->ms[par][cv.rank][1] = pub[1];
        __threadfence_system();
        *reinterpret_cast<volatile unsigned int*>(&b->ms_flag[par][cv.rank]) = cv.epoch;
      }
    }
  }
}

// ---- weights from (max, sum): w = exp(u - max) / sum, optional clamp; accumulates sum(w) in fp64 -------------
// density (density_experiment.py:638-641): clamp to [lo, hi] iff max w > hi, and max w == fl(1 / sum) because the
// largest exp() term is exactly 1.  toy (toy_experiment.py:440,453-459): w is first renormalised by its own sum
// (== 1 up to rounding; the kernel folds that first division into `inv_first`), clamp iff max > hi.
__global__ void __launch_bounds__(kMixThreads) weight_apply_kernel(const float* __restrict__ G_ll, long long B,
                                                                  const float* __restrict__ ms, float lo, float hi,
                                                                  float* __restrict__ w, double* __restrict__ wsum,
                                                                  float* __restrict__ stats_opt, CommView cv, unsigned int* ticket,
                                                                  int* status) {
  __shared__ double sm[32];
  __shared__ float gms[2];
  if (cv.world > 1) {
    // GLOBAL batch softmax: every block of every rank merges the ranks' (max, sum exp) pairs in rank order -> identical bits
    if (threadIdx.x < cv.world) comm_wait_flag(&cv.blk[cv.rank]->ms_flag[cv.epoch & 1u][threadIdx.x], cv.epoch, status);
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      const volatile float* v = &cv.blk[cv.rank]->ms[cv.epoch & 1u][0][0];
      float Mg = -INFINITY;
      for (int r = 0; r < cv.world; ++r) Mg = fmaxf(Mg, v[2 * r]);
      float Sg = 0.f;
      for (int r = 0; r < cv.world; ++r) { const float mr = v[2 * r]; if (mr != -INFINITY) Sg += v[2 * r + 1] * expf(mr - Mg); }
      gms[0] = Mg; gms[1] = Sg;
    }
    __syncthreads();
  }
  const float M = (cv.world > 1) ? gms[0] : ms[0], S = (cv.world > 1) ? gms[1] : ms[1];
  const float wmax = 1.0f / S;
  const bool clamp = wmax > hi;
  double acc = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const bool vec = ((reinterpret_cast<uintptr_t>(G_ll) | reinterpret_cast<uintptr_t>(w)) & 15) == 0;
  const long long B4 = vec ? (B >> 2) : 0;                                 // 128-bit body, scalar tail
  const float4* G4 = reinterpret_cast<const float4*>(G_ll);
  auto apply4 = [&](const float4 g, long long i) {
    float4 v;
    v.x = expf(-g.x - M) / S; v.y = expf(-g.y - M) / S; v.z = expf(-g.z - M) / S; v.w = expf(-g.w - M) / S;
    if (clamp) {
      v.x = fmaxf(fminf(v.x, hi), lo); v.y = fmaxf(fminf(v.y, hi), lo);
      v.z = fmaxf(fminf(v.z, hi), lo); v.w = fmaxf(fminf(v.w, hi), lo);
    }
    reinterpret_cast<float4*>(w)[i] = v;
    acc += ((double)v.x + (double)v.y) + ((double)v.z + (double)v.w);
  };
  long long i = i0;
  for (; i + 3 * stride < B4; i += 4 * stride) {                          // four 128-bit loads in flight per thread
    const float4 g0 = __ldg(G4 + i), g1 = __ldg(G4 + i + stride), g2 = __ldg(G4 + i + 2 * stride), g3 = __ldg(G4 + i + 3 * stride);
    apply4(g0, i); apply4(g1, i + stride); apply4(g2, i + 2 * stride); apply4(g3, i + 3 * stride);
  }
  for (; i < B4; i += stride) apply4(__ldg(G4 + i), i);
  for (long long i = 4 * B4 + i0; i < B; i += stride) {
    float v = expf(-__ldg(G_ll + i) - M) / S;
    if (clamp) v = fmaxf(fminf(v, hi), lo);
    w[i] = v;
    acc += (double)v;
  }
  acc = warp_sum(acc);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) sm[wid] = acc;
  __syncthreads();
  if (wid == 0) {
    double t = (lane < (int)(blockDim.x >> 5)) ? sm[lane] : 0.0;
    t = warp_sum(t);
    if (lane == 0) atomicAdd(wsum, t);
  }
  if (stats_opt != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    stats_opt[0] = M; stats_opt[1] = S; stats_opt[2] = clamp ? 1.f : 0.f;
  }
  if (cv.world > 1) {   // the last block to finish publishes this shard's sum of weights into every rank's block
    __shared__ bool is_last;
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
      __threadfence();
      if (threadIdx.x == 0) *ticket = 0u;
      if (threadIdx.x < cv.world) {
        const double local = *reinterpret_cast<volatile double*>(wsum);
        CommBlock* b = cv.blk[threadIdx.x];
        const int par = cv.epoch & 1u;
        b->wsum[par][cv.rank] = local;
        __threadfence_system();
        *reinterpret_cast<volatile unsigned int*>(&b->ws_flag[par][cv.rank]) = cv.epoch;
      }
    }
  }
}

__global__ void __launch_bounds__(kMixThreads) weight_renorm_kernel(float* __restrict__ w, long long B,
                                                                   const double* __restrict__ wsum, int always,
                                                                   float* __restrict__ stats_opt, CommView cv, int* status) {
  __shared__ double gsum;
  if (cv.world > 1) {   // global sum of weights = the ranks' sums added in rank order (identical on every rank)
    if (threadIdx.x < cv.world) comm_wait_flag(&cv.blk[cv.rank]->ws_flag[cv.epoch & 1u][threadIdx.x], cv.epoch, status);
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      const volatile double* v = &cv.blk[cv.rank]->wsum[cv.epoch & 1u][0];
      double t = 0.0;
      for (int r = 0; r < cv.world; ++r) t += v[r];
      gsum = t;
    }
    __syncthreads();
  }
  const float s = (cv.world > 1) ? (float)gsum : (float)(*wsum);
  if (stats_opt != nullptr && blockIdx.x == 0 && threadIdx.x == 0) stats_opt[3] = s;
  if (!always && s == 1.0f) return;            // `if weights.sum() != 1.0` density_experiment.py:640 (toy: always)
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long B4 = ((reinterpret_cast<uintptr_t>(w) & 15) == 0) ? (B >> 2) : 0;
  float4* w4 = reinterpret_cast<float4*>(w);
  auto div4 = [&](float4 v, long long i) { v.x = v.x / s; v.y = v.y / s; v.z = v.z / s; v.w = v.w / s; w4[i] = v; };
  long long i = i0;
  for (; i + 3 * stride < B4; i += 4 * stride) {                          // four 128-bit loads in flight per thread
    const float4 v0 = w4[i], v1 = w4[i + stride], v2 = w4[i + 2 * stride], v3 = w4[i + 3 * stride];
    div4(v0, i); div4(v1, i + stride); div4(v2, i + 2 * stride); div4(v3, i + 3 * stride);
  }
  for (; i < B4; i += stride) div4(w4[i], i);
  for (long long i = 4 * B4 + i0; i < B; i += stride) w[i] = w[i] / s;
}

__global__ void zero_double_kernel(double* p) { *p = 0.0; }

// Component-parallel fallback for the coupling kernels that do not store into peer memory themselves: copies this rank's
// log q block [B, nc] into components [col0, col0 + nc) of every rank's COMPONENT-major gather buffer [C][tstride rows].
__global__ void __launch_bounds__(kMixThreads) comm_scatter_logq_kernel(const float* __restrict__ local, long long B, int nc, CommView cv,
                                                                       long long tstride, int col0) {
  const long long total = B * nc;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i / B); const long long r = i - (long long)c * B;       // consecutive threads = consecutive rows
    const float v = local[r * nc + c];
    for (int q = 0; q < cv.world; ++q) cv.gather[q][(cv.epoch & 1u) * cv.gather_stride + (col0 + c) * tstride + r] = v;
  }
}

// ---- inverse-CDF resampling: fp64 inclusive scan of w, then left binary search per uniform ---------------------
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;                      // per thread
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ inline double block_exclusive_scan(double v, double* sm /* [32] */, double* total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    double t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) sm[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    double s = (lane < (int)(blockDim.x >> 5)) ? sm[lane] : 0.0;
    double si = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      double t = __shfl_up_sync(0xffffffffu, si, o);
      if (lane >= o) si += t;
    }
    sm[lane] = si - s;                              // exclusive warp offsets
    if (lane == 31) *total = si;
  }
  __syncthreads();
  const double r = sm[wid] + inc - v;
  __syncthreads();
  return r;
}

// pass 1: per-tile sums
__global__ void __launch_bounds__(kScanThreads) scan_tile_sums_kernel(const float* __restrict__ w, long long B,
                                                                     double* __restrict__ tile_sums) {
  __shared__ double sm[32];
  const long long base = (long long)blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) if (base + i < B) s += (double)w[base + i];   // sequential within a thread
  s = warp_sum(s);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) sm[wid] = s;
  __syncthreads();
  if (wid == 0) {
    double t = (lane < kScanThreads / 32) ? sm[lane] : 0.0;
    t = warp_sum(t);
    if (lane == 0) tile_sums[blockIdx.x] = t;
  }
}
// pass 2: exclusive scan of tile sums (single block, sequential chunks), total at tile_offs[num_tiles]
__global__ void __launch_bounds__(kScanThreads) scan_tile_offsets_kernel(const double* __restrict__ tile_sums,
                                                                        int num_tiles, double* __restrict__ tile_offs) {
  __shared__ double sm[32];
  __shared__ double total;
  double carry = 0.0;
  for (int base = 0; base < num_tiles; base += kScanThreads) {
    const int i = base + threadIdx.x;
    const double v = (i < num_tiles) ? tile_sums[i] : 0.0;
    const double ex = block_exclusive_scan(v, sm, &total);
    if (i < num_tiles) tile_offs[i] = carry + ex;
    carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) tile_offs[num_tiles] = carry;
}
// pass 3: cum[i] = (offset + inclusive prefix) / total
__global__ void __launch_bounds__(kScanThreads) scan_finalize_kernel(const float* __restrict__ w, long long B,
                                                                    const double* __restrict__ tile_offs, int num_tiles,
                                                                    double* __restrict__ cum) {
  __shared__ double sm[32];
  __shared__ double total_tile;
  const long long base = (long long)blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  double v[kScanItems];
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) { v[i] = (base + i < B) ? (double)w[base + i] : 0.0; s += v[i]; }
  double run = tile_offs[blockIdx.x] + block_exclusive_scan(s, sm, &total_tile);
  const double total = tile_offs[num_tiles];
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    run += v[i];
    if (base + i < B) cum[base + i] = run / total;
  }
}
// idx[i] = #{k : cum_k < u_i}  (searchsorted side='left'), clamped to B-1
__global__ void __launch_bounds__(kMixThreads) resample_search_kernel(const double* __restrict__ cum, long long B,
                                                                     const double* __restrict__ u, long long n,
                                                                     long long* __restrict__ idx) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double ui = u[i];
    long long lo = 0, hi = B;
    while (lo < hi) {
      const long long mid = lo + ((hi - lo) >> 1);
      if (__ldg(cum + mid) < ui) lo = mid + 1; else hi = mid;
    }
    idx[i] = lo < B - 1 ? lo : B - 1;
  }
}

// out[i, :] = x[idx[i], :]   (density_experiment.py:644).  One warp per row, lanes stride the row.
__global__ void __launch_bounds__(kMixThreads) gather_rows_kernel(const float* __restrict__ x, int D,
                                                                 const long long* __restrict__ idx, long long n,
                                                                 float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long i = warp; i < n; i += nwarps) {
    const float* src = x + idx[i] * (long long)D;
    float* dst = out + i * (long long)D;
    for (int j = lane; j < D; j += 32) dst[j] = __ldg(src + j);
  }
}

// ---- planning of an inverse launch over many components (gbnf_mixture_inverse) ------------------------------------------------
// A stable counting sort of the rows by component id: bins 0 .. n_comp - 1 are the components, bin n_comp takes the ids outside
// [0, n_comp) (status word [3] is raised and their rows are left out of the work units).  hist is bin-major [n_comp + 1][nblk]
// over blocks of kSortRows rows; the scan turns it into each (bin, block)'s first sorted position and writes the unit table.
constexpr int kSortRows = 1024;   // rows per block of the count and scatter kernels, one per thread

__device__ __forceinline__ int sort_bin(const long long* comp, long long i, long long B, int n_comp) {
  if (i >= B) return -1;
  const long long v = comp[i];
  return (v < 0 || v >= n_comp) ? n_comp : (int)v;
}

__global__ void __launch_bounds__(kSortRows) mix_sort_count_kernel(const long long* __restrict__ comp, long long B, int n_comp,
                                                                  int nblk, int* __restrict__ hist, int* status) {
  __shared__ int cnt[kMaxComponents + 1];
  for (int b = threadIdx.x; b <= n_comp; b += blockDim.x) cnt[b] = 0;
  __syncthreads();
  const int v = sort_bin(comp, (long long)blockIdx.x * kSortRows + threadIdx.x, B, n_comp);
  if (v == n_comp) *reinterpret_cast<volatile int*>(status + 3) = 1;
  if (v >= 0) atomicAdd(&cnt[v], 1);
  __syncthreads();
  for (int b = threadIdx.x; b <= n_comp; b += blockDim.x) hist[(long long)b * nblk + blockIdx.x] = cnt[b];
}

// One block: exclusive scan of hist in place, then the unit table -- component c's sorted segment cut into ceil(count_c / R)
// units of R rows (the last one shorter), components in order, empty components without units.  *n_units = the table's length
// (<= ceil(B / R) + n_comp).
__global__ void __launch_bounds__(kSortRows) mix_sort_scan_kernel(int* __restrict__ hist, int nblk, int n_comp, int R,
                                                                 int4* __restrict__ units, int* __restrict__ n_units) {
  __shared__ int wsum[kSortRows / 32];
  __shared__ int first[kMaxComponents + 1];    // first sorted row of each bin
  __shared__ int ufirst[kMaxComponents + 1];   // first unit of each component, then the unit count
  const int N = (n_comp + 1) * nblk;
  const int per = (N + kSortRows - 1) / kSortRows;
  const int lo = min(N, (int)threadIdx.x * per), hi = min(N, lo + per);
  int s = 0;
  for (int i = lo; i < hi; ++i) s += hist[i];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) wsum[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    const int w = wsum[lane];
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
    wsum[lane] = wi - w;
  }
  __syncthreads();
  int run = wsum[wid] + inc - s;
  for (int i = lo; i < hi; ++i) { const int v = hist[i]; hist[i] = run; run += v; }
  __syncthreads();
  for (int b = threadIdx.x; b <= n_comp; b += blockDim.x) first[b] = hist[(long long)b * nblk];
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int c = 0; c < n_comp; ++c) { ufirst[c] = t; t += (first[c + 1] - first[c] + R - 1) / R; }
    ufirst[n_comp] = t;
    *n_units = t;
  }
  __syncthreads();
  for (int c = 0; c < n_comp; ++c) {
    const int cnt = first[c + 1] - first[c], nu = ufirst[c + 1] - ufirst[c];
    for (int t = threadIdx.x; t < nu; t += blockDim.x) units[ufirst[c] + t] = make_int4(c, first[c] + t * R, min(R, cnt - t * R), 0);
  }
}

// perm[position] = row and iperm[row] = position: a row's position is its bin's first position in its block plus the rows of the
// same bin before it in the block (earlier warps' counts, then its rank among its warp's matching lanes), so the order is stable.
__global__ void __launch_bounds__(kSortRows) mix_sort_scatter_kernel(const long long* __restrict__ comp, long long B, int n_comp,
                                                                    int nblk, const int* __restrict__ hist,
                                                                    long long* __restrict__ perm, long long* __restrict__ iperm) {
  __shared__ int wcnt[kSortRows / 32][kMaxComponents + 1];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long i = (long long)blockIdx.x * kSortRows + threadIdx.x;
  const int v = sort_bin(comp, i, B, n_comp);
  const unsigned peers = __match_any_sync(0xffffffffu, v);
  const int rank = __popc(peers & ((1u << lane) - 1u));
  for (int w = 0; w < kSortRows / 32; ++w)
    for (int b = threadIdx.x; b <= n_comp; b += blockDim.x) wcnt[w][b] = 0;
  __syncthreads();
  if (v >= 0 && rank == 0) wcnt[wid][v] = __popc(peers);
  __syncthreads();
  if (v >= 0) {
    long long pos = hist[(long long)v * nblk + blockIdx.x] + rank;
    for (int w = 0; w < wid; ++w) pos += wcnt[w][v];
    perm[pos] = i;
    iperm[i] = pos;
  }
}

// The unit table of ONE component over rows in their own order (gbnf_component_inverse): unit t = rows [t R, min((t + 1) R, B)).
__global__ void component_units_kernel(int c, long long B, int R, int4* __restrict__ units, int* __restrict__ n_units) {
  const int nu = (int)((B + R - 1) / R);
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nu; t += gridDim.x * blockDim.x)
    units[t] = make_int4(c, t * R, (int)min((long long)R, B - (long long)t * R), 0);
  if (blockIdx.x == 0 && threadIdx.x == 0) *n_units = nu;
}

}  // namespace gbnf
