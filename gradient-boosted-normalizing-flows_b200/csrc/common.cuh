// Shared definitions for the GBNF B200 kernels: packed-parameter layout, small device helpers.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include "../../include/gbnf.h"

namespace gbnf {

constexpr int kMaxComponents = 256;   // coef table in shared memory
constexpr int kMaxD = 256;
constexpr int kMaxRanks = 8;            // GPUs of one node that can share an exchange (gbnf_comm_init)
constexpr int kEpPad = 64;             // padded length of the gather-order step tables

// ---- packed parameter layout ---------------------------------------------------------------------------
// One Linear layer of one coupling net (nn.Linear weight [N_out, K_in], models/layers.py:218-239).
//   fp32 path : wblob holds Wt[Kp][Np] float (transposed, N contiguous), Kp % 32 == 0, Np % 64 == 0, zero padded.
//   f16 path  : wblob holds Kp/16 "k-slabs"; slab s is the UMMA canonical K-major no-swizzle image of
//               W[0:Np, 16s:16s+16]:  [Np/8 row groups][2 k-chunks][8 rows][8 halves]  (SBO = 256 B, LBO = 128 B),
//               Kp % 16 == 0, Np % 16 == 0, zero padded.  A slab is Np*32 bytes and is what one bulk-TMA moves.
//               With NC < Np (pipelined kernel, coupling_tc2.cuh) the image is N-chunk major:
//               [Np/NC chunks][Kp/16 k-slabs][NC x 16] with the same canonical layout inside each NC x 16 slab.
struct LayerDesc {
  int K_in, N_out, Kp, Np;
  int NC, NC2;       // N-chunk width of the f16 image (== Np for the single-chunk layout); NC2 != 0: width of the odd
                     // chunks (chunk widths alternate NC, NC2, NC, ...: h = 512 in the pipelined kernel uses 128 / 64)
  long long w_off;   // element offset into wblob (float for fp32, __half for f16)
  long long b_off;   // float offset into fblob; Np entries, zero padded
};

// One coupling step of one component.  The kernels never physically permute z: column j of the reference's
// tensor lives at physical column sigma[j] of the resident row and the composed maps are resolved at pack time
// (models/layers.py:661-668 Permute1d, models/transformations.py:568-576 flip).
struct StepDesc {
  int in_dim, out_dim;   // |z1| (MLP input), |z2| (transformed half)
  int has_affine;        // ActNorm1d (glow) or eval-mode BatchNorm (realnvp) present
  int has_invconv;       // Glow: a dense D x D step (InvertibleConv1x1) follows the ActNorm instead of a permutation (fp32 path)
  long long vec_off;     // fblob: add[Dv] | mul[Dv] | off[Dv]  (physical column order), y = (z + add) * mul + off
  long long idx_off;     // iblob: idx1[in_dim] | idx2[out_dim]  physical columns of z1 / z2
  // Branch-free tables of the pipelined tensor-core kernel, in GATHER order and padded to kEpPad entries:
  //   fblob @ ep_off  : float4 {add, mul, off, column as int bits}[kEpPad] in z1 order, then the same in z2 order
  //                     (16-byte aligned); padding has mul = 0 (yields 0) and points at the scratch column D; then the two
  //                     tables of the INVERSE affine {-off, 1 / mul, -add, column}[kEpPad] (sampling direction)
  long long ep_off;
  long long eidx_off;
  // invconv (fp32 path): wblob float offsets of the forward / inverse matrices in the GEMM layout Wt[Kp][Np] (k = physical input
  // column, n = physical output column; the permutation composed so far is folded in at pack time) and a zero bias [Np] in fblob
  long long icw_off, icwinv_off, icb_off;
  int ic_Kp, ic_Np;
  LayerDesc layer[2][GBNF_MAX_LAYERS];   // net 0: glow block / realnvp t_net; net 1: realnvp s_net
};

struct CompDesc {
  long long sigma_off;   // iblob: final logical->physical map [D]
  long long const_off;   // fblob: [0] = sum of all data-independent log-det terms, [1] = packed flag
  long long base_off;    // fblob: mean_phys[Dv] | inv2var_phys[Dv]  (toy base), [2*Dv] = -sum(log s) - D/2 log 2pi
  long long dense_off;   // fblob: {fblob[const_off], fblob[base_off + 2*Dv]} again, in a dense per-component float2 table
                         // (CouplingArgs::cc_off + 2 c): one independent load instead of descriptor -> offset -> value
};

struct ModelDims {
  int kind, D, Dv, h, K, C, depth, act, coupling, base, nlayers, nnets;
};

// ---- kernel argument block -----------------------------------------------------------------------------
struct CouplingArgs {
  const float* x;
  long long B;
  int c0, c1;
  float* logq;   int ld_logq;      // nullable
  float* z_out;  float* ldj_out;   // nullable (c1 == c0 + 1)
  const float* rho; int n_mix; int skip_c; int mix_mode; float* G_ll;   // G_ll nullable
  const StepDesc* steps;           // [C*K]
  const CompDesc* comps;           // [C]
  const float* fblob;
  const int* iblob;
  const void* wblob;
  long long cc_off;                // fblob: dense float2 table of per-component constants (CompDesc::dense_off)
  ModelDims md;
  int num_tiles;
  // pipelined kernel only: a row tile's components are split over `split` work units (better wave quantisation, more
  // CTAs for small batches).  Every unit leaves its terms coef_c + log q_c in lse_terms; the last unit of a tile to
  // arrive reduces them in component order, so G_ll does not depend on the split (nor on the batch size).
  int split, comps_per_unit, num_units;
  float* lse_terms;                // [num_tiles * 128][n_mix]
  unsigned int* tile_ctr;          // [num_tiles], zero between launches (reset by the last arriver)
  // component-parallel multi-GPU (gbnf_mixture_component_parallel): when n_peers > 0 every log q value is ALSO stored into the
  // gather buffer of every rank (peer memory over NVLink): COMPONENT-major, element (row, peer_col0 + (c - c0)) at
  // [(peer_col0 + c - c0) * peer_ld + row], so that the 32 rows of a warp form one 128-byte NVLink write per peer
  float* logq_peers[kMaxRanks];
  int n_peers, peer_ld, peer_col0;
  int terms_only;                  // 1: write the mixture terms of [c0, c1) but leave the tile's logsumexp to a LATER launch of the
                                   // remaining components (an odd number of components: two-chain kernel on the even part, then
                                   // the single-chain kernel on the last component, which reduces all n_mix terms)
  int* error_flag;                 // status words in MAPPED HOST memory (the host can read them after a trap, without a
                                   // synchronisation): [0] watchdog code of a timed-out wait, [1] fp16 weight overflow (pack),
                                   // [2] a value entering an fp16 GEMM operand was not finite in fp16
  long long* prof;                 // optional cycle counters (CTA 0), see gbnf_get_profile
};

// ---- peer-memory exchange between the ranks of one node (one process per GPU; gbnf_comm_init) ---------------------------------
// Every rank owns one CommBlock in its own HBM, exported with cudaIpcGetMemHandle and mapped by all peers.  A rank PUBLISHES a
// value by storing it into slot [parity][its rank] of EVERY rank's block (plain stores over NVLink), then a system-scope fence,
// then the epoch number into the matching flag word; a rank CONSUMES by spinning on the flags of its OWN block (local L2) until
// they show the current epoch.  Slots are double buffered by epoch parity: a rank cannot run two epochs ahead of a peer, because
// passing epoch e + 1's wait needs the peer's e + 1 value, which the peer only publishes after all its epoch-e reads.
struct CommBlock {
  float ms[2][kMaxRanks][2];              // batch softmax statistics (max, sum exp) of each rank's row shard
  unsigned int ms_flag[2][kMaxRanks];
  double wsum[2][kMaxRanks];              // sum of the (clamped) weights of each rank's row shard
  unsigned int ws_flag[2][kMaxRanks];
  unsigned int done_flag[2][kMaxRanks];   // component-parallel: rank r has written its log q block into everybody's gather buffer
};
struct CommView {
  CommBlock* blk[kMaxRanks];              // blk[r]: rank r's block (blk[rank] is local)
  float* gather[kMaxRanks];               // gather[r]: rank r's [2][cap_rows * ld] log q gather buffers
  long long gather_stride;                // floats per parity buffer
  int rank, world;
  unsigned int epoch;
};
constexpr long long kCommSpinLimit = 4000000000LL;   // ~2 s: a missing peer must not hang the GPU
__device__ __forceinline__ void comm_wait_flag(const unsigned int* flag, unsigned int epoch, int* status) {
  const volatile unsigned int* f = flag;
  if (*f == epoch) return;
  const long long t0 = clock64();
  while (*f != epoch) {
    if (clock64() - t0 > kCommSpinLimit) {
      if (status) *reinterpret_cast<volatile int*>(status) = 40;
      __threadfence_system();
      __trap();
    }
  }
}

// ---- device helpers ------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Flat-form mixture coefficients (SURVEY 8 a9): coef[c] = log r_c + sum_{j>c, j!=skip} log(1 - r_j), r_0 = 1,
// r_c = rho_c / sum_{j<=c} rho_j (GBNF_MIX_SIMPLEX, density_experiment.py:618) or rho_c (GBNF_MIX_RAW_RHO,
// models/boosted_flow.py:132-133).  Non-participating components get -inf.  Called by ONE thread.
__device__ inline void mixture_coefficients(const float* __restrict__ rho, int n, int skip_c, int mix_mode,
                                            float* coef) {
  double acc = 0.0;   // sum_{j > c} log(1 - r_j)
  double pre = 0.0;
  for (int c = 0; c < n; ++c) pre += (double)rho[c];
  for (int c = n - 1; c >= 0; --c) {
    double r = 1.0;
    if (c > 0) r = (mix_mode == GBNF_MIX_RAW_RHO) ? (double)rho[c] : (double)rho[c] / pre;
    pre -= (double)rho[c];
    if (c == skip_c) { coef[c] = -INFINITY; continue; }
    coef[c] = (float)(log(r) + acc);
    if (c > 0) acc += log(1.0 - r);
  }
}

// Online logsumexp accumulator: (m, s) such that the running value is m + log s.
struct OnlineLse {
  float m, s;
  __device__ __forceinline__ void init() { m = -INFINITY; s = 0.f; }
  __device__ __forceinline__ void add(float t) {
    if (t == -INFINITY) return;
    if (t > m) { s = s * expf(m - t) + 1.f; m = t; }
    else       { s += expf(t - m); }
  }
  // torch.logsumexp semantics: no finite term -> -inf, a NaN term -> NaN, a +inf term -> +inf (the n_mix == 0 case
  // "G_ll = zeros", density_experiment.py:612, is handled on the host with a memset and never reaches this)
  __device__ __forceinline__ float value() const { return (s == 0.f) ? -INFINITY : m + logf(s); }
};

}  // namespace gbnf
