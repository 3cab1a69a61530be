/*
 * gbnf.h -- C ABI of the B200-native boosted-mixture density path (libgbnf_b200.so).
 *
 * Scope: the ONE hot path of robert-giaquinto/gradient-boosted-normalizing-flows named in BASELINE.json:
 * per-component log q_c(x) for C fixed RealNVP / Glow coupling stacks, the rho-weighted logsumexp mixture,
 * the boosting weights, inverse-CDF resampling.  The reference has no FFI (it is pure PyTorch); each entry
 * point below cites the reference Python it replaces (paths relative to the reference tree).
 *
 * Conventions
 *   - plain C types only; every pointer named d_* / documented "device" is a CUDA device pointer that the
 *     caller owns (PyTorch tensors in practice) and that is only BORROWED for the duration of the call;
 *   - all tensors are contiguous row-major, float32 unless stated; indices are int64;
 *   - every launch goes on the caller's stream (`stream` is a cudaStream_t passed as void*); no entry point
 *     synchronises unless documented (gbnf_pack_component in the f16 modes, gbnf_check_status, the diagnostics);
 *   - every entry point runs on the handle's device and restores the caller's current device before returning;
 *   - the kernels report through status words in mapped host memory, read (without a synchronisation) at the
 *     top of every entry point: an in-kernel watchdog timeout (GBNF_ERR_CUDA, with the code of the wait that
 *     timed out), a value that fp16 cannot hold entering a tensor-core GEMM operand (GBNF_ERR_NUMERIC) or a component id
 *     outside [0, n_comp) given to gbnf_mixture_inverse (GBNF_ERR_INVALID) is
 *     reported by the first call made after the offending launch finished; gbnf_check_status() synchronises the
 *     stream and reports at once;
 *   - fp16 tensor-core modes: inputs, activations and weights must be finite in fp16 (|v| <= 65504); density data
 *     is standardised upstream (utils/miniboone.py:57-65), raw data should use GBNF_GEMM_FP32;
 *   - every entry returns 0 on success or a negative gbnf_status; gbnf_last_error() gives the text
 *     (thread-local); no C++ exception crosses the boundary;
 *   - one handle per device; calls on one handle are not re-entrant;
 *   - there is NO CPU fallback: without a CUDA device gbnf_create fails with GBNF_ERR_CUDA.
 */
#ifndef GBNF_H_
#define GBNF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GBNF_ABI_VERSION 2   /* 2: gbnf_step_params.invconv_*, gbnf_config.glow_invconv, GBNF_ACT_RESIDUAL */
#define GBNF_MAX_LAYERS 6 /* depth + 2 <= 6 */

typedef struct gbnf_ctx* gbnf_handle;

typedef enum {
  GBNF_OK = 0,
  GBNF_ERR_INVALID = -1, /* bad argument / unsupported configuration */
  GBNF_ERR_CUDA = -2,    /* CUDA runtime error (text in gbnf_last_error) */
  GBNF_ERR_STATE = -3,   /* e.g. component not packed yet */
  GBNF_ERR_NUMERIC = -4  /* weights / inputs / activations not representable in the selected GEMM operand type */
} gbnf_status;

enum { GBNF_KIND_REALNVP = 0, GBNF_KIND_GLOW = 1 };              /* models/boosted_flow.py:44-50 */
enum { GBNF_ACT_TANH = 0, GBNF_ACT_RELU = 1, GBNF_ACT_MIXED = 2, /* models/realnvp.py:47-66 (mixed: t=ReLU, s=Tanh) */
       GBNF_ACT_RESIDUAL = 3 };   /* ResidualNet coupling networks (models/layers.py:246-301, selected at models/realnvp.py:59-60): Linear,
                                     `depth` pre-activation ReLU blocks of two Linears with a skip, Linear = 2 depth + 2 Linear layers in
                                     W[net][0 .. 2 depth + 1] (initial, block 0 first, block 0 second, ..., final); RealNVP only (upstream's Glow
                                     names ResidualNet without importing it, models/glow.py:294); depth <= 2,
                                     GBNF_GEMM_FP32 only (the tensor-core kernels keep activations as fp16 MMA operands: no skip path) */
enum { GBNF_COUPLING_AFFINE = 0, GBNF_COUPLING_ADDITIVE = 1 };     /* models/glow.py:326-338 */
enum { GBNF_BASE_STD_NORMAL = 0, GBNF_BASE_DIAG_NORMAL = 1 };     /* utils/distributions.py:44 | generative_flow.py:38-42 */
enum {
  GBNF_GEMM_FP32 = 0,  /* CUDA-core fp32 FMA, libm-accurate tanh: reference-class numerics (~1e-6 rel)          */
  GBNF_GEMM_F16_TC = 1, /* tcgen05 tensor cores, fp16 operands, fp32 accumulate in TMEM, tanh via ex2+rcp
                           (abs err ~1e-7): <= 1e-4 rel on log q                                                   */
  GBNF_GEMM_F16_TC_FAST = 2 /* same GEMMs, tanh.approx.f32 (one MUFU op, rel err 2^-11): <= 2e-4 rel on log q      */
};
/* Hidden widths in the f16 modes: coupling_network_depth 1 serves any h <= 1024 (D <= 64), depth > 1 any h <= 512.  The
 * kernels run the width padded with zero units (depth 1: h <= 512 to a multiple of 128 unless it is one of 64, h > 512 to
 * 1024; depth > 1: to a multiple of 64), which gives the results of the true width bit for bit.  Wider networks, and
 * depth > 1 above 512, need GBNF_GEMM_FP32. */
enum { GBNF_WEIGHTS_DENSITY = 0, GBNF_WEIGHTS_TOY = 1 }; /* density_experiment.py:627-641 | toy_experiment.py:440-459 */
enum {
  GBNF_MIX_SIMPLEX = 0,   /* logsumexp_c(log(rho_c / sum rho) + log q_c): density_experiment.py:612-622              */
  GBNF_MIX_RAW_RHO = 1,   /* the un-normalised-rho recursion of _rho_gradients: models/boosted_flow.py:132-133       */
  GBNF_MIX_GEOMETRIC = 2  /* sum_c rho_c log q_c / sum_c rho_c (components with rho_c == 0 left out): the "all
                             components" panel of plot_boosted_fwd_flow_density, utils/density_plotting.py:199-226;
                             only on materialised log q (gbnf_mixture_logdensity), not in gbnf_fused_eval          */
};

typedef struct {
  int32_t kind;      /* GBNF_KIND_* */
  int32_t D;         /* features (args.z_size) */
  int32_t h;         /* hidden width (args.h_size) */
  int32_t K;         /* coupling steps per component (args.num_flows) */
  int32_t C;         /* components (args.num_components) */
  int32_t depth;     /* args.coupling_network_depth (hidden->hidden layers) */
  int32_t act;       /* GBNF_ACT_* (args.coupling_network) */
  int32_t coupling;  /* GBNF_COUPLING_* (args.flow_coupling, glow only) */
  int32_t base;      /* GBNF_BASE_* */
  int32_t gemm_mode; /* GBNF_GEMM_* */
  int32_t device;    /* CUDA device ordinal */
  int32_t glow_invconv; /* 1: the Glow steps mix the channels with InvertibleConv1x1 (args.flow_permutation == 'invconv',
                           models/glow.py:275-278, models/layers.py:722-796) instead of Permute1d: a dense D x D step fused between
                           ActNorm and the coupling; gbnf_step_params.invconv_* are read and perm is ignored; GBNF_GEMM_FP32 only */
} gbnf_config;

/* Raw fp32 parameters of ONE coupling step, as they sit in the reference modules' tensors (device pointers).
 * Glow  (models/glow.py:265-308): an_bias/an_logs = ActNorm1d.bias/logs [D]; perm = Permute1d.indices int64 [D]
 *        (NOT in state_dict, models/layers.py:637); net 0 = block.network Linear layers.
 * RealNVP (models/realnvp.py:35-76): net 0 = t_net (flow_param[k][0]), net 1 = s_net (flow_param[k][1]);
 *        bn_* = flow_param[k][2] (log_gamma, beta, running_mean, running_var) or all NULL.
 * W[n][l] is nn.Linear.weight [out_features, in_features] row-major, b[n][l] its bias; l = 0 .. depth+1. */
typedef struct {
  const float* an_bias;
  const float* an_logs;
  const int64_t* perm;
  const float* bn_log_gamma;
  const float* bn_beta;
  const float* bn_mean;
  const float* bn_var;
  const float* W[2][GBNF_MAX_LAYERS];
  const float* b[2][GBNF_MAX_LAYERS];
  /* Glow with config.glow_invconv: the step's 1x1 convolution weight as InvertibleConv1x1.get_weight(reverse=False) returns it
   * (models/layers.py:751-779; LU-decomposed or plain), [D, D] row-major, z_out[i] = sum_j w[i][j] z_in[j]; its inverse (NULL:
   * the sampling direction is refused for this component); and ONE float = dlogdet for a feature vector (sum(log_s) or
   * slogdet(weight)).  NULL for every other configuration. */
  const float* invconv_w;
  const float* invconv_winv;
  const float* invconv_logdet;
} gbnf_step_params;

typedef struct {
  int32_t flip_init;             /* RealNVPFlow(flip_init=c), models/boosted_flow.py:46 */
  int32_t n_steps;               /* must equal config.K */
  const gbnf_step_params* steps; /* HOST array of n_steps entries holding DEVICE pointers */
} gbnf_component_params;

/* ---- lifecycle -------------------------------------------------------------------------------------- */
/* Replaces BoostedFlow.__init__'s device-side state (models/boosted_flow.py:22-50). */
int gbnf_create(gbnf_handle* out, const gbnf_config* cfg);
void gbnf_destroy(gbnf_handle h);
const char* gbnf_last_error(void);
int gbnf_abi_version(void);

/* Re-tile one component's parameters into the handle's packed blob (device -> device, on `stream`).
 * Call after construction, after every load() (utils/utilities.py:42-75) and whenever a component's
 * parameters changed before it is evaluated as a fixed component.  In the f16 modes this call SYNCHRONISES the
 * stream (it reads the fp16 weight-overflow word and returns GBNF_ERR_NUMERIC when a weight is not finite in fp16). */
int gbnf_pack_component(gbnf_handle h, int32_t c, const gbnf_component_params* p, void* stream);

/* Toy path base density Normal(mean[D], scale[D]) (models/generative_flow.py:22-23,38-42). Device pointers; the
 * vectors are COPIED (stream-ordered), the caller's tensors are not referenced after the call. */
int gbnf_set_base(gbnf_handle h, const float* d_mean, const float* d_scale, void* stream);

/* ---- the hot path ----------------------------------------------------------------------------------- */
/* log q_c(x) for c in [c0, c1): replaces the loop `model(x=x, components=c)` + log_normal_standard(z)+ldj
 * (density_experiment.py:613-616, models/boosted_flow.py:220-228, models/glow.py:92-110,
 * models/realnvp.py:115-127).  d_logq is [B, c1-c0].  d_z_opt [B, D] / d_ldj_opt [B] (may be NULL) receive the
 * flow output of component c0 and require c1 == c0+1 (the 5-tuple's z and log_det_j). */
int gbnf_component_logq(gbnf_handle h, const float* d_x, int64_t B, int32_t c0, int32_t c1, float* d_logq,
                        float* d_z_opt, float* d_ldj_opt, void* stream);

/* Inverse direction (sampling): x = f_c^{-1}(z) for ONE component -- the exact inverse of gbnf_component_logq's flow, walked
 * from the last coupling step to the first (coupling^-1, permutation^-1, ActNorm^-1 / eval-BatchNorm^-1).  Replaces
 * `model(z=z, components=c, reverse=True)`: models/boosted_flow.py:209-218, models/glow.py:112-123,344-366,
 * models/realnvp.py:97-113 (upstream's RealNVP decode pairs the wrong halves and its 1-D affine Glow decode raises; this is
 * the mathematical inverse, pinned by decode(encode(x)) == x and by the reference's additive-Glow decode).
 * d_z [B, D] in the flow's output column order, d_x [B, D]; d_ldj_opt [B] (may be NULL) receives the log-det of the
 * inverse map (= -log_det_j of the forward map at x).  Served in GBNF_GEMM_FP32 and, in the f16 tensor-core modes, by the
 * pipelined kernel (depth 1, hidden width up to 512 except 64, 192, 320 and 448) and the CTA-pair kernel (depth 1,
 * 512 < h <= 1024, Glow and RealNVP); handles that run the serial tensor-core kernel (depth > 1, or h = 64 / 192 / 320 /
 * 448) return GBNF_ERR_INVALID. */
int gbnf_component_inverse(gbnf_handle h, const float* d_z, int64_t B, int32_t c, float* d_x, float* d_ldj_opt, void* stream);

/* x[i] = f_{comp[i]}^{-1}(z[i]) for every row i; comp[i] in [0, n_comp).  One coupling launch over all components.  No host
   synchronisation.  The log-det of the inverse map goes to d_ldj_opt when it is not NULL.
 * Sampling from the whole mixture (models/boosted_flow.py:209-218 with a component per sample): d_comp is int64 [B] (device), in
 * any order.  The rows are sorted by component on the device (a stable counting sort), z is gathered into that order, one inverse
 * launch covers every component's rows, and x / ldj are gathered back to the caller's order; each row gets the bits
 * gbnf_component_inverse gives it.  Components 0 .. n_comp - 1 must be packed, and served as for gbnf_component_inverse (the same
 * refusals, before anything is written).  An id outside [0, n_comp) is found on the device: its rows are left out and the next
 * entry point, or gbnf_check_status, returns GBNF_ERR_INVALID.  The scratch (8 D + 20 bytes a row, up to 2^22 rows
 * a launch; larger batches go through in slices) is kept on the handle and grows with B: after one call at a batch size, calls
 * at that size allocate nothing, so they can be captured in a CUDA graph. */
int gbnf_mixture_inverse(gbnf_handle h, const float* d_z, int64_t B, const int64_t* d_comp, int32_t n_comp,
                         float* d_x, float* d_ldj_opt, void* stream);

/* Mixture log-density from materialised per-component log q (d_logq is [B, ld], first n_comp columns used):
 * the 2-term logsumexp recursion of density_experiment.py:612-622 / :561-571 evaluated in its flat form
 * G = logsumexp_c(coef_c + logq_c) (SURVEY 8 a9).  d_rho is the RAW rho buffer [>= n_comp] (device);
 * skip_c >= 0 leaves that component out as toy_experiment.py:414-417 does (-1: none);
 * mix_mode GBNF_MIX_RAW_RHO reproduces BoostedFlow._rho_gradients (models/boosted_flow.py:124-134);
 * GBNF_MIX_GEOMETRIC returns the rho-weighted MEAN of log q_c (the log of the grid density that
 * utils/density_plotting.py:185-226 plots for the whole model).
 * n_comp == 0 writes zeros (density_experiment.py:612). */
int gbnf_mixture_logdensity(gbnf_handle h, const float* d_logq, int64_t B, int32_t ld, int32_t n_comp,
                            const float* d_rho, int32_t skip_c, int32_t mix_mode, float* d_G_ll, void* stream);

/* Single-pass fused path: components [0, n_comp) + mixture; the [B, C] matrix never goes to HBM unless
 * d_logq_opt (ld = n_comp) is given.  (The batch softmax statistics of -G_ll are NOT a by-product of this call:
 * gbnf_boost_weights makes its own one-sweep reduction over G_ll, 4 bytes per row -- 0.4 % of the fused step at the
 * headline configuration, profiles/r02c_launches_cfg3_steps.csv.) */
int gbnf_fused_eval(gbnf_handle h, const float* d_x, int64_t B, int32_t n_comp, const float* d_rho,
                    int32_t skip_c, int32_t mix_mode, float* d_G_ll, float* d_logq_opt, void* stream);

/* Boosting weights (utils/utilities.py:12-14 + density_experiment.py:627-641; toy_experiment.py:440,453-459):
 * w = softmax_B(-G_ll); density: if max w > clamp_hi: clip to [clamp_lo, clamp_hi]; if sum != 1: renormalise.
 * toy: renormalise; if max w > clamp_hi: clip, renormalise.   d_stats (device, 4 floats, may be NULL) receives
 * {max_B(-G_ll), sum_B exp(-G_ll - max), clamped flag, sum w before the final renormalisation}. */
int gbnf_boost_weights(gbnf_handle h, const float* d_G_ll, int64_t B, float clamp_lo, float clamp_hi,
                       int32_t mode, float* d_w, float* d_stats, void* stream);

/* The same in three stages, for batch-parallel multi-GPU runs where the two batch reductions are all-reduced
 * between the stages by the caller (torch.distributed / NCCL):
 *   stage 1: d_ms[0] = max_B(-G_ll), d_ms[1] = sum_B exp(-G_ll - d_ms[0])               (local shard)
 *   stage 2: w from global (max, sum); clamp decision from the global sum; d_wsum[0] = local sum of w (fp64)
 *   stage 3: w *= 1/d_wsum[0] when d_wsum[0] != 1                                         (global sum) */
int gbnf_weight_stats(gbnf_handle h, const float* d_G_ll, int64_t B, float* d_ms, void* stream);
int gbnf_weight_apply(gbnf_handle h, const float* d_G_ll, int64_t B, const float* d_ms, float clamp_lo,
                      float clamp_hi, int32_t mode, float* d_w, double* d_wsum, void* stream);
int gbnf_weight_renorm(gbnf_handle h, float* d_w, int64_t B, const double* d_wsum, int32_t mode, void* stream);

/* ---- training step of the NEW component (density_experiment.py:647-661, 361-374) ------------------------------
 * Gradients of any loss L(z, log_det_j) of component c's flow with respect to all of its parameters, given the upstream
 * gradients dL/dz [B, D] and dL/dlog_det_j [B] (for the boosted objective nll = mean(-(log N(z) + ldj)): dz = z / B,
 * dldj = -1 / B).  Recompute-in-kernel: the forward value comes from gbnf_component_logq and saves nothing; this call
 * recomputes the activations (fp32 CUDA-core arithmetic, reference-class numerics) and runs the backward sweep.
 * `p` holds the component's CURRENT raw parameters (as for gbnf_pack_component), `grads` the same tensors' gradient
 * buffers, which are OVERWRITTEN.  Glow components with a permutation (tanh / relu) and RealNVP components WITHOUT BatchNorm
 * (tanh / relu / mixed; models/transformations.py:560-579 -- train-mode BatchNorm couples the rows of a batch), with
 * every coupling_network_depth gbnf_create accepts (0 to 4: W / b / grads carry depth + 2 layers per network), h <= 512,
 * D <= 64.  The per-row kernel keeps every step's input and coupling-network outputs in shared memory, so
 * K x (D + 64 x networks per step) must fit in it beside the h-wide activation rows (227 KB in all; the hidden layers of a
 * deeper network reuse the same rows, so this bound does not depend on the depth): the deepest component served at
 * D = 2 / 21 / 43 / 64 is, at h = 512, K = 27 / 20 / 15 / 12 for Glow and 14 / 11 / 9 / 8 for RealNVP; at h = 64,
 * K = 47 / 36 / 28 / 23 and 24 / 20 / 17 / 15.  The device scratch the call keeps (B x K x (2 (depth + 1) x round_up(h, 64)
 * + 64) floats per network) grows with the depth; an allocation failure returns GBNF_ERR_CUDA before `grads` is written.
 * Other configurations return GBNF_ERR_INVALID before anything is written (`grads` and the handle stay as they were) and
 * train through the caller's autograd.
 * d_dx_opt [B, D] (may be NULL) receives dL/dx. */
typedef struct {
  float* an_bias;
  float* an_logs;
  float* W[2][GBNF_MAX_LAYERS];
  float* b[2][GBNF_MAX_LAYERS];
} gbnf_step_grads;
int gbnf_component_backward(gbnf_handle h, int32_t c, const gbnf_component_params* p, const float* d_x, int64_t B,
                            const float* d_dz, const float* d_dldj, const gbnf_step_grads* grads, float* d_dx_opt,
                            void* stream);

/* ---- sampling with gradients: backward of the inverse map (reparameterised samples, BoostedFlow.rsample) -------------------
 * Gradients of any loss L(x, ldj_inv) of the inverse map x = f_c^{-1}(z) (gbnf_component_inverse / gbnf_mixture_inverse) with
 * respect to the parameters of the components, given the upstream gradients dL/dx [B, D] and dL/dldj_inv [B] (for reverse KL,
 * log q_c(x) = log N(z) - ldj_inv).  Recompute-in-kernel from z: the forward call saves nothing and its scratch is not read (other
 * inverse calls may run in between); fp32 CUDA-core arithmetic whatever the GEMM mode.  The same envelope, shared-memory bound and
 * scratch as gbnf_component_backward: Glow components with a permutation (tanh / relu, affine or additive) and RealNVP components
 * WITHOUT BatchNorm (tanh / relu / mixed), coupling_network_depth 0 to 4, h <= 512, D <= 64, K within the bound listed there;
 * 1 <= B <= 2^22.  The components must be packed (as for the forward call).  `p` holds their CURRENT raw parameters, `grads` the
 * gradient buffers, which are OVERWRITTEN (a component that drew no rows gets zeros).  Every refusal (GBNF_ERR_INVALID for a
 * configuration outside the envelope, GBNF_ERR_STATE for an unpacked component) comes before anything is written: `grads`,
 * d_dz_opt and the handle stay as they were.  Weight and bias gradients are deterministic (no atomics); the ActNorm gradients
 * are accumulated with atomics.  No host synchronisation.  d_dz_opt [B, D] (may be NULL) receives dL/dz.
 *   gbnf_component_inverse_backward: component c, d_z in row order.
 *   gbnf_mixture_inverse_backward:   x[i] = f_{comp[i]}^{-1}(z[i]) as for gbnf_mixture_inverse: p[n_comp] (host array), grads[n_comp]
 *                                    (host array; grads[c] == NULL: component c needs no parameter gradient).  The rows are
 *                                    sorted by component on the device again; the weight gradients of component c sum its rows in
 *                                    their order, so they equal, bit for bit, a gbnf_component_inverse_backward call on those rows
 *                                    alone.  An id outside [0, n_comp) is reported as for gbnf_mixture_inverse (its row's dz is
 *                                    not written). */
int gbnf_component_inverse_backward(gbnf_handle h, int32_t c, const gbnf_component_params* p, const float* d_z, int64_t B,
                                    const float* d_dx, const float* d_dldj, const gbnf_step_grads* grads, float* d_dz_opt,
                                    void* stream);
int gbnf_mixture_inverse_backward(gbnf_handle h, const gbnf_component_params* p, const float* d_z, int64_t B,
                                  const int64_t* d_comp, int32_t n_comp, const float* d_dx, const float* d_dldj,
                                  const gbnf_step_grads* const* grads, float* d_dz_opt, void* stream);

/* ---- multi-GPU on one node: one process per GPU, values exchanged through PEER MEMORY over NVLink ------------
 * The reference has no distributed code (SURVEY 2); this is the library-owned collective SURVEY 8(b) lists as
 * gbnf_comm_init.  No NCCL call sits on the data path: a rank publishes a value by storing it into every rank's
 * exchange block (cudaIpc-mapped device memory) followed by a flag word, and consumes by spinning on its own block
 * inside the kernel that needs the value (bounded: a missing peer raises watchdog code 40 after ~2 s).
 *   1. every rank: gbnf_comm_local_handle(h, max_rows, handle64)   allocates its block (+ a COMPONENT-major [2][C][max_rows]
 *      gather buffer for the component-parallel layout: 128 consecutive rows of one component are one contiguous NVLink
 *      write; max_rows MUST be the same on every rank, it is the buffer's row stride) and returns the 64-byte
 *      cudaIpcMemHandle_t;
 *   2. the caller all-gathers the handles with whatever plumbing it has (torch.distributed in gbnf_b200/dist.py);
 *   3. every rank: gbnf_comm_init(h, rank, world, handles[world][64]); a barrier; then, in the SAME order on every rank:
 *   gbnf_boost_weights_dist          batch-parallel: this rank's rows, boosting weights under the GLOBAL batch softmax
 *                                    (density_experiment.py:627-641 on the union of all shards); every rank merges the
 *                                    ranks' (max, sum exp) and sum-of-weights in rank order -> bitwise identical scalars
 *   gbnf_mixture_component_parallel  component-parallel: rank g evaluates components [g n/G, (g+1) n/G) of ALL rows, the
 *                                    coupling kernel's epilogue stores log q straight into every rank's gather buffer,
 *                                    the mixture kernel waits for all blocks (density_experiment.py:612-622)
 *   gbnf_comm_destroy (after a barrier: peers must have stopped writing). world <= 8. */
int gbnf_comm_local_handle(gbnf_handle h, int64_t max_rows, void* out_handle64);
int gbnf_comm_init(gbnf_handle h, int32_t rank, int32_t world, const void* all_handles);
int gbnf_comm_destroy(gbnf_handle h);
int gbnf_boost_weights_dist(gbnf_handle h, const float* d_G_ll, int64_t B, float clamp_lo, float clamp_hi, int32_t mode,
                            float* d_w, float* d_stats, void* stream);
int gbnf_mixture_component_parallel(gbnf_handle h, const float* d_x, int64_t B, int32_t n_comp, const float* d_rho,
                                    int32_t skip_c, int32_t mix_mode, float* d_G_ll, void* stream);

/* Inverse-CDF resampling, the contract that pins torch.multinomial(w, B, replacement=True)
 * (density_experiment.py:643): idx[i] = #{k : cum_k < u_i}, cum = cumsum_fp64(w) / sum_fp64(w).
 * d_u: float64 uniforms [n] (device). */
int gbnf_resample(gbnf_handle h, const float* d_w, int64_t B, const double* d_u, int64_t n, int64_t* d_idx,
                  void* stream);

/* x_resampled = x[idx] (density_experiment.py:644). d_out [n, D]. */
int gbnf_gather_rows(gbnf_handle h, const float* d_x, int32_t D, const int64_t* d_idx, int64_t n, float* d_out,
                     void* stream);

/* Data-dependent ActNorm initialisation from one batch (ActNorm.initialize_parameters, models/layers.py:473-486):
 * bias[c] = -mean_B x[:, c]; logs[c] = log(scale / (sqrt(mean_B (x[:, c] + bias[c])^2) + 1e-6)).  d_x [B, D], d_bias / d_logs [D]
 * (device).  Needs no handle: it runs on the CURRENT device, on the caller's stream, before any component is packed. */
int gbnf_actnorm_init(const float* d_x, int64_t B, int32_t D, float scale, float* d_bias, float* d_logs, void* stream);

/* Host helper: component id under the same CDF rule for "1:c" / "1:c-1" / "-c" (models/boosted_flow.py:76-91).
 * rho_host is a HOST array; exclude >= 0 zeroes that entry first. */
int gbnf_sample_component(const float* rho_host, int32_t n, double u, int32_t exclude, int32_t* j_out);

/* ---- introspection (tests, bench) ------------------------------------------------------------------- */
typedef struct {
  int32_t gemm_mode;       /* as configured */
  int32_t rows_per_cta;    /* row-tile height of the coupling kernel */
  int32_t smem_bytes;      /* dynamic shared memory per CTA */
  int32_t tmem_cols;       /* TMEM columns allocated per CTA (0 for the fp32 path) */
  int32_t num_sms;         /* SMs on the device */
  int32_t grid;            /* CTAs launched by the last coupling launch */
  int64_t packed_bytes;    /* size of the packed parameter blob */
  int64_t launches;        /* kernels launched through this handle so far */
  int32_t pipelined;       /* 2: CTA-pair tensor-core kernel for 512 < h <= 1024 (coupling_tc3.cuh), 1: chunk-pipelined tensor-core
                              kernel (coupling_tc2.cuh), 0: serial tensor-core / fp32 kernel */
  int32_t two_chain;       /* 1: the last coupling launch ran the two-chain schedule (coupling_tc4.cuh: Glow / affine / tanh, h = 512,
                              an even number of components per work unit); 2: the interleaved s / t schedule (coupling_tc5.cuh:
                              RealNVP / tanh, h = 256) */
} gbnf_info;
int gbnf_get_info(gbnf_handle h, gbnf_info* out);

/* Synchronises `stream` and returns the status the kernels left (GBNF_OK, GBNF_ERR_NUMERIC, or GBNF_ERR_CUDA with the
 * watchdog code in gbnf_last_error).  The drop-in's NaN guard (density_experiment.py:671-672) calls this. */
int gbnf_check_status(gbnf_handle h, void* stream);

/* Cycle counters of CTA 0 of the last tensor-core coupling launch (synchronises the device; diagnostics only):
 * [0..7] MMA warp: total, wait a_ready, wait weights, issue; [8..15] epilogue thread 0: total, wait accumulator,
 * hidden epilogues, last-layer/coupling, prologue (load/affine/gather); [16..] producer: total, wait empty. */
int gbnf_get_profile(gbnf_handle h, int64_t* out32);

/* Event trace (clock64 stamps) of one coupling pass of CTA 0 of the last pipelined tensor-core launch made with
 * GBNF_PROF=1 in the environment; 256 entries, layout in tools/tc_trace.py (synchronises; diagnostics only). */
int gbnf_get_trace(gbnf_handle h, int64_t* out256);

#ifdef __cplusplus
}
#endif
#endif /* GBNF_H_ */
