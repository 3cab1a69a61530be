// C-ABI entry points of libgbnf_b200.so (declared in include/gbnf.h).  Host-side planning of the packed layout,
// workspace management and kernel launches.  No torch types, no exceptions across the boundary.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "pack.cuh"
#include "mixture.cuh"
#include "actnorm_init.cuh"
#include "coupling_fp32.cuh"
#include "coupling_tc.cuh"
#include "coupling_tc2.cuh"
#include "coupling_tc3.cuh"
#include "coupling_tc4.cuh"
#include "coupling_tc5.cuh"
#include "train_bwd.cuh"

using namespace gbnf;

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e_ = (expr);                                                                    \
    if (e_ != cudaSuccess)                                                                      \
      return fail(GBNF_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));           \
  } while (0)

// Every entry point runs on the handle's device and leaves the caller's current device as it found it (a single-process
// multi-GPU PyTorch program must not have its current device changed behind its back).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
inline long long round_up_ll(long long v, long long m) { return (v + m - 1) / m * m; }

}  // namespace

// The coupling kernel a handle plans for its shape: fp32 (coupling_fp32.cuh), serial (coupling_tc.cuh), pipelined
// (coupling_tc2.cuh) or CTA pair for h = 1024 (coupling_tc3.cuh), at the padded width of plan_layout.
enum class CouplingKernel { kFp32, kSerial, kPipelined, kPair };
// A shape-specific kernel a launch of a pipelined plan may take instead (the values are gbnf_info::two_chain): the two-chain
// schedule for Glow / affine / tanh at h = 512 (coupling_tc4.cuh) or the interleaved s / t networks for RealNVP / tanh at h = 256
// (coupling_tc5.cuh).  The two shapes never overlap.
enum class AltKernel { kNone = 0, kTwoChain = 1, kInterleaved = 2 };

struct gbnf_ctx {
  gbnf_config cfg{};
  ModelDims md{};
  int num_sms = 0;
  std::vector<StepDesc> steps_h;
  std::vector<CompDesc> comps_h;
  std::vector<char> packed;
  std::vector<char> inv_ok;      // invconv components: 0 when the pack came without the inverse matrices
  StepDesc* steps_d = nullptr;
  CompDesc* comps_d = nullptr;
  float* fblob = nullptr;
  int* iblob = nullptr;
  void* wblob = nullptr;
  long long f_count = 0, i_count = 0, w_bytes = 0, cc_off = 0;
  float* base_mean = nullptr;    // handle-owned copies of the toy base density vectors [D] (gbnf_set_base)
  float* base_scale = nullptr;
  bool base_set = false;
  gbnf_step_params* step_params_d = nullptr;
  // workspace
  float* partial = nullptr;      // [max_grid][2]
  unsigned int* ticket = nullptr;
  float* ms = nullptr;           // [2]
  double* wsum = nullptr;        // [1]
  double* cum = nullptr;         // [cap]
  double* tile_sums = nullptr;   // [cap_tiles]
  double* tile_offs = nullptr;   // [cap_tiles + 1]
  long long cum_cap = 0;
  int* flags_host = nullptr;     // status words in mapped pinned host memory: [0] watchdog code of a timed-out in-kernel wait,
  int* flags = nullptr;          // [1] fp16 weight overflow (pack), [2] non-finite fp16 GEMM operand; `flags` = device alias
  float* lse_part = nullptr;     // pipelined kernel: per-row mixture terms coef_c + log q_c (reduced by the last unit of a tile)
  unsigned int* tile_ctr = nullptr;
  long long lse_cap = 0, ctr_cap = 0;
  long long* prof = nullptr;     // [32] cycle counters + [32..288) event trace written by CTA 0 of the tensor-core kernel
  // coupling launch plan
  int rows_per_cta = 0, ld = 0, out_max = 0, tmem_cols = 0;
  size_t smem_bytes = 0;
  CouplingKernel kernel = CouplingKernel::kFp32;
  TcPlan tc{};                   // plan of `kernel` (tensor-core kernels)
  AltKernel alt = AltKernel::kNone;   // the alternative a launch of a pipelined plan may take for this shape
  TcPlan alt_plan{};
  AltKernel last_alt = AltKernel::kNone;   // the alternative the most recent coupling launch took
  bool tc4_force = false;        // GBNF_TC4=2
  int tc3_pairs = 0;             // CTA pairs the device keeps resident at once (cudaOccupancyMaxActiveClusters)
  int profiling = 0;             // GBNF_PROF=1: cycle counters + event trace, 2: event trace only (gbnf_get_profile / _trace)
  int last_grid = 0;
  long long launches = 0;
  // peer-memory exchange (gbnf_comm_*): one allocation = CommBlock (4 KB) + 2 parity gather buffers [comm_rows x C] floats
  void* comm_mem = nullptr;
  void* comm_peer_mem[kMaxRanks] = {};
  long long comm_rows = 0;
  bool comm_ready = false;
  CommView cv{};
  float* cp_tmp = nullptr;       // component-parallel fallback: local log q block before the scatter kernel
  long long cp_tmp_cap = 0;
  // backward of the component under training (gbnf_component_backward)
  float* tr_w = nullptr;         // fp32 copies of its weights in both layouts + padded biases + 1024 zeros
  long long tr_w_floats = 0;
  float* tr_scratch = nullptr;   // per-step activations / d pre-activations [B][...]
  long long tr_rows = 0, tr_per_row = 0;
  int tr_njobs = 0;
  TrainStep* tr_steps_d = nullptr;
  TrainPackJob* tr_pack_d = nullptr;
  WgradJob* tr_jobs_d = nullptr;
  std::vector<TrainStep> tr_steps_h;
  std::vector<TrainPackJob> tr_pack_h;
  std::vector<WgradJob> tr_jobs_h;
};
constexpr size_t kCommBlockBytes = 4096;
static_assert(sizeof(CommBlock) <= kCommBlockBytes, "CommBlock does not fit its slot");

namespace {

const char* watchdog_text(int code) {
  switch (code) {
    case 10: return "TMA producer waiting for a free ring stage";
    case 11: return "TMA producer waiting for a free last-layer weight buffer";
    case 20: return "MMA issuer waiting for the A0 operand";
    case 21: return "MMA issuer waiting for a weight stage";
    case 22: return "MMA issuer waiting for an A1 quarter";
    case 23: return "MMA issuer waiting for a packed A2 piece";
    case 24: return "MMA issuer waiting for last-layer weights";
    case 25: return "MMA issuer waiting for a shipped-half slot to be read";
    case 26: return "MMA issuer waiting for a last-layer piece product to be read";
    case 27: return "MMA issuer waiting for the last-layer accumulator to be read";
    case 28: return "MMA issuer waiting for layer-1 chunk 2 to be read";
    case 30: return "epilogue waiting for a layer-1 accumulator";
    case 31: return "epilogue waiting for a layer-2 accumulator";
    case 32: return "epilogue waiting for the last-layer accumulator";
    case 40: return "waiting for a peer rank's value in the exchange block (a rank is missing or out of step)";
    default: return "in-kernel wait";
  }
}
// Status words the kernels leave in mapped host memory (readable without a synchronisation, and after a trap).  Called at the
// top of every entry point: an error raised by an EARLIER launch is reported by the first call that sees it.
int check_status(gbnf_ctx* h) {
  if (!h->flags_host) return GBNF_OK;
  volatile int* f = h->flags_host;
  if (f[0] != 0) {
    const int code = f[0];
    return fail(GBNF_ERR_CUDA, "kernel watchdog: a bounded wait timed out (code " + std::to_string(code) + ": " + watchdog_text(code) +
                                   "); the kernel trapped and the CUDA context is unusable");
  }
  if (f[2] != 0) {
    f[2] = 0;
    return fail(GBNF_ERR_NUMERIC, "an input or activation of an earlier launch was not finite in fp16 (|v| > 65504, inf or NaN): its "
                                  "results are invalid; standardise the data or use GBNF_GEMM_FP32");
  }
  return GBNF_OK;
}
int cuda_fail(gbnf_ctx* h, const char* what, cudaError_t e) {
  std::string msg = std::string(what) + ": " + cudaGetErrorString(e);
  if (h && h->flags_host && h->flags_host[0] != 0)
    msg += " [kernel watchdog code " + std::to_string(h->flags_host[0]) + ": " + watchdog_text(h->flags_host[0]) + "]";
  return fail(GBNF_ERR_CUDA, msg);
}
#define CUDA_TRY_H(h, expr)                                              \
  do {                                                                   \
    cudaError_t e_ = (expr);                                             \
    if (e_ != cudaSuccess) return cuda_fail((h), #expr, e_);             \
  } while (0)
#define ENTER(h)                                                         \
  DeviceGuard guard_((h)->cfg.device);                                   \
  do { int rc_ = check_status(h); if (rc_ != GBNF_OK) return rc_; } while (0)

int plan_layout(gbnf_ctx* h) {
  const gbnf_config& c = h->cfg;
  ModelDims& md = h->md;
  md.kind = c.kind; md.D = c.D; md.Dv = (c.D + 1) | 1;   // odd stride (bank-conflict free) with at least one scratch column at index D
  md.h = c.h; md.K = c.K; md.C = c.C; md.depth = c.depth;
  md.act = c.act; md.coupling = c.coupling; md.base = c.base;
  md.nlayers = (c.act == GBNF_ACT_RESIDUAL) ? 2 * c.depth + 2 : c.depth + 2;
  md.nnets = (c.kind == GBNF_KIND_REALNVP) ? 2 : 1;
  const bool f16 = (c.gemm_mode != GBNF_GEMM_FP32);
  const int kq = f16 ? 16 : kF32KT, nq = f16 ? 16 : kF32NT;
  const int h0 = c.D / 2, h1 = c.D - h0;
  // f16: the tensor-core kernels run the hidden width padded to a width they serve.  A padded hidden unit has zero weights
  // and a zero bias, so it computes act(0) = 0 exactly and meets zero weights in the next layer: the results are those of
  // the true width, bit for bit.  md.h = h_pad is the geometry every tensor-core plan and kernel reads; the hidden layers'
  // K_in / N_out keep the true width (the raw row stride and the zero-fill bound of the pack).
  int h_pad = c.h;
  if (f16 && c.h % 64 != 0 && c.h <= 512) h_pad = (c.depth == 1) ? round_up(c.h, kT2Chunk) : round_up(c.h, 64);
  else if (f16 && c.depth == 1 && c.h > 512 && c.h <= kT3H) h_pad = kT3H;
  md.h = h_pad;
  long long f = 0, i = 0, w = 0;   // running offsets (floats / ints / weight elements)
  h->steps_h.assign((size_t)c.C * c.K, StepDesc{});
  h->comps_h.assign((size_t)c.C, CompDesc{});
  h->out_max = 0;
  int kp0_max = 0, np_last_max = 0;
  for (int cc = 0; cc < c.C; ++cc) {
    for (int k = 0; k < c.K; ++k) {
      StepDesc& sd = h->steps_h[(size_t)cc * c.K + k];
      bool flipped = (c.kind == GBNF_KIND_REALNVP) && (((k + cc) % 2) > 0);
      sd.in_dim = flipped ? h1 : h0;
      sd.out_dim = flipped ? h0 : h1;
      sd.has_affine = 0;   // filled at pack time (device does not read this copy); see pack
      sd.vec_off = f; f += round_up_ll(3LL * md.Dv, 4);
      sd.idx_off = i; i += round_up_ll(sd.in_dim + sd.out_dim, 4);
      f = round_up_ll(f, 4);
      sd.ep_off = f; f += 16LL * kEpPad;
      sd.eidx_off = 0;
      sd.has_invconv = (c.kind == GBNF_KIND_GLOW && c.glow_invconv) ? 1 : 0;
      if (sd.has_invconv) {
        sd.ic_Kp = round_up(c.D, kF32KT); sd.ic_Np = round_up(c.D, kF32NT);
        sd.icw_off = w; w += (long long)sd.ic_Kp * sd.ic_Np;
        sd.icwinv_off = w; w += (long long)sd.ic_Kp * sd.ic_Np;
        sd.icb_off = f; f += round_up_ll(sd.ic_Np, 4);
        kp0_max = std::max(kp0_max, sd.ic_Kp); np_last_max = std::max(np_last_max, sd.ic_Np);   // the dense step goes through the activation buffers
      }
      h->out_max = std::max(h->out_max, sd.out_dim);
      int n_last = sd.out_dim;
      if (c.kind == GBNF_KIND_GLOW && c.coupling == GBNF_COUPLING_AFFINE) n_last = 2 * sd.out_dim;
      for (int net = 0; net < md.nnets; ++net) {
        for (int l = 0; l < md.nlayers; ++l) {
          LayerDesc& L = sd.layer[net][l];
          L.K_in = (l == 0) ? sd.in_dim : c.h;
          L.N_out = (l == md.nlayers - 1) ? n_last : c.h;
          L.Kp = (l == 0) ? round_up(L.K_in, kq) : f16 ? h_pad : round_up(c.h, kF32KT);
          L.Np = (l == md.nlayers - 1) ? round_up(L.N_out, nq) : f16 ? h_pad : round_up(c.h, nq);
          L.NC = L.Np; L.NC2 = 0;
          L.w_off = w; w += (long long)L.Kp * L.Np;
          L.b_off = f; f += round_up_ll(L.Np, 4);
          if (l == 0) kp0_max = std::max(kp0_max, L.Kp);
          if (l == md.nlayers - 1) np_last_max = std::max(np_last_max, L.Np);
        }
      }
    }
    CompDesc& cd = h->comps_h[cc];
    cd.sigma_off = i; i += round_up_ll(c.D, 4);
    cd.const_off = f; f += 4;
    cd.base_off = f; f += round_up_ll(2LL * md.Dv + 1, 4);
  }
  f = round_up_ll(f, 4);
  h->cc_off = f;
  for (int cc = 0; cc < c.C; ++cc) h->comps_h[cc].dense_off = f + 2LL * cc;
  f += round_up_ll(2LL * c.C, 4);
  h->f_count = f; h->i_count = i;
  h->w_bytes = w * (f16 ? (long long)sizeof(__half) : (long long)sizeof(float));
  if (!f16) {
    const int hp = round_up(c.h, kF32NT);
    h->rows_per_cta = (hp <= 256) ? 64 : (hp <= 512) ? 32 : 16;
    h->ld = std::max(hp, std::max(kp0_max, np_last_max)) + 4;
    size_t fl = (size_t)((h->rows_per_cta * md.Dv + 3) & ~3) + 2ull * h->rows_per_cta * h->ld + 2ull * kF32KT * kF32NT +
                (size_t)h->rows_per_cta * h->out_max + kMaxComponents + 3ull * h->rows_per_cta;
    h->smem_bytes = fl * sizeof(float);
    h->tmem_cols = 0;
    if (h->smem_bytes > 227 * 1024) return fail(GBNF_ERR_INVALID, "fp32 path: hidden width too large for shared memory");
  } else {
    h->kernel = tc2_eligible(md, h->steps_h) ? CouplingKernel::kPipelined
              : tc3_eligible(md, h->steps_h) ? CouplingKernel::kPair : CouplingKernel::kSerial;
    std::string why;
    if (h->kernel == CouplingKernel::kPair) {
      if (!tc3_make_plan(md, h->steps_h, &h->tc)) return fail(GBNF_ERR_INVALID, "f16 tensor-core path (h = 1024): shared memory budget exceeded");
    } else if (h->kernel == CouplingKernel::kPipelined) {
      if (!tc2_make_plan(md, h->steps_h, &h->tc)) return fail(GBNF_ERR_INVALID, "f16 tensor-core path: shared memory budget exceeded");
      for (StepDesc& sd : h->steps_h)
        for (int net = 0; net < md.nnets; ++net) {
          sd.layer[net][0].NC = kT2Chunk;
          sd.layer[net][1].NC = kT2Chunk; sd.layer[net][1].NC2 = (md.h == 512) ? kT2Piece : 0;
        }
      // the alternatives run on the same packed image (GBNF_TC4=0 keeps the single-chain kernel, GBNF_TC5=0 the serial-network
      // kernel: bitwise references for the tests, A/B measurements)
      const char* tc4_env = std::getenv("GBNF_TC4");
      const char* tc5_env = std::getenv("GBNF_TC5");
      if (tc4_eligible(md, h->steps_h) && !(tc4_env && tc4_env[0] == '0') && tc4_make_plan(md, h->steps_h, &h->alt_plan))
        h->alt = AltKernel::kTwoChain;
      else if (tc5_eligible(md, h->steps_h) && !(tc5_env && tc5_env[0] == '0') && tc5_make_plan(md, h->steps_h, &h->alt_plan))
        h->alt = AltKernel::kInterleaved;
      h->tc4_force = h->alt == AltKernel::kTwoChain && tc4_env && tc4_env[0] == '2';
    } else if (!tc_make_plan(md, h->steps_h, &h->tc, &why)) {
      return fail(GBNF_ERR_INVALID, "f16 tensor-core path: " + why);
    }
    h->tc.tanh_mode = (c.gemm_mode == GBNF_GEMM_F16_TC_FAST) ? 0 : 1;
    h->alt_plan.tanh_mode = h->tc.tanh_mode;
    { const char* pe = std::getenv("GBNF_PROF"); h->profiling = (pe && pe[0] >= '1' && pe[0] <= '2') ? pe[0] - '0' : 0; }
    h->rows_per_cta = 128;
    h->smem_bytes = h->tc.smem_bytes;
    h->tmem_cols = h->tc.tmem_cols;
  }
  return GBNF_OK;
}

int grid_for(const gbnf_ctx* h, long long n_items, int per_block) {
  long long need = (n_items + per_block - 1) / per_block;
  long long cap = (long long)h->num_sms * 8;
  return (int)std::max(1LL, std::min(need, cap));
}

int ensure_scan_workspace(gbnf_ctx* h, long long B) {
  if (B <= h->cum_cap) return GBNF_OK;
  if (h->cum) { cudaFree(h->cum); cudaFree(h->tile_sums); cudaFree(h->tile_offs); h->cum = nullptr; }
  long long cap = std::max(B, 1LL << 16);
  long long tiles = (cap + kScanTile - 1) / kScanTile;
  CUDA_TRY(cudaMalloc(&h->cum, cap * sizeof(double)));
  CUDA_TRY(cudaMalloc(&h->tile_sums, tiles * sizeof(double)));
  CUDA_TRY(cudaMalloc(&h->tile_offs, (tiles + 1) * sizeof(double)));
  h->cum_cap = cap;
  return GBNF_OK;
}

// Launch arguments that come from the handle (packed model, status words); the caller fills in rows, components and outputs.
CouplingArgs coupling_args(const gbnf_ctx* h) {
  CouplingArgs a{};
  a.steps = h->steps_d; a.comps = h->comps_d; a.fblob = h->fblob; a.iblob = h->iblob; a.wblob = h->wblob; a.md = h->md;
  a.cc_off = h->cc_off;
  a.error_flag = h->flags;
  return a;
}

int launch_coupling(gbnf_ctx* h, const float* x, long long B, int c0, int c1, float* logq, int ld_logq, float* z_out,
                    float* ldj_out, const float* rho, int n_mix, int skip_c, int mix_mode, float* G_ll, cudaStream_t st,
                    bool to_peers = false, int peer_ld = 0, int peer_col0 = 0, bool terms_only = false) {
  for (int c = c0; c < c1; ++c)
    if (!h->packed[c]) return fail(GBNF_ERR_STATE, "component " + std::to_string(c) + " has not been packed");
  if (B == 0) return GBNF_OK;
  // rows are independent: very large batches go through in slices, which bounds the per-launch scratch (mixture terms)
  // and keeps the tile count inside an int
  constexpr long long kMaxRowsPerLaunch = 1LL << 22;
  if (B > kMaxRowsPerLaunch) {
    for (long long r0 = 0; r0 < B; r0 += kMaxRowsPerLaunch) {
      const long long nb = std::min(kMaxRowsPerLaunch, B - r0);
      int rc = launch_coupling(h, x + r0 * h->md.D, nb, c0, c1, logq ? logq + r0 * ld_logq : nullptr, ld_logq,
                               z_out ? z_out + r0 * h->md.D : nullptr, ldj_out ? ldj_out + r0 : nullptr, rho, n_mix, skip_c,
                               mix_mode, G_ll ? G_ll + r0 : nullptr, st, false, 0, 0);
      if (rc != GBNF_OK) return rc;
    }
    return GBNF_OK;
  }
  // An ODD number (>= 3) of components on a shape the two-chain kernel serves: the even part goes through it (mixture terms only),
  // the last component through the single-chain kernel, whose last-unit reduce covers all n_mix terms (stream order makes the first
  // launch's terms visible).  5 - 16 % faster than the single-chain kernel on all of them (training: the fixed mixture has
  // 1 .. C - 1 components).
  if (h->alt == AltKernel::kTwoChain && h->profiling == 0 && !terms_only && z_out == nullptr && ldj_out == nullptr && !to_peers && (c1 - c0) >= 3 && ((c1 - c0) & 1)) {
    int rc = launch_coupling(h, x, B, c0, c1 - 1, logq, ld_logq, nullptr, nullptr, rho, n_mix, skip_c, mix_mode, G_ll, st, false, 0, 0, true);
    if (rc != GBNF_OK) return rc;
    return launch_coupling(h, x, B, c1 - 1, c1, logq ? logq + (c1 - 1 - c0) : nullptr, ld_logq, nullptr, nullptr, rho, n_mix, skip_c, mix_mode,
                           G_ll, st, false, 0, 0, false);
  }
  CouplingArgs a = coupling_args(h);
  a.terms_only = terms_only ? 1 : 0;
  a.x = x; a.B = B; a.c0 = c0; a.c1 = c1; a.logq = logq; a.ld_logq = ld_logq; a.z_out = z_out; a.ldj_out = ldj_out;
  a.rho = rho; a.n_mix = n_mix; a.skip_c = skip_c; a.mix_mode = mix_mode; a.G_ll = G_ll;
  if (to_peers) {
    a.n_peers = h->cv.world; a.peer_ld = peer_ld; a.peer_col0 = peer_col0;
    for (int q = 0; q < h->cv.world; ++q) a.logq_peers[q] = h->cv.gather[q] + (h->cv.epoch & 1u) * h->cv.gather_stride;
  }
  a.prof = h->prof;
  const int R = h->rows_per_cta;
  a.num_tiles = (int)((B + R - 1) / R);
  a.split = 1; a.comps_per_unit = c1 - c0; a.num_units = a.num_tiles;
  const bool pair = h->kernel == CouplingKernel::kPair;
  const int workers = pair ? h->tc3_pairs : h->num_sms;        // CTAs, or CTA pairs, that run concurrently
  AltKernel alt = (h->alt == AltKernel::kInterleaved && h->profiling == 0) ? AltKernel::kInterleaved : AltKernel::kNone;
  if (h->kernel == CouplingKernel::kPipelined || pair) {
    // split every tile's components over S units when that shortens the critical CTA (waves x components per unit)
    const int ncomp = c1 - c0;
    long long best = -1;
    // The two-chain kernel pairs the two halves of a unit's components: every unit needs the same, even number of them.  A pass
    // of it takes ~0.8 of a single-chain pass, which the cost model weighs against the coarser units (GBNF_TC4=2: always
    // prefer it when a split allows it -- tests).
    const bool tc4_ok = h->alt == AltKernel::kTwoChain && h->profiling != 2 && z_out == nullptr;
    bool best_two = false;
    for (int S = 1; S <= ncomp; S *= 2) {
      const int cpu = (ncomp + S - 1) / S;
      const int units = a.num_tiles * ((ncomp + cpu - 1) / cpu);
      const bool two = tc4_ok && cpu % 2 == 0 && ncomp % cpu == 0;
      long long cost = (long long)((units + workers - 1) / workers) * cpu * (two ? 4 : 5);
      if (h->tc4_force && !two) cost += 1LL << 40;
      if (best < 0 || cost < best) { best = cost; a.comps_per_unit = cpu; a.split = (ncomp + cpu - 1) / cpu; best_two = two; }
    }
    if (best_two) alt = AltKernel::kTwoChain;
    a.num_units = a.num_tiles * a.split;
    if (G_ll != nullptr) {
      const long long need = (long long)a.num_tiles * R * std::max(1, n_mix);
      if (need > h->lse_cap) {
        if (h->lse_part) cudaFree(h->lse_part);
        h->lse_part = nullptr; h->lse_cap = 0;
        CUDA_TRY(cudaMalloc(&h->lse_part, need * sizeof(float)));
        h->lse_cap = need;
      }
      if (a.num_tiles > h->ctr_cap) {
        if (h->tile_ctr) cudaFree(h->tile_ctr);
        h->tile_ctr = nullptr; h->ctr_cap = 0;
        const long long cap = std::max<long long>(a.num_tiles, 1024);
        CUDA_TRY(cudaMalloc(&h->tile_ctr, cap * sizeof(unsigned int)));
        CUDA_TRY(cudaMemsetAsync(h->tile_ctr, 0, cap * sizeof(unsigned int), st));
        h->ctr_cap = cap;
      }
      a.lse_terms = h->lse_part; a.tile_ctr = h->tile_ctr;
    }
  }
  int grid = std::min(a.num_units, workers);
  { const char* ge = std::getenv("GBNF_GRID"); if (ge && std::atoi(ge) > 0) grid = std::min(grid, std::atoi(ge)); }   // diagnostics: fewer CTAs
  h->last_grid = pair ? 2 * grid : grid;
  h->last_alt = alt;
  int rc = 0;
  if (alt == AltKernel::kTwoChain) rc = tc4_launch(a, h->alt_plan, grid, st, h->profiling);
  else if (alt == AltKernel::kInterleaved) rc = tc5_launch(a, h->alt_plan, grid, st);
  else if (h->kernel == CouplingKernel::kPipelined) rc = tc2_launch(a, h->tc, grid, st, h->profiling);
  else if (pair) rc = tc3_launch(a, h->tc, grid, st, h->profiling);
  else if (h->kernel == CouplingKernel::kSerial) rc = tc_launch(a, h->tc, grid, st);
  else if (R == 64) coupling_fp32_kernel<64><<<grid, kF32Threads, h->smem_bytes, st>>>(a, h->ld, h->out_max);
  else if (R == 32) coupling_fp32_kernel<32><<<grid, kF32Threads, h->smem_bytes, st>>>(a, h->ld, h->out_max);
  else coupling_fp32_kernel<16><<<grid, kF32Threads, h->smem_bytes, st>>>(a, h->ld, h->out_max);
  if (rc != 0) return fail(GBNF_ERR_INVALID, "f16 tensor-core path: launch configuration rejected");
  h->launches++;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

}  // namespace

extern "C" {

int gbnf_abi_version(void) { return GBNF_ABI_VERSION; }
const char* gbnf_last_error(void) { return g_last_error.c_str(); }

int gbnf_create(gbnf_handle* out, const gbnf_config* cfg) {
  if (!out || !cfg) return fail(GBNF_ERR_INVALID, "null argument");
  *out = nullptr;
  const gbnf_config& c = *cfg;
  if (c.kind != GBNF_KIND_REALNVP && c.kind != GBNF_KIND_GLOW) return fail(GBNF_ERR_INVALID, "unknown component kind");
  if (c.D < 2 || c.D >= kMaxD) return fail(GBNF_ERR_INVALID, "D must be in [2, 255]");
  if (c.h < 1 || c.K < 1 || c.C < 1 || c.C > kMaxComponents) return fail(GBNF_ERR_INVALID, "bad h / K / C");
  if (c.depth < 0 || c.depth + 2 > GBNF_MAX_LAYERS) return fail(GBNF_ERR_INVALID, "coupling_network_depth out of range");
  if (c.act < 0 || c.act > GBNF_ACT_RESIDUAL || c.coupling < 0 || c.coupling > 1 || c.base < 0 || c.base > 1)
    return fail(GBNF_ERR_INVALID, "bad act / coupling / base");
  if (c.act == GBNF_ACT_RESIDUAL) {
    if (c.kind != GBNF_KIND_REALNVP) return fail(GBNF_ERR_INVALID, "ResidualNet coupling networks are RealNVP only (upstream's Glow cannot build them: models/glow.py:294)");
    if (c.depth < 1 || 2 * c.depth + 2 > GBNF_MAX_LAYERS) return fail(GBNF_ERR_INVALID, "ResidualNet: coupling_network_depth (blocks) must be 1 or 2");
    if (c.gemm_mode != GBNF_GEMM_FP32) return fail(GBNF_ERR_INVALID, "ResidualNet coupling networks run in GBNF_GEMM_FP32 only");
  }
  if (c.act == GBNF_ACT_MIXED && c.kind != GBNF_KIND_REALNVP) return fail(GBNF_ERR_INVALID, "mixed nets are RealNVP only");
  if (c.gemm_mode < GBNF_GEMM_FP32 || c.gemm_mode > GBNF_GEMM_F16_TC_FAST) return fail(GBNF_ERR_INVALID, "bad gemm_mode");
  if (c.glow_invconv != 0 && c.glow_invconv != 1) return fail(GBNF_ERR_INVALID, "glow_invconv must be 0 or 1");
  if (c.glow_invconv && c.kind != GBNF_KIND_GLOW) return fail(GBNF_ERR_INVALID, "glow_invconv needs kind == GBNF_KIND_GLOW");
  if (c.glow_invconv && c.gemm_mode != GBNF_GEMM_FP32)
    return fail(GBNF_ERR_INVALID, "Glow steps with an invertible 1x1 convolution run in GBNF_GEMM_FP32 only");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(GBNF_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
  if (c.device < 0 || c.device >= ndev) return fail(GBNF_ERR_INVALID, "bad device ordinal");
  DeviceGuard guard_(c.device);
  cudaDeviceProp prop{};
  CUDA_TRY(cudaGetDeviceProperties(&prop, c.device));
  if (prop.major < 10) return fail(GBNF_ERR_CUDA, "device is not sm_100-class (kernels are built for sm_100a only)");

  gbnf_ctx* h = new (std::nothrow) gbnf_ctx();
  if (!h) return fail(GBNF_ERR_INVALID, "out of host memory");
  h->cfg = c;
  h->num_sms = prop.multiProcessorCount;
  int rc = plan_layout(h);
  if (rc != GBNF_OK) { delete h; return rc; }
  h->packed.assign((size_t)c.C, 0);
  h->inv_ok.assign((size_t)c.C, 1);
#define CREATE_TRY(expr)                                                                                 \
  do {                                                                                                   \
    cudaError_t e_ = (expr);                                                                             \
    if (e_ != cudaSuccess) { gbnf_destroy(h); return fail(GBNF_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); } \
  } while (0)
  CREATE_TRY(cudaMalloc(&h->steps_d, h->steps_h.size() * sizeof(StepDesc)));
  CREATE_TRY(cudaMalloc(&h->comps_d, h->comps_h.size() * sizeof(CompDesc)));
  CREATE_TRY(cudaMalloc(&h->fblob, std::max(1LL, h->f_count) * sizeof(float)));
  CREATE_TRY(cudaMalloc(&h->iblob, std::max(1LL, h->i_count) * sizeof(int)));
  CREATE_TRY(cudaMalloc(&h->wblob, std::max(16LL, h->w_bytes)));
  CREATE_TRY(cudaMemset(h->fblob, 0, std::max(1LL, h->f_count) * sizeof(float)));
  CREATE_TRY(cudaMalloc(&h->step_params_d, (size_t)c.K * sizeof(gbnf_step_params)));
  CREATE_TRY(cudaMalloc(&h->partial, (size_t)h->num_sms * 8 * 2 * sizeof(float)));
  CREATE_TRY(cudaMalloc(&h->ticket, 2 * sizeof(unsigned int)));
  CREATE_TRY(cudaMemset(h->ticket, 0, 2 * sizeof(unsigned int)));
  CREATE_TRY(cudaMalloc(&h->ms, 2 * sizeof(float)));
  CREATE_TRY(cudaMalloc(&h->wsum, sizeof(double)));
  CREATE_TRY(cudaHostAlloc((void**)&h->flags_host, 4 * sizeof(int), cudaHostAllocMapped));
  std::memset(h->flags_host, 0, 4 * sizeof(int));
  CREATE_TRY(cudaHostGetDevicePointer((void**)&h->flags, h->flags_host, 0));
  if (c.base == GBNF_BASE_DIAG_NORMAL) {
    CREATE_TRY(cudaMalloc(&h->base_mean, (size_t)c.D * sizeof(float)));
    CREATE_TRY(cudaMalloc(&h->base_scale, (size_t)c.D * sizeof(float)));
  }
  CREATE_TRY(cudaMalloc(&h->prof, 288 * sizeof(long long)));
  CREATE_TRY(cudaMemset(h->prof, 0, 288 * sizeof(long long)));
  CREATE_TRY(cudaMemcpy(h->comps_d, h->comps_h.data(), h->comps_h.size() * sizeof(CompDesc), cudaMemcpyHostToDevice));
  if (c.gemm_mode == GBNF_GEMM_FP32) {
    // the attribute is per FUNCTION, shared by all handles in the process: always raise it to the device maximum
    const int max_smem = 227 * 1024;
    CREATE_TRY(cudaFuncSetAttribute(coupling_fp32_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    CREATE_TRY(cudaFuncSetAttribute(coupling_fp32_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    CREATE_TRY(cudaFuncSetAttribute(coupling_fp32_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    CREATE_TRY(cudaFuncSetAttribute(coupling_fp32_inverse_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    CREATE_TRY(cudaFuncSetAttribute(coupling_fp32_inverse_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    CREATE_TRY(cudaFuncSetAttribute(coupling_fp32_inverse_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
  } else {
    CREATE_TRY(tc_configure(h->tc));
    CREATE_TRY(tc2_configure());
    CREATE_TRY(tc3_configure());
    CREATE_TRY(tc4_configure());
    CREATE_TRY(tc5_configure());
    if (h->kernel == CouplingKernel::kPair) h->tc3_pairs = tc3_max_pairs(h->tc, h->num_sms);
  }
#undef CREATE_TRY
  *out = h;
  return GBNF_OK;
}

void gbnf_destroy(gbnf_handle h) {
  if (!h) return;
  gbnf_comm_destroy(h);
  DeviceGuard guard_(h->cfg.device);
  cudaFree(h->base_mean); cudaFree(h->base_scale);
  if (h->flags_host) cudaFreeHost(h->flags_host);
  h->flags_host = nullptr; h->flags = nullptr;
  cudaFree(h->steps_d); cudaFree(h->comps_d); cudaFree(h->fblob); cudaFree(h->iblob); cudaFree(h->wblob);
  cudaFree(h->step_params_d); cudaFree(h->partial); cudaFree(h->ticket); cudaFree(h->ms); cudaFree(h->wsum);
  cudaFree(h->lse_part); cudaFree(h->tile_ctr);
  cudaFree(h->tr_w); cudaFree(h->tr_scratch); cudaFree(h->tr_steps_d); cudaFree(h->tr_pack_d); cudaFree(h->tr_jobs_d);
  cudaFree(h->cum); cudaFree(h->tile_sums); cudaFree(h->tile_offs); cudaFree(h->prof);
  delete h;
}

int gbnf_set_base(gbnf_handle h, const float* d_mean, const float* d_scale, void* stream) {
  if (!h) return fail(GBNF_ERR_INVALID, "null handle");
  if (h->cfg.base != GBNF_BASE_DIAG_NORMAL) return fail(GBNF_ERR_INVALID, "handle was not created with GBNF_BASE_DIAG_NORMAL");
  if (!d_mean || !d_scale) return fail(GBNF_ERR_INVALID, "null base pointers");
  ENTER(h);
  // copied (stream-ordered): the caller's tensors are only borrowed for the duration of the call
  CUDA_TRY_H(h, cudaMemcpyAsync(h->base_mean, d_mean, (size_t)h->cfg.D * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  CUDA_TRY_H(h, cudaMemcpyAsync(h->base_scale, d_scale, (size_t)h->cfg.D * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  h->base_set = true;
  std::fill(h->packed.begin(), h->packed.end(), 0);   // base constants live in each component's pack
  return GBNF_OK;
}

int gbnf_pack_component(gbnf_handle h, int32_t c, const gbnf_component_params* p, void* stream) {
  if (!h || !p || !p->steps) return fail(GBNF_ERR_INVALID, "null argument");
  if (c < 0 || c >= h->cfg.C) return fail(GBNF_ERR_INVALID, "component index out of range");
  if (p->n_steps != h->cfg.K) return fail(GBNF_ERR_INVALID, "n_steps != K");
  if (h->cfg.kind == GBNF_KIND_REALNVP && p->flip_init != c)
    return fail(GBNF_ERR_INVALID, "RealNVP component c must have flip_init == c (models/boosted_flow.py:46)");
  if (h->cfg.base == GBNF_BASE_DIAG_NORMAL && !h->base_set) return fail(GBNF_ERR_STATE, "call gbnf_set_base first");
  cudaStream_t st = (cudaStream_t)stream;
  ENTER(h);
  const ModelDims& md = h->md;
  const bool f16 = (h->cfg.gemm_mode != GBNF_GEMM_FP32);
  StepDesc* sd_h = &h->steps_h[(size_t)c * md.K];
  h->inv_ok[c] = 1;
  for (int k = 0; k < md.K; ++k) {
    const gbnf_step_params& sp = p->steps[k];
    if (h->cfg.kind == GBNF_KIND_GLOW) {
      if (!sp.an_bias || !sp.an_logs) return fail(GBNF_ERR_INVALID, "glow step needs an_bias / an_logs");
      if (h->cfg.glow_invconv) {
        if (!sp.invconv_w || !sp.invconv_logdet) return fail(GBNF_ERR_INVALID, "glow_invconv: the step needs invconv_w and invconv_logdet");
        if (!sp.invconv_winv) h->inv_ok[c] = 0;
      } else if (!sp.perm) {
        return fail(GBNF_ERR_INVALID, "glow step needs perm");
      }
      sd_h[k].has_affine = 1;
    } else {
      const int nbn = (sp.bn_log_gamma != nullptr) + (sp.bn_beta != nullptr) + (sp.bn_mean != nullptr) + (sp.bn_var != nullptr);
      if (nbn != 0 && nbn != 4) return fail(GBNF_ERR_INVALID, "BatchNorm pointers must be all set or all NULL");
      sd_h[k].has_affine = (nbn == 4);
    }
    for (int net = 0; net < md.nnets; ++net)
      for (int l = 0; l < md.nlayers; ++l)
        if (!sp.W[net][l] || !sp.b[net][l]) return fail(GBNF_ERR_INVALID, "missing Linear weight / bias pointer");
  }
  // stream-ordered pageable copies: the driver stages the host data before returning
  CUDA_TRY(cudaMemcpyAsync(h->steps_d + (size_t)c * md.K, sd_h, (size_t)md.K * sizeof(StepDesc), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(h->step_params_d, p->steps, (size_t)md.K * sizeof(gbnf_step_params), cudaMemcpyHostToDevice, st));
  PackMetaArgs ma{};
  ma.steps = h->step_params_d; ma.sdesc = h->steps_d + (size_t)c * md.K; ma.cdesc = h->comps_h[c]; ma.md = md;
  ma.flip_init = p->flip_init; ma.base_mean = h->base_mean; ma.base_scale = h->base_scale; ma.fblob = h->fblob; ma.iblob = h->iblob;
  ma.wblob_f32 = f16 ? nullptr : (float*)h->wblob;
  pack_meta_kernel<<<1, 32, 0, st>>>(ma);
  h->launches++;
  for (int k = 0; k < md.K; ++k) {
    const gbnf_step_params& sp = p->steps[k];
    for (int net = 0; net < md.nnets; ++net)
      for (int l = 0; l < md.nlayers; ++l) {
        const LayerDesc& L = sd_h[k].layer[net][l];
        const long long total = (long long)L.Kp * L.Np;
        const int grid = (int)std::min<long long>((total + 255) / 256, (long long)h->num_sms * 8);
        if (h->kernel == CouplingKernel::kPair)
          pack_weight_tc3_kernel<<<grid, 256, 0, st>>>(sp.W[net][l], sp.b[net][l], L, l, (__half*)h->wblob, h->fblob, h->flags + 1);
        else if (f16)
          pack_weight_f16_kernel<<<grid, 256, 0, st>>>(sp.W[net][l], sp.b[net][l], L, (__half*)h->wblob, h->fblob, h->flags + 1);
        else
          pack_weight_fp32_kernel<<<grid, 256, 0, st>>>(sp.W[net][l], sp.b[net][l], L, (float*)h->wblob, h->fblob);
        h->launches++;
      }
  }
  CUDA_TRY_H(h, cudaGetLastError());
  if (f16) {
    CUDA_TRY_H(h, cudaStreamSynchronize(st));          // documented in gbnf.h: the one entry point that synchronises
    if (h->flags_host[1]) {
      h->flags_host[1] = 0;
      return fail(GBNF_ERR_NUMERIC, "a weight is not finite in fp16; use GBNF_GEMM_FP32 for this model");
    }
  }
  h->packed[c] = 1;
  return GBNF_OK;
}

int gbnf_component_logq(gbnf_handle h, const float* d_x, int64_t B, int32_t c0, int32_t c1, float* d_logq,
                        float* d_z_opt, float* d_ldj_opt, void* stream) {
  if (!h) return fail(GBNF_ERR_INVALID, "null handle");
  if (B < 0 || c0 < 0 || c1 > h->cfg.C || c0 >= c1) return fail(GBNF_ERR_INVALID, "bad B or component range");
  if ((d_z_opt || d_ldj_opt) && c1 != c0 + 1) return fail(GBNF_ERR_INVALID, "z / ldj outputs need a single component");
  if (B == 0) return GBNF_OK;   // empty batch: nothing to do (pointers of empty tensors may be NULL)
  if (!d_x) return fail(GBNF_ERR_INVALID, "null x");
  if (!d_logq && !d_z_opt && !d_ldj_opt) return fail(GBNF_ERR_INVALID, "no output requested");
  ENTER(h);
  return launch_coupling(h, d_x, B, c0, c1, d_logq, c1 - c0, d_z_opt, d_ldj_opt, nullptr, 0, -1, 0, nullptr,
                         (cudaStream_t)stream);
}

int gbnf_component_inverse(gbnf_handle h, const float* d_z, int64_t B, int32_t c, float* d_x, float* d_ldj_opt, void* stream) {
  if (!h) return fail(GBNF_ERR_INVALID, "null handle");
  if (B < 0 || c < 0 || c >= h->cfg.C) return fail(GBNF_ERR_INVALID, "bad B or component index");
  if (B == 0) return GBNF_OK;
  if (!d_z || !d_x) return fail(GBNF_ERR_INVALID, "null pointer");
  if (!h->packed[c]) return fail(GBNF_ERR_STATE, "component " + std::to_string(c) + " has not been packed");
  if (h->cfg.glow_invconv && !h->inv_ok[c])
    return fail(GBNF_ERR_STATE, "inverse direction: component " + std::to_string(c) + " was packed without invconv_winv");
  const bool f16 = h->cfg.gemm_mode != GBNF_GEMM_FP32;
  if (f16 && h->kernel == CouplingKernel::kSerial)
    return fail(GBNF_ERR_INVALID, "inverse direction: the serial tensor-core kernel (hidden width 64, 192, 320 or 448, or depth > 1) "
                                  "does not serve it; use GBNF_GEMM_FP32 for this configuration");
  const bool pair = h->kernel == CouplingKernel::kPair;
  ENTER(h);
  cudaStream_t st = (cudaStream_t)stream;
  constexpr long long kMaxRowsPerLaunch = 1LL << 22;
  for (long long r0 = 0; r0 < B; r0 += kMaxRowsPerLaunch) {
    const long long nb = std::min(kMaxRowsPerLaunch, (long long)B - r0);
    CouplingArgs a = coupling_args(h);
    a.x = d_z + r0 * h->md.D; a.B = nb; a.c0 = c; a.c1 = c + 1; a.z_out = d_x + r0 * h->md.D; a.ldj_out = d_ldj_opt ? d_ldj_opt + r0 : nullptr;
    a.n_mix = 0; a.skip_c = -1;
    const int R = h->rows_per_cta;
    a.num_tiles = (int)((nb + R - 1) / R);
    a.split = 1; a.comps_per_unit = 1; a.num_units = a.num_tiles;
    const int grid = std::min(a.num_tiles, pair ? h->tc3_pairs : h->num_sms);     // CTAs, or CTA pairs
    h->last_grid = pair ? 2 * grid : grid;
    if (!f16) {
      if (R == 64) coupling_fp32_inverse_kernel<64><<<grid, kF32Threads, h->smem_bytes, st>>>(a, h->ld, h->out_max);
      else if (R == 32) coupling_fp32_inverse_kernel<32><<<grid, kF32Threads, h->smem_bytes, st>>>(a, h->ld, h->out_max);
      else coupling_fp32_inverse_kernel<16><<<grid, kF32Threads, h->smem_bytes, st>>>(a, h->ld, h->out_max);
    } else if (pair) {
      tc3_launch_inverse(a, h->tc, grid, st);
    } else {
      tc2_launch_inverse(a, h->tc, grid, st);
    }
    h->launches++;
    CUDA_TRY_H(h, cudaGetLastError());
  }
  return GBNF_OK;
}

int gbnf_mixture_logdensity(gbnf_handle h, const float* d_logq, int64_t B, int32_t ld, int32_t n_comp,
                            const float* d_rho, int32_t skip_c, int32_t mix_mode, float* d_G_ll, void* stream) {
  if (!h) return fail(GBNF_ERR_INVALID, "null handle");
  if (B < 0 || n_comp < 0 || n_comp > kMaxComponents || ld < n_comp) return fail(GBNF_ERR_INVALID, "bad B / n_comp / ld");
  if (skip_c == 0) return fail(GBNF_ERR_INVALID, "skip_c == 0 is not reachable in the reference (toy_experiment.py:409)");
  if (mix_mode < GBNF_MIX_SIMPLEX || mix_mode > GBNF_MIX_GEOMETRIC) return fail(GBNF_ERR_INVALID, "bad mix_mode");
  if (mix_mode == GBNF_MIX_GEOMETRIC && (skip_c >= 0 || n_comp == 0))
    return fail(GBNF_ERR_INVALID, "the geometric mixture (utils/density_plotting.py:199-226) takes >= 1 component and no skip_c");
  if (B == 0) return GBNF_OK;
  if (!d_G_ll || (n_comp > 0 && (!d_logq || !d_rho))) return fail(GBNF_ERR_INVALID, "null pointer");
  ENTER(h);
  if (n_comp == 0) {   // G_ll = zeros, density_experiment.py:612
    CUDA_TRY_H(h, cudaMemsetAsync(d_G_ll, 0, (size_t)B * sizeof(float), (cudaStream_t)stream));
    return GBNF_OK;
  }
  mixture_lse_kernel<<<grid_for(h, B, kMixThreads), kMixThreads, 0, (cudaStream_t)stream>>>(d_logq, B, ld, n_comp, d_rho,
                                                                                         skip_c, mix_mode, d_G_ll, CommView{}, h->flags);
  h->launches++;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

int gbnf_fused_eval(gbnf_handle h, const float* d_x, int64_t B, int32_t n_comp, const float* d_rho, int32_t skip_c,
                    int32_t mix_mode, float* d_G_ll, float* d_logq_opt, void* stream) {
  if (!h) return fail(GBNF_ERR_INVALID, "null handle");
  if (B < 0 || n_comp < 0 || n_comp > h->cfg.C) return fail(GBNF_ERR_INVALID, "bad B / n_comp");
  if (skip_c == 0) return fail(GBNF_ERR_INVALID, "skip_c == 0 is not reachable in the reference (toy_experiment.py:409)");
  if (mix_mode != GBNF_MIX_SIMPLEX && mix_mode != GBNF_MIX_RAW_RHO)
    return fail(GBNF_ERR_INVALID, "fused path: mix_mode must be GBNF_MIX_SIMPLEX or GBNF_MIX_RAW_RHO (the geometric mixture works "
                                  "on materialised log q: gbnf_component_logq + gbnf_mixture_logdensity)");
  if (B == 0) return GBNF_OK;
  if (!d_G_ll) return fail(GBNF_ERR_INVALID, "null G_ll");
  ENTER(h);
  if (n_comp == 0) {   // G_ll = zeros, density_experiment.py:612
    CUDA_TRY(cudaMemsetAsync(d_G_ll, 0, (size_t)B * sizeof(float), (cudaStream_t)stream));
    return GBNF_OK;
  }
  if (!d_x || !d_rho) return fail(GBNF_ERR_INVALID, "null pointer");
  return launch_coupling(h, d_x, B, 0, n_comp, d_logq_opt, n_comp, nullptr, nullptr, d_rho, n_comp, skip_c, mix_mode, d_G_ll,
                         (cudaStream_t)stream);
}

int gbnf_weight_stats(gbnf_handle h, const float* d_G_ll, int64_t B, float* d_ms, void* stream) {
  if (!h || !d_G_ll || !d_ms || B <= 0) return fail(GBNF_ERR_INVALID, "bad argument");
  ENTER(h);
  softmax_stats_kernel<<<grid_for(h, B, kMixThreads * 4), kMixThreads, 0, (cudaStream_t)stream>>>(d_G_ll, B, h->partial,
                                                                                              h->ticket, d_ms, CommView{});
  h->launches++;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

int gbnf_weight_apply(gbnf_handle h, const float* d_G_ll, int64_t B, const float* d_ms, float clamp_lo, float clamp_hi,
                      int32_t mode, float* d_w, double* d_wsum, void* stream) {
  (void)mode;
  if (!h || !d_G_ll || !d_ms || !d_w || !d_wsum || B <= 0) return fail(GBNF_ERR_INVALID, "bad argument");
  ENTER(h);
  cudaStream_t st = (cudaStream_t)stream;
  zero_double_kernel<<<1, 1, 0, st>>>(d_wsum);
  weight_apply_kernel<<<grid_for(h, B, kMixThreads * 4), kMixThreads, 0, st>>>(d_G_ll, B, d_ms, clamp_lo, clamp_hi, d_w,
                                                                             d_wsum, nullptr, CommView{}, h->ticket + 1, h->flags);
  h->launches += 2;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

int gbnf_weight_renorm(gbnf_handle h, float* d_w, int64_t B, const double* d_wsum, int32_t mode, void* stream) {
  if (!h || !d_w || !d_wsum || B <= 0) return fail(GBNF_ERR_INVALID, "bad argument");
  ENTER(h);
  weight_renorm_kernel<<<grid_for(h, B, kMixThreads * 4), kMixThreads, 0, (cudaStream_t)stream>>>(
      d_w, B, d_wsum, mode == GBNF_WEIGHTS_TOY ? 1 : 0, nullptr, CommView{}, h->flags);
  h->launches++;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

int gbnf_boost_weights(gbnf_handle h, const float* d_G_ll, int64_t B, float clamp_lo, float clamp_hi, int32_t mode,
                       float* d_w, float* d_stats, void* stream) {
  if (!h || !d_G_ll || !d_w || B <= 0) return fail(GBNF_ERR_INVALID, "bad argument");
  if (mode != GBNF_WEIGHTS_DENSITY && mode != GBNF_WEIGHTS_TOY) return fail(GBNF_ERR_INVALID, "bad weights mode");
  ENTER(h);
  cudaStream_t st = (cudaStream_t)stream;
  const int g = grid_for(h, B, kMixThreads * 4);
  softmax_stats_kernel<<<g, kMixThreads, 0, st>>>(d_G_ll, B, h->partial, h->ticket, h->ms, CommView{});
  zero_double_kernel<<<1, 1, 0, st>>>(h->wsum);
  weight_apply_kernel<<<g, kMixThreads, 0, st>>>(d_G_ll, B, h->ms, clamp_lo, clamp_hi, d_w, h->wsum, d_stats, CommView{}, h->ticket + 1, h->flags);
  weight_renorm_kernel<<<g, kMixThreads, 0, st>>>(d_w, B, h->wsum, mode == GBNF_WEIGHTS_TOY ? 1 : 0, d_stats, CommView{}, h->flags);
  h->launches += 4;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

// ---- training: gradients of the component that is being trained ------------------------------------------------------------------
int gbnf_component_backward(gbnf_handle h, int32_t c, const gbnf_component_params* p, const float* d_x, int64_t B, const float* d_dz,
                            const float* d_dldj, const gbnf_step_grads* grads, float* d_dx_opt, void* stream) {
  if (!h || !p || !p->steps || !grads || !d_x || !d_dz || !d_dldj) return fail(GBNF_ERR_INVALID, "null argument");
  if (c < 0 || c >= h->cfg.C || p->n_steps != h->cfg.K) return fail(GBNF_ERR_INVALID, "bad component index / n_steps");
  const gbnf_config& cf = h->cfg;
  const bool glow = cf.kind == GBNF_KIND_GLOW;
  if (cf.glow_invconv || cf.depth != 1 || cf.act == GBNF_ACT_RESIDUAL || (glow && cf.act == GBNF_ACT_MIXED) || cf.h > 512 || cf.D > 64)
    return fail(GBNF_ERR_INVALID, "fused backward: Glow (with a permutation) or RealNVP (without BatchNorm) components with "
                                  "coupling_network_depth 1, tanh / relu (RealNVP: or mixed) networks, h <= 512, D <= 64 (others train "
                                  "through the caller's autograd)");
  if (!glow && p->flip_init != c) return fail(GBNF_ERR_INVALID, "RealNVP component c must have flip_init == c (models/boosted_flow.py:46)");
  if (B <= 0) return fail(GBNF_ERR_INVALID, "empty batch");
  ENTER(h);
  cudaStream_t st = (cudaStream_t)stream;
  const int K = cf.K, D = cf.D, hD0 = D / 2, hD1 = D - hD0;
  const int nnets = glow ? 1 : 2;
  const int hp = round_up(cf.h, 64);
  // per-step geometry: RealNVP steps alternate |z1| / |z2| when D is odd (flipped iff (k + c) is odd, models/realnvp.py:37-43)
  struct Geo { int in_dim, out_dim, Kd[3], Nn[3], Kp[3], Np[3], NKp[3], KNp[3]; long long wfloats; };
  std::vector<Geo> geo(K);
  long long need_w = 1024;
  int ldz1 = 0;
  for (int k = 0; k < K; ++k) {
    Geo& g = geo[k];
    const bool flipped = !glow && (((k + c) % 2) > 0);
    g.in_dim = flipped ? hD1 : hD0; g.out_dim = flipped ? hD0 : hD1;
    const int n3 = glow ? ((cf.coupling == GBNF_COUPLING_AFFINE) ? 2 * g.out_dim : g.out_dim) : g.out_dim;
    const int Kd[3] = {g.in_dim, cf.h, cf.h}, Nn[3] = {cf.h, cf.h, n3};
    g.wfloats = 0;
    for (int l = 0; l < 3; ++l) {
      g.Kd[l] = Kd[l]; g.Nn[l] = Nn[l];
      g.Kp[l] = round_up(Kd[l], kF32KT); g.Np[l] = round_up(Nn[l], kF32NT);
      g.NKp[l] = round_up(Nn[l], kF32KT); g.KNp[l] = round_up(Kd[l], kF32NT);
      g.wfloats += (long long)g.Kp[l] * g.Np[l] + (long long)g.NKp[l] * g.KNp[l] + g.Np[l];
    }
    g.wfloats *= nnets;
    need_w += g.wfloats;
    ldz1 = std::max(ldz1, g.Kp[0]);
  }
  // every refusal comes before the first allocation, memset or copy: a refused call leaves the handle and `grads` untouched
  for (int k = 0; k < K; ++k) {
    const gbnf_step_params& sp = p->steps[k];
    const gbnf_step_grads& sg = grads[k];
    if (glow) {
      if (!sp.an_bias || !sp.an_logs || !sp.perm || !sg.an_bias || !sg.an_logs) return fail(GBNF_ERR_INVALID, "glow step needs ActNorm / perm / gradient pointers");
    } else if (sp.bn_log_gamma || sp.bn_beta || sp.bn_mean || sp.bn_var) {
      return fail(GBNF_ERR_INVALID, "fused backward: RealNVP steps with BatchNorm train through the caller's autograd (train-mode batch "
                                    "statistics couple the rows of a batch)");
    }
    for (int net = 0; net < nnets; ++net)
      for (int l = 0; l < 3; ++l)
        if (!sp.W[net][l] || !sp.b[net][l] || !sg.W[net][l] || !sg.b[net][l]) return fail(GBNF_ERR_INVALID, "missing Linear weight / bias / gradient pointer");
  }
  const int ld = std::max(hp, ldz1) + 4;
  const size_t smem = train_bwd_smem_bytes(K, D, nnets, ld);
  if (smem > kTrMaxSmem)
    return fail(GBNF_ERR_INVALID, "fused backward: the shared-memory history of K = " + std::to_string(K) + " steps at D = " + std::to_string(D) +
                                  ", h = " + std::to_string(cf.h) + " needs " + std::to_string(smem) + " bytes > " + std::to_string(kTrMaxSmem) +
                                  " (train through the caller's autograd)");
  if (need_w > h->tr_w_floats) {
    if (h->tr_w) cudaFree(h->tr_w);
    h->tr_w = nullptr; h->tr_w_floats = 0;
    CUDA_TRY_H(h, cudaMalloc(&h->tr_w, need_w * sizeof(float)));
    h->tr_w_floats = need_w;
  }
  const long long per_row = (long long)ldz1 + nnets * (4LL * hp + 64);
  if (B > h->tr_rows || per_row > h->tr_per_row) {
    if (h->tr_scratch) cudaFree(h->tr_scratch);
    h->tr_scratch = nullptr; h->tr_rows = 0;
    const long long rows = std::max<long long>(std::max<long long>(B, h->tr_rows), 1024);
    CUDA_TRY_H(h, cudaMalloc(&h->tr_scratch, (size_t)rows * per_row * K * sizeof(float)));
    h->tr_rows = rows; h->tr_per_row = per_row;
  }
  const int njobs = K * nnets * 3;
  if (!h->tr_steps_d || njobs > h->tr_njobs) {
    if (h->tr_steps_d) { cudaFree(h->tr_steps_d); cudaFree(h->tr_pack_d); cudaFree(h->tr_jobs_d); }
    CUDA_TRY_H(h, cudaMalloc(&h->tr_steps_d, (size_t)K * sizeof(TrainStep)));
    CUDA_TRY_H(h, cudaMalloc(&h->tr_pack_d, (size_t)njobs * sizeof(TrainPackJob)));
    CUDA_TRY_H(h, cudaMalloc(&h->tr_jobs_d, (size_t)njobs * sizeof(WgradJob)));
    h->tr_njobs = njobs;
  }
  h->tr_steps_h.assign(K, TrainStep{}); h->tr_pack_h.assign((size_t)njobs, TrainPackJob{}); h->tr_jobs_h.assign((size_t)njobs, WgradJob{});
  float* w = h->tr_w;
  float* zeros = h->tr_w + (need_w - 1024);
  int tile0 = 0, job = 0;
  for (int k = 0; k < K; ++k) {
    const gbnf_step_params& sp = p->steps[k];
    const gbnf_step_grads& sg = grads[k];
    const Geo& g = geo[k];
    TrainStep& ts = h->tr_steps_h[k];
    if (glow) {
      ts.an_bias = sp.an_bias; ts.an_logs = sp.an_logs; ts.perm = (const long long*)sp.perm;
      ts.g_bias = sg.an_bias; ts.g_logs = sg.an_logs;
    }
    ts.flipped = (!glow && (((k + c) % 2) > 0)) ? 1 : 0; ts.in_dim = g.in_dim; ts.out_dim = g.out_dim;
    float* sc = h->tr_scratch + (size_t)k * h->tr_rows * per_row;
    ts.z1 = sc; sc += h->tr_rows * ldz1;
    for (int l = 0; l < 3; ++l) { ts.Kp[l] = g.Kp[l]; ts.Np[l] = g.Np[l]; ts.NKp[l] = g.NKp[l]; ts.KNp[l] = g.KNp[l]; }
    // note: z1 rows are stored with stride Kp[0] of THIS step (<= ldz1)
    for (int net = 0; net < nnets; ++net) {
      ts.h1[net] = sc; sc += h->tr_rows * hp;
      ts.h2[net] = sc; sc += h->tr_rows * hp;
      ts.d1[net] = sc; sc += h->tr_rows * hp;
      ts.d2[net] = sc; sc += h->tr_rows * hp;
      ts.d3[net] = sc; sc += h->tr_rows * 64;
      for (int l = 0; l < 3; ++l) {
        TrainPackJob& pj = h->tr_pack_h[(size_t)job];
        pj.W = sp.W[net][l]; pj.b = sp.b[net][l]; pj.N = g.Nn[l]; pj.Kd = g.Kd[l]; pj.Kp = g.Kp[l]; pj.Np = g.Np[l]; pj.NKp = g.NKp[l]; pj.KNp = g.KNp[l];
        pj.Wt = w; w += (long long)g.Kp[l] * g.Np[l];
        pj.Wn = w; w += (long long)g.NKp[l] * g.KNp[l];
        pj.bp = w; w += g.Np[l];
        ts.Wt[net][l] = pj.Wt; ts.Wn[net][l] = pj.Wn; ts.b[net][l] = pj.bp;
        WgradJob& wj = h->tr_jobs_h[(size_t)job];
        wj.dact = (l == 0) ? ts.d1[net] : (l == 1) ? ts.d2[net] : ts.d3[net];  wj.ld_d = (l == 2) ? g.Np[2] : hp;
        wj.in = (l == 0) ? ts.z1 : (l == 1) ? ts.h1[net] : ts.h2[net];          wj.ld_i = (l == 0) ? g.Kp[0] : hp;
        wj.dW = sg.W[net][l]; wj.db = sg.b[net][l]; wj.N = g.Nn[l]; wj.Kd = g.Kd[l];
        wj.tiles_n = (g.Nn[l] + 63) / 64; wj.tiles_k = (g.Kd[l] + 63) / 64; wj.tile0 = tile0;
        tile0 += wj.tiles_n * wj.tiles_k;
        ++job;
      }
    }
    if (glow) {
      CUDA_TRY_H(h, cudaMemsetAsync(sg.an_bias, 0, (size_t)D * sizeof(float), st));
      CUDA_TRY_H(h, cudaMemsetAsync(sg.an_logs, 0, (size_t)D * sizeof(float), st));
    }
  }
  CUDA_TRY_H(h, cudaMemcpyAsync(h->tr_steps_d, h->tr_steps_h.data(), (size_t)K * sizeof(TrainStep), cudaMemcpyHostToDevice, st));
  CUDA_TRY_H(h, cudaMemcpyAsync(h->tr_pack_d, h->tr_pack_h.data(), (size_t)njobs * sizeof(TrainPackJob), cudaMemcpyHostToDevice, st));
  CUDA_TRY_H(h, cudaMemcpyAsync(h->tr_jobs_d, h->tr_jobs_h.data(), (size_t)njobs * sizeof(WgradJob), cudaMemcpyHostToDevice, st));
  CUDA_TRY_H(h, cudaMemsetAsync(zeros, 0, 1024 * sizeof(float), st));
  train_pack_kernel<<<dim3(32, njobs), 256, 0, st>>>(h->tr_pack_d);
  TrainArgs ta{};
  ta.x = d_x; ta.B = B; ta.dz = d_dz; ta.dldj = d_dldj; ta.steps = h->tr_steps_d; ta.K = K; ta.D = D; ta.h = cf.h; ta.hp = hp;
  ta.act = cf.act; ta.coupling = cf.coupling; ta.kind = cf.kind; ta.nnets = nnets; ta.ld = ld; ta.zeros = zeros; ta.dx = d_dx_opt;
  CUDA_TRY_H(h, cudaFuncSetAttribute(train_bwd_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTrMaxSmem));
  train_bwd_rows_kernel<<<(unsigned)((B + kTrR - 1) / kTrR), kF32Threads, smem, st>>>(ta);
  train_wgrad_kernel<<<tile0, 256, 0, st>>>(h->tr_jobs_d, njobs, B);
  h->launches += 3;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

// ---- multi-GPU: peer-memory exchange over NVLink (one process per GPU; handles exchanged by the caller's plumbing) ---------------
int gbnf_comm_local_handle(gbnf_handle h, int64_t max_rows, void* out_handle64) {
  if (!h || !out_handle64 || max_rows < 0) return fail(GBNF_ERR_INVALID, "bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  ENTER(h);
  if (h->comm_ready) return fail(GBNF_ERR_STATE, "the exchange is already initialised (gbnf_comm_destroy first)");
  if (h->comm_mem) { cudaFree(h->comm_mem); h->comm_mem = nullptr; }
  const long long rows = std::max<long long>(max_rows, 1);
  const size_t bytes = kCommBlockBytes + 2ull * (size_t)rows * h->cfg.C * sizeof(float);
  CUDA_TRY_H(h, cudaMalloc(&h->comm_mem, bytes));
  CUDA_TRY_H(h, cudaMemset(h->comm_mem, 0, bytes));
  CUDA_TRY_H(h, cudaDeviceSynchronize());
  h->comm_rows = rows;
  cudaIpcMemHandle_t ipc;
  CUDA_TRY_H(h, cudaIpcGetMemHandle(&ipc, h->comm_mem));
  std::memcpy(out_handle64, &ipc, 64);
  return GBNF_OK;
}

int gbnf_comm_init(gbnf_handle h, int32_t rank, int32_t world, const void* all_handles) {
  if (!h || !all_handles || world < 1 || world > kMaxRanks || rank < 0 || rank >= world) return fail(GBNF_ERR_INVALID, "bad rank / world (<= 8)");
  if (!h->comm_mem) return fail(GBNF_ERR_STATE, "call gbnf_comm_local_handle first");
  ENTER(h);
  CommView cv{};
  cv.rank = rank; cv.world = world; cv.epoch = 0;
  cv.gather_stride = h->comm_rows * h->cfg.C;
  for (int r = 0; r < world; ++r) {
    void* base = h->comm_mem;
    if (r != rank) {
      cudaIpcMemHandle_t ipc;
      std::memcpy(&ipc, (const char*)all_handles + 64 * r, 64);
      CUDA_TRY_H(h, cudaIpcOpenMemHandle(&base, ipc, cudaIpcMemLazyEnablePeerAccess));
      h->comm_peer_mem[r] = base;
    }
    cv.blk[r] = reinterpret_cast<CommBlock*>(base);
    cv.gather[r] = reinterpret_cast<float*>((char*)base + kCommBlockBytes);
  }
  h->cv = cv;
  h->comm_ready = true;
  return GBNF_OK;
}

int gbnf_comm_destroy(gbnf_handle h) {
  if (!h) return fail(GBNF_ERR_INVALID, "null handle");
  DeviceGuard guard_(h->cfg.device);
  for (int r = 0; r < kMaxRanks; ++r)
    if (h->comm_peer_mem[r]) { cudaIpcCloseMemHandle(h->comm_peer_mem[r]); h->comm_peer_mem[r] = nullptr; }
  if (h->comm_mem) { cudaFree(h->comm_mem); h->comm_mem = nullptr; }
  if (h->cp_tmp) { cudaFree(h->cp_tmp); h->cp_tmp = nullptr; h->cp_tmp_cap = 0; }
  h->comm_ready = false;
  h->cv = CommView{};
  return GBNF_OK;
}

int gbnf_boost_weights_dist(gbnf_handle h, const float* d_G_ll, int64_t B, float clamp_lo, float clamp_hi, int32_t mode,
                            float* d_w, float* d_stats, void* stream) {
  if (!h || !d_G_ll || !d_w || B <= 0) return fail(GBNF_ERR_INVALID, "bad argument (every rank needs at least one row)");
  if (mode != GBNF_WEIGHTS_DENSITY && mode != GBNF_WEIGHTS_TOY) return fail(GBNF_ERR_INVALID, "bad weights mode");
  if (!h->comm_ready) return fail(GBNF_ERR_STATE, "gbnf_comm_init has not been called");
  ENTER(h);
  cudaStream_t st = (cudaStream_t)stream;
  h->cv.epoch += 1;
  const int g = grid_for(h, B, kMixThreads * 4);
  softmax_stats_kernel<<<g, kMixThreads, 0, st>>>(d_G_ll, B, h->partial, h->ticket, h->ms, h->cv);
  zero_double_kernel<<<1, 1, 0, st>>>(h->wsum);
  weight_apply_kernel<<<g, kMixThreads, 0, st>>>(d_G_ll, B, h->ms, clamp_lo, clamp_hi, d_w, h->wsum, d_stats, h->cv, h->ticket + 1, h->flags);
  weight_renorm_kernel<<<g, kMixThreads, 0, st>>>(d_w, B, h->wsum, mode == GBNF_WEIGHTS_TOY ? 1 : 0, d_stats, h->cv, h->flags);
  h->launches += 4;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

int gbnf_mixture_component_parallel(gbnf_handle h, const float* d_x, int64_t B, int32_t n_comp, const float* d_rho, int32_t skip_c,
                                    int32_t mix_mode, float* d_G_ll, void* stream) {
  if (!h || !d_x || !d_rho || !d_G_ll || B <= 0) return fail(GBNF_ERR_INVALID, "bad argument");
  if (!h->comm_ready) return fail(GBNF_ERR_STATE, "gbnf_comm_init has not been called");
  const int world = h->cv.world, rank = h->cv.rank;
  if (n_comp < world || n_comp > h->cfg.C || n_comp % world != 0)
    return fail(GBNF_ERR_INVALID, "component-parallel evaluation needs n_comp to be a positive multiple of the world size");
  if (B > h->comm_rows) return fail(GBNF_ERR_INVALID, "batch larger than the gather buffer given to gbnf_comm_local_handle");
  if (skip_c == 0) return fail(GBNF_ERR_INVALID, "skip_c == 0 is not reachable in the reference (toy_experiment.py:409)");
  if (mix_mode != GBNF_MIX_SIMPLEX && mix_mode != GBNF_MIX_RAW_RHO) return fail(GBNF_ERR_INVALID, "bad mix_mode");
  ENTER(h);
  cudaStream_t st = (cudaStream_t)stream;
  h->cv.epoch += 1;
  const int per = n_comp / world, c0 = rank * per;
  const int ld = h->cfg.C;
  const long long tstride = h->comm_rows;                   // gather buffers are component-major: [C][comm_rows]
  if (h->kernel == CouplingKernel::kPipelined || h->kernel == CouplingKernel::kPair) {
    // fused: the coupling kernel's epilogue stores log q into every rank's gather buffer
    int rc = launch_coupling(h, d_x, B, c0, c0 + per, nullptr, per, nullptr, nullptr, nullptr, 0, -1, 0, nullptr, st, true, (int)tstride, c0);
    if (rc != GBNF_OK) return rc;
  } else {
    const long long need = (long long)B * per;
    if (need > h->cp_tmp_cap) {
      if (h->cp_tmp) cudaFree(h->cp_tmp);
      h->cp_tmp = nullptr; h->cp_tmp_cap = 0;
      CUDA_TRY_H(h, cudaMalloc(&h->cp_tmp, need * sizeof(float)));
      h->cp_tmp_cap = need;
    }
    int rc = launch_coupling(h, d_x, B, c0, c0 + per, h->cp_tmp, per, nullptr, nullptr, nullptr, 0, -1, 0, nullptr, st);
    if (rc != GBNF_OK) return rc;
    comm_scatter_logq_kernel<<<grid_for(h, need, kMixThreads), kMixThreads, 0, st>>>(h->cp_tmp, B, per, h->cv, tstride, c0);
    h->launches++;
  }
  const float* mine = h->cv.gather[rank] + (h->cv.epoch & 1u) * h->cv.gather_stride;
  mixture_lse_kernel<<<grid_for(h, B, kMixThreads), kMixThreads, 0, st>>>(mine, B, ld, n_comp, d_rho, skip_c, mix_mode, d_G_ll, h->cv, h->flags, tstride);
  h->launches++;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

int gbnf_resample(gbnf_handle h, const float* d_w, int64_t B, const double* d_u, int64_t n, int64_t* d_idx, void* stream) {
  if (!h || !d_w || B <= 0 || n < 0) return fail(GBNF_ERR_INVALID, "bad argument");
  if (n == 0) return GBNF_OK;
  if (!d_u || !d_idx) return fail(GBNF_ERR_INVALID, "null pointer");
  ENTER(h);
  int rc = ensure_scan_workspace(h, B);
  if (rc != GBNF_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int tiles = (int)((B + kScanTile - 1) / kScanTile);
  scan_tile_sums_kernel<<<tiles, kScanThreads, 0, st>>>(d_w, B, h->tile_sums);
  scan_tile_offsets_kernel<<<1, kScanThreads, 0, st>>>(h->tile_sums, tiles, h->tile_offs);
  scan_finalize_kernel<<<tiles, kScanThreads, 0, st>>>(d_w, B, h->tile_offs, tiles, h->cum);
  resample_search_kernel<<<grid_for(h, n, kMixThreads), kMixThreads, 0, st>>>(h->cum, B, d_u, n, (long long*)d_idx);
  h->launches += 4;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

int gbnf_gather_rows(gbnf_handle h, const float* d_x, int32_t D, const int64_t* d_idx, int64_t n, float* d_out, void* stream) {
  if (!h || D <= 0 || n < 0) return fail(GBNF_ERR_INVALID, "bad argument");
  if (n == 0) return GBNF_OK;
  if (!d_x || !d_idx || !d_out) return fail(GBNF_ERR_INVALID, "null pointer");
  ENTER(h);
  gather_rows_kernel<<<grid_for(h, n * 32, kMixThreads), kMixThreads, 0, (cudaStream_t)stream>>>(
      d_x, D, (const long long*)d_idx, n, d_out);
  h->launches++;
  CUDA_TRY_H(h, cudaGetLastError());
  return GBNF_OK;
}

int gbnf_actnorm_init(const float* d_x, int64_t B, int32_t D, float scale, float* d_bias, float* d_logs, void* stream) {
  if (B <= 0 || D <= 0 || D > kAnThreads || !(scale > 0.f)) return fail(GBNF_ERR_INVALID, "actnorm init: need B >= 1, 1 <= D <= 256, scale > 0");
  if (!d_x || !d_bias || !d_logs) return fail(GBNF_ERR_INVALID, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0, sms = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  int Dp = 1;
  while (Dp < D) Dp <<= 1;
  const int rpb = kAnThreads / Dp;
  const int grid = (int)std::max<long long>(1, std::min<long long>((B + rpb - 1) / rpb, (long long)sms * 8));
  double* acc = nullptr;
  CUDA_TRY(cudaMallocAsync((void**)&acc, 2 * (size_t)D * sizeof(double), st));
  CUDA_TRY(cudaMemsetAsync(acc, 0, 2 * (size_t)D * sizeof(double), st));
  actnorm_colsum_kernel<false><<<grid, kAnThreads, 0, st>>>(d_x, B, D, Dp, nullptr, acc);
  actnorm_bias_kernel<<<(D + 63) / 64, 64, 0, st>>>(acc, B, D, d_bias);
  actnorm_colsum_kernel<true><<<grid, kAnThreads, 0, st>>>(d_x, B, D, Dp, d_bias, acc + D);
  actnorm_logs_kernel<<<(D + 63) / 64, 64, 0, st>>>(acc + D, B, D, scale, d_logs);
  cudaError_t e = cudaGetLastError();
  cudaFreeAsync(acc, st);
  if (e != cudaSuccess) return fail(GBNF_ERR_CUDA, cudaGetErrorString(e));
  return GBNF_OK;
}

int gbnf_sample_component(const float* rho_host, int32_t n, double u, int32_t exclude, int32_t* j_out) {
  if (!rho_host || !j_out || n <= 0 || exclude >= n) return fail(GBNF_ERR_INVALID, "bad argument");
  double total = 0.0;
  for (int i = 0; i < n; ++i) if (i != exclude) total += (double)rho_host[i];
  if (!(total > 0.0)) return fail(GBNF_ERR_INVALID, "rho has no mass");
  double run = 0.0;
  int j = 0;
  for (int i = 0; i < n; ++i) {
    run += (i == exclude) ? 0.0 : (double)rho_host[i];
    if (run / total < u) j = i + 1; else break;
  }
  *j_out = std::min(j, n - 1);
  return GBNF_OK;
}

int gbnf_check_status(gbnf_handle h, void* stream) {
  if (!h) return fail(GBNF_ERR_INVALID, "null handle");
  DeviceGuard guard_(h->cfg.device);
  cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(h, "cudaStreamSynchronize", e);
  return check_status(h);
}

int gbnf_get_profile(gbnf_handle h, int64_t* out32) {
  if (!h || !out32) return fail(GBNF_ERR_INVALID, "null argument");
  ENTER(h);
  CUDA_TRY(cudaMemcpy(out32, h->prof, 32 * sizeof(long long), cudaMemcpyDeviceToHost));
  return GBNF_OK;
}

int gbnf_get_trace(gbnf_handle h, int64_t* out256) {
  if (!h || !out256) return fail(GBNF_ERR_INVALID, "null argument");
  ENTER(h);
  CUDA_TRY(cudaMemcpy(out256, h->prof + 32, 256 * sizeof(long long), cudaMemcpyDeviceToHost));
  return GBNF_OK;
}

int gbnf_get_info(gbnf_handle h, gbnf_info* out) {
  if (!h || !out) return fail(GBNF_ERR_INVALID, "null argument");
  out->gemm_mode = h->cfg.gemm_mode;
  out->rows_per_cta = h->rows_per_cta;
  out->smem_bytes = (int32_t)h->smem_bytes;
  out->tmem_cols = h->tmem_cols;
  out->num_sms = h->num_sms;
  out->grid = h->last_grid;
  out->packed_bytes = h->w_bytes + h->f_count * 4 + h->i_count * 4;
  out->launches = h->launches;
  out->pipelined = h->kernel == CouplingKernel::kPair ? 2 : h->kernel == CouplingKernel::kPipelined ? 1 : 0;
  out->two_chain = (int32_t)h->last_alt;
  return GBNF_OK;
}

}  // extern "C"
