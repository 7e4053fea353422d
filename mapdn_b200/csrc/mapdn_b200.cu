// C-ABI of the batched MAPDN voltage-control env (include/mapdn_b200.h): handle management,
// one-off Ybus assembly + symbolic analysis of the radial network, kernel launches.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/mapdn_b200.h"
#include "env_kernel.cuh"

// kernel<<<grid, block, smem, stream>>>(args...); under MAPDN_HOST_EMU (tests/emu: the library compiled with g++ for the
// CPU SIMT emulation, test infrastructure) the same launch runs on OS threads
#ifdef MAPDN_HOST_EMU
#define MAPDN_LAUNCH(kernel, grid, block, smem, stream, ...) emu::launch(kernel, grid, block, smem, stream, __VA_ARGS__)
#else
#define MAPDN_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<grid, block, smem, stream>>>(__VA_ARGS__)
#endif

namespace mapdn {

static thread_local std::string g_last_error;

static mapdn_status fail(mapdn_status st, const std::string& msg) {
  g_last_error = msg;
  return st;
}

#define MAPDN_CUDA(expr)                                                                        \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return fail(MAPDN_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
  } while (0)

// Every entry point runs on the handle's device and leaves the calling thread's current device as it found it
// (the caller -- PyTorch, CuPy -- tracks the current device through the CUDA runtime).
struct DeviceGuard {
  int prev = -1, dev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) : dev(device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
  }
  ~DeviceGuard() { if (prev >= 0 && prev != dev) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define MAPDN_ON_DEVICE(device)          \
  DeviceGuard _device_guard(device);     \
  MAPDN_CUDA(_device_guard.err)

// ------------------------------------------------------------------------------------------------
// Ybus assembly on the device (PYPOWER makeYbus, SURVEY Appendix A.3). Runs once per handle: the
// topology never changes between env steps (the reference rebuilds Ybus inside every pp.runpp).
// ------------------------------------------------------------------------------------------------
__global__ void ybus_branch_kernel(int n_br, const double* __restrict__ r, const double* __restrict__ x,
                                   const double* __restrict__ b, const double* __restrict__ g,
                                   const double* __restrict__ tap, const double* __restrict__ shift_deg,
                                   const unsigned char* __restrict__ status, double* __restrict__ ybr /*[n_br,8]*/) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_br) return;
  const double st = status[k] ? 1.0 : 0.0;
  const double den = r[k] * r[k] + x[k] * x[k];
  // Ys = stat / (r + jx); an out-of-service branch contributes exactly zero (also when r = x = 0)
  const double ys_g = status[k] ? r[k] / den : 0.0, ys_b = status[k] ? -x[k] / den : 0.0;
  const double ytt_g = ys_g + 0.5 * st * g[k], ytt_b = ys_b + 0.5 * st * b[k];   // Ys + j*Bc/2, Bc = b - jg
  const double t = (tap[k] == 0.0) ? 1.0 : tap[k];
  double sn, cs;
  sincos(shift_deg[k] * (3.14159265358979323846 / 180.0), &sn, &cs);
  const double tr = t * cs, ti = t * sn;                                  // tau = tap * exp(j*shift)
  const double t2 = tr * tr + ti * ti;
  // Yff = Ytt / (tau conj(tau)); Yft = -Ys / conj(tau); Ytf = -Ys / tau
  double* o = ybr + 8 * k;
  o[0] = ytt_g / t2; o[1] = ytt_b / t2;
  // -Ys/conj(tau) = -Ys * tau / |tau|^2
  o[2] = -(ys_g * tr - ys_b * ti) / t2; o[3] = -(ys_g * ti + ys_b * tr) / t2;
  // -Ys/tau = -Ys * conj(tau) / |tau|^2
  o[4] = -(ys_g * tr + ys_b * ti) / t2; o[5] = -(-ys_g * ti + ys_b * tr) / t2;
  o[6] = ytt_g; o[7] = ytt_b;
}

__global__ void ybus_diag_kernel(int n_bus, int n_br, const int* __restrict__ from, const int* __restrict__ to,
                                 const double* __restrict__ ybr, const double* __restrict__ gs,
                                 const double* __restrict__ bs, double inv_base, double* __restrict__ ydiag /*[n_bus,2]*/) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_bus) return;
  double g = gs[i] * inv_base, b = bs[i] * inv_base;                      // Ysh = (GS + jBS)/baseMVA
  for (int k = 0; k < n_br; ++k) {
    if (from[k] == i) { g += ybr[8 * k + 0]; b += ybr[8 * k + 1]; }
    if (to[k] == i) { g += ybr[8 * k + 6]; b += ybr[8 * k + 7]; }
  }
  ydiag[2 * i] = g; ydiag[2 * i + 1] = b;
}

// ---- small gather kernels over the env state kept in HBM ----
__global__ void scale_copy_kernel(long long n, const double* __restrict__ in, double scale, double* __restrict__ out) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = in[i] * scale;
}
__global__ void int_to_double_kernel(long long n, const int* __restrict__ in, double* __restrict__ out) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = static_cast<double>(in[i]);
}
__global__ void i64_to_double_kernel(long long n, const long long* __restrict__ in, double* __restrict__ out) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = static_cast<double>(in[i]);
}

// get_obs() from the state in HBM (reference :232-316), driven by the precomputed obs program
__global__ void get_obs_kernel(const __grid_constant__ Params p) {
  const int tot = p.n_sgen * p.obs_dim;
  const long long gid = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (gid >= static_cast<long long>(p.nb) * tot) return;
  const int env = static_cast<int>(gid / tot), idx = static_cast<int>(gid - static_cast<long long>(env) * tot);
  const size_t eN = static_cast<size_t>(env) * p.n_bus, eG = static_cast<size_t>(env) * p.n_sgen;
  const unsigned src = __ldg(p.obs_src + idx);   // cold copy of the obs program (kind | node)
  const int kind = static_cast<int>(src >> 28), ix = static_cast<int>(src & 0x0FFFFFFFu);
  // node id -> bus id (npq = slack)
  auto bus = [&](int i) { return (i == p.npq) ? p.slack_bus : __ldg(p.bus_of_node + i); };
  double v = 0.0;
  if (kind == OBS_P || kind == OBS_Q) {
    v = (kind == OBS_P) ? p.res_p[eN + bus(ix)] : p.res_q[eN + bus(ix)];
    for (int t = __ldg(p.obs_xptr + idx), te = __ldg(p.obs_xptr + idx + 1); t < te; ++t) {
      const int sg = __ldg(p.obs_xidx + t);
      v += (kind == OBS_P) ? p.cur_pv[eG + sg] : p.cur_q[eG + sg];
    }
  } else if (kind == OBS_PV) v = p.cur_pv[eG + ix];
  else if (kind == OBS_QSG) v = p.cur_q[eG + ix];
  else if (kind == OBS_VM) v = p.res_vm[eN + bus(ix)];
  else if (kind == OBS_VA) v = p.res_va[eN + bus(ix)];
  p.obs[gid] = v;
}

// get_state() (reference :213-230): [P_bus | Q_bus | pv | q | vm | va(deg)] restricted to state_space
__global__ void get_state_kernel(const __grid_constant__ Params p) {
  const long long gid = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (gid >= static_cast<long long>(p.nb) * p.state_dim) return;
  const int env = static_cast<int>(gid / p.state_dim), idx = static_cast<int>(gid - static_cast<long long>(env) * p.state_dim);
  const size_t eN = static_cast<size_t>(env) * p.n_bus, eG = static_cast<size_t>(env) * p.n_sgen;
  const unsigned src = __ldg(p.state_src + idx);
  const int kind = static_cast<int>(src >> 28), ix = static_cast<int>(src & 0x0FFFFFFFu);
  double v = 0.0;
  if (kind == OBS_PBUS) v = p.res_p[eN + ix];
  else if (kind == OBS_QBUS) v = p.res_q[eN + ix];
  else if (kind == OBS_PV) v = p.cur_pv[eG + ix];
  else if (kind == OBS_QSG) v = p.cur_q[eG + ix];
  else if (kind == OBS_VM) v = p.res_vm[eN + ix];
  else if (kind == OBS_VA_DEG) v = p.res_va[eN + ix] * 57.295779513082320876798;
  p.state[gid] = v;
}

}  // namespace mapdn

using namespace mapdn;

// ------------------------------------------------------------------------------------------------
struct mapdn_env {
  int device = 0;
  mapdn_cfg cfg{};
  mapdn_dims dims{};
  Params base{};                       // static + state pointers; io fields filled per call
  std::vector<void*> allocs;           // everything cudaMalloc'ed
  int G = 8, threads = 128, epb = 16, smem = 0, max_blocks = 0, helper_threads = 32;
  bool dense = false;                  // meshed net: dense-LU fallback solver
  long long launches = 0;
  // Ybus pieces kept for the test hook
  std::vector<double> ybr, ydiag;
  std::vector<int> br_from, br_to;
  // device-side staging buffers of the *_host entry points
  double *d_stage_actions = nullptr, *d_stage_reward = nullptr, *d_stage_info = nullptr, *d_stage_obs = nullptr;
  unsigned char* d_stage_term = nullptr;
  int obs_zero_off = 0;                // slab offset of the constant-zero slot the obs padding reads
  std::vector<int> agent_len, agent_off;   // compact observation rows: true length / offset of every agent's block
  int compact_row = 0;                 // entries per compact row (sum of agent_len, rounded up to a multiple of 4)
  std::vector<const void*> pinned_ok;  // host buffers already verified as pinned (mapdn_step_host_pinned)
};

namespace {

template <class T>
mapdn_status dev_upload(mapdn_env* e, const std::vector<T>& v, const T** out) {
  void* d = nullptr;
  const size_t bytes = std::max<size_t>(v.size() * sizeof(T), 16);
  MAPDN_CUDA(cudaMalloc(&d, bytes));
  e->allocs.push_back(d);
  if (!v.empty()) MAPDN_CUDA(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = static_cast<const T*>(d);
  return MAPDN_OK;
}

template <class T>
mapdn_status dev_alloc(mapdn_env* e, size_t count, T** out) {
  void* d = nullptr;
  const size_t bytes = std::max<size_t>(count * sizeof(T), 16);
  MAPDN_CUDA(cudaMalloc(&d, bytes));
  MAPDN_CUDA(cudaMemset(d, 0, bytes));
  e->allocs.push_back(d);
  *out = static_cast<T*>(d);
  return MAPDN_OK;
}

template <class T>
std::vector<T> vec_or(const T* p, size_t n, T fill) {
  return p ? std::vector<T>(p, p + n) : std::vector<T>(n, fill);
}

using KernelFn = void (*)(const Params);
constexpr int kHelperPairsPerWarp = 256;   // Box-Muller pairs of a CTA round per helper warp (1024 measured slower: +2 us on case33)

template <int G>
KernelFn kernel_for_mode(int mode) {
  switch (mode) {
    case MODE_SOLVE: return env_kernel<G, MODE_SOLVE>;
    case MODE_STEP: return env_kernel<G, MODE_STEP>;
    case MODE_DROOP: return env_kernel<G, MODE_DROOP>;
    default: return env_kernel<G, MODE_RESET>;
  }
}

KernelFn kernel_for(int G, int mode, bool dense = false) {
  if (dense) {
    switch (mode) {
      case MODE_SOLVE: return env_kernel<32, MODE_SOLVE, true>;
      case MODE_STEP: return env_kernel<32, MODE_STEP, true>;
      case MODE_DROOP: return env_kernel<32, MODE_DROOP, true>;
      default: return env_kernel<32, MODE_RESET, true>;
    }
  }
  switch (G) {
    case 4: return kernel_for_mode<4>(mode);
    case 8: return kernel_for_mode<8>(mode);
    case 16: return kernel_for_mode<16>(mode);
    case 64: return kernel_for_mode<64>(mode);
    case 128: return kernel_for_mode<128>(mode);
    default: return kernel_for_mode<32>(mode);
  }
}

// smem per env in double2 units: (npq + 1) node records of 9 double2, sgen p/q, scratch of ng + 2 nl
// doubles. For G = 4 two envs share a quarter-warp of a 128-bit access, so their slabs must start
// 64 B apart modulo 128 B.
// The prologue stages 2 n_load scaled load values per env. They fit the Newton fields of the node records (12 dead
// doubles per record, see env_kernel.cuh) unless the net has very many loads per bus.
bool stage_fits_records(int npq, int nl) { return 2 * nl <= 12 * (npq + 2); }

// scratch doubles per env: next pv row / droop voltages [n_sgen], the partial sums per warp of the multi-warp group
// reductions, and the staged loads when they do not fit the records
int scratch_doubles_for(int ng, int nl, int G, bool stage_rec) {
  return ng + (G > 32 ? 10 * (G / 32) : 0) + (stage_rec ? 0 : 2 * nl);
}

int env_stride2_for(int npq, int ng, int nl, int G, bool stage_rec) {
  int stride = kNodeArrays2 * (npq + 2) + ng + (scratch_doubles_for(ng, nl, G, stage_rec) + 1) / 2;
  if (G == 4) while ((stride * 16) % 128 != 64) ++stride;
  return stride;
}

mapdn_status launch_env_kernel(mapdn_env* e, int mode, Params& p, cudaStream_t st) {
  KernelFn fn = kernel_for(e->G, mode, e->dense);
  const int needed = (p.nb + e->epb - 1) / e->epb;
  int grid = std::min(needed, std::max(1, e->max_blocks));
  const int rounds = (needed + grid - 1) / grid;
  grid = (needed + rounds - 1) / rounds;       // balance the persistent loop
#ifdef MAPDN_PROFILE
  static long long* d_prof = nullptr;
  if (!d_prof) cudaMalloc(&d_prof, 16 * sizeof(long long));
  cudaMemset(d_prof, 0, 16 * sizeof(long long));
  p.prof = d_prof;
#endif
  p.helper_threads = e->helper_threads;
  MAPDN_LAUNCH(fn, grid, e->threads + (mode == MODE_STEP ? e->helper_threads : 0), e->smem, st, p);   // MODE_STEP: + helper warps
  MAPDN_CUDA(cudaGetLastError());
  e->launches++;
#ifdef MAPDN_PROFILE
  {
    long long hp[16];
    cudaDeviceSynchronize();
    cudaMemcpy(hp, d_prof, sizeof(hp), cudaMemcpyDeviceToHost);
    static const char* nm[12] = {"-", "setup+prologue", "init/update", "edges", "F/diag", "elim", "backsub", "reload+slack",
                                 "q+nextrow", "BP/OP+bus+lines", "reward/info", "obs/state"};
    long long tot = 0;
    for (int k = 0; k < 12; ++k) tot += hp[k];
    fprintf(stderr, "[prof mode=%d nb=%d] total %lld cyc:", mode, p.nb, tot);
    for (int k = 1; k < 12; ++k) fprintf(stderr, " %s=%lld", nm[k], hp[k]);
    if (hp[14] > 0)
      fprintf(stderr, " | forward-sweep step: %lld executions in %lld solves, load wait %lld + arithmetic %lld cyc per step",
              hp[14], hp[15], hp[12] / hp[14], hp[13] / hp[14]);
    fprintf(stderr, "\n");
  }
#endif
  return MAPDN_OK;
}

}  // namespace

extern "C" {

int32_t mapdn_abi_version(void) { return MAPDN_ABI_VERSION; }
const char* mapdn_last_error(void) { return g_last_error.c_str(); }

mapdn_status mapdn_destroy(mapdn_env* e) {
  if (!e) return MAPDN_OK;
  DeviceGuard guard(e->device);
  for (void* d : e->allocs) cudaFree(d);
  delete e;
  return MAPDN_OK;
}

mapdn_status mapdn_create(const mapdn_net_desc* net, const mapdn_profile_desc* prof, const mapdn_cfg* cfg,
                          int32_t device, mapdn_env** out) {
  if (!net || !cfg || !out) return fail(MAPDN_ERR_INVALID, "null argument");
  *out = nullptr;
  const int n = net->n_bus, nbr = net->n_branch, nl = net->n_load, ng = net->n_sgen;
  if (n < 2 || n > 65000) return fail(MAPDN_ERR_INVALID, "n_bus must be in [2, 65000]");
  if (nbr < 1 || nl < 0 || ng < 1) return fail(MAPDN_ERR_INVALID, "need >=1 branch and >=1 sgen");
  if (cfg->batch < 1) return fail(MAPDN_ERR_INVALID, "batch must be >= 1");
  if (!net->br_from || !net->br_to || !net->br_r || !net->br_x || !net->sgen_bus || !net->sgen_zone ||
      !net->bus_zone || (nl > 0 && !net->load_bus))
    return fail(MAPDN_ERR_INVALID, "missing required network array");
  if (net->slack_bus < 0 || net->slack_bus >= n) return fail(MAPDN_ERR_INVALID, "slack_bus out of range");
  if (!(net->base_mva > 0)) return fail(MAPDN_ERR_INVALID, "base_mva must be positive");
  if (cfg->barrier < 0 || cfg->barrier > 4) return fail(MAPDN_ERR_INVALID, "unknown voltage barrier");
  if (cfg->lanes_per_env != 0 && cfg->lanes_per_env != 4 && cfg->lanes_per_env != 8 && cfg->lanes_per_env != 16 &&
      cfg->lanes_per_env != 32 && cfg->lanes_per_env != 64 && cfg->lanes_per_env != 128)
    return fail(MAPDN_ERR_INVALID, "lanes_per_env must be 0, 4, 8, 16, 32, 64 or 128");
  for (int k = 0; k < nbr; ++k)
    if (net->br_from[k] < 0 || net->br_from[k] >= n || net->br_to[k] < 0 || net->br_to[k] >= n ||
        net->br_from[k] == net->br_to[k])
      return fail(MAPDN_ERR_INVALID, "branch endpoint out of range");
  for (int l = 0; l < nl; ++l)
    if (net->load_bus[l] < 0 || net->load_bus[l] >= n) return fail(MAPDN_ERR_INVALID, "load_bus out of range");
  for (int j = 0; j < ng; ++j)
    if (net->sgen_bus[j] < 0 || net->sgen_bus[j] >= n) return fail(MAPDN_ERR_INVALID, "sgen_bus out of range");
  if (prof) {
    if (!prof->pv || !prof->load_p || !prof->load_q || !prof->pv_std || !prof->load_p_std ||
        !prof->load_q_std || !prof->s_max || prof->n_rows < 2 || prof->steps_per_hour < 1)
      return fail(MAPDN_ERR_INVALID, "incomplete profile description");
  }
  MAPDN_ON_DEVICE(device);
  mapdn_env* e = new (std::nothrow) mapdn_env();
  if (!e) return fail(MAPDN_ERR_NOMEM, "out of host memory");
  e->device = device;
  e->cfg = *cfg;
  mapdn_status st = MAPDN_OK;
  auto bail = [&](mapdn_status s) { mapdn_destroy(e); return s; };
#define TRY(expr) do { st = (expr); if (st != MAPDN_OK) return bail(st); } while (0)
#define TRY_CUDA(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { \
      fail(MAPDN_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); return bail(MAPDN_ERR_CUDA); } } while (0)

  // ---- 1. Ybus on the device ----
  std::vector<double> br_r(net->br_r, net->br_r + nbr), br_x(net->br_x, net->br_x + nbr);
  std::vector<double> br_b = vec_or(net->br_b, nbr, 0.0), br_g = vec_or(net->br_g, nbr, 0.0);
  std::vector<double> br_tap = vec_or(net->br_tap, nbr, 1.0), br_sh = vec_or(net->br_shift_deg, nbr, 0.0);
  std::vector<unsigned char> br_st = vec_or<unsigned char>(net->br_status, nbr, 1);
  std::vector<unsigned char> br_line = vec_or<unsigned char>(net->br_is_line, nbr, 1);
  std::vector<double> gs = vec_or(net->bus_gs_mw, n, 0.0), bs = vec_or(net->bus_bs_mvar, n, 0.0);
  e->br_from.assign(net->br_from, net->br_from + nbr);
  e->br_to.assign(net->br_to, net->br_to + nbr);
  for (int k = 0; k < nbr; ++k)
    if (br_st[k] && br_r[k] == 0.0 && br_x[k] == 0.0) return bail(fail(MAPDN_ERR_INVALID, "zero-impedance branch"));
  {
    const double *d_r, *d_x, *d_b, *d_g, *d_tap, *d_sh, *d_gs, *d_bs;
    const unsigned char* d_st;
    const int *d_f, *d_t;
    double *d_ybr, *d_ydiag;
    TRY(dev_upload(e, br_r, &d_r)); TRY(dev_upload(e, br_x, &d_x)); TRY(dev_upload(e, br_b, &d_b));
    TRY(dev_upload(e, br_g, &d_g)); TRY(dev_upload(e, br_tap, &d_tap)); TRY(dev_upload(e, br_sh, &d_sh));
    TRY(dev_upload(e, br_st, &d_st)); TRY(dev_upload(e, e->br_from, &d_f)); TRY(dev_upload(e, e->br_to, &d_t));
    TRY(dev_upload(e, gs, &d_gs)); TRY(dev_upload(e, bs, &d_bs));
    TRY(dev_alloc(e, static_cast<size_t>(8) * nbr, &d_ybr)); TRY(dev_alloc(e, static_cast<size_t>(2) * n, &d_ydiag));
    MAPDN_LAUNCH(ybus_branch_kernel, (nbr + 127) / 128, 128, 0, 0, nbr, d_r, d_x, d_b, d_g, d_tap, d_sh, d_st, d_ybr);
    MAPDN_LAUNCH(ybus_diag_kernel, (n + 127) / 128, 128, 0, 0, n, nbr, d_f, d_t, d_ybr, d_gs, d_bs, 1.0 / net->base_mva, d_ydiag);
    TRY_CUDA(cudaGetLastError());
    e->launches += 2;
    e->ybr.resize(static_cast<size_t>(8) * nbr);
    e->ydiag.resize(static_cast<size_t>(2) * n);
    TRY_CUDA(cudaMemcpy(e->ybr.data(), d_ybr, e->ybr.size() * sizeof(double), cudaMemcpyDeviceToHost));
    TRY_CUDA(cudaMemcpy(e->ydiag.data(), d_ydiag, e->ydiag.size() * sizeof(double), cudaMemcpyDeviceToHost));
  }

  // ---- 2. symbolic analysis: merge parallel branches, check the net is radial, build the forest
  //         of PQ buses (slack removed) and re-root every tree at its centre ----
  struct Pair { double gab = 0, bab = 0, gba = 0, bba = 0; };   // Y[a,b], Y[b,a] with a < b
  std::map<std::pair<int, int>, Pair> pairs;
  for (int k = 0; k < nbr; ++k) {
    if (!br_st[k]) continue;
    const int f = e->br_from[k], t = e->br_to[k];
    const double* y = &e->ybr[8 * static_cast<size_t>(k)];
    Pair& pr = pairs[{std::min(f, t), std::max(f, t)}];
    if (f < t) { pr.gab += y[2]; pr.bab += y[3]; pr.gba += y[4]; pr.bba += y[5]; }   // Ybus[f,t]+=Yft, [t,f]+=Ytf
    else       { pr.gba += y[2]; pr.bba += y[3]; pr.gab += y[4]; pr.bab += y[5]; }
  }
  auto yoff = [&](int a, int b, double& g, double& bb) {          // Ybus[a,b]
    const Pair& pr = pairs[{std::min(a, b), std::max(a, b)}];
    if (a < b) { g = pr.gab; bb = pr.bab; } else { g = pr.gba; bb = pr.bba; }
  };
  const int slack = net->slack_bus;
  std::vector<std::vector<int>> adj(n);
  for (auto& kv : pairs) { adj[kv.first.first].push_back(kv.first.second); adj[kv.first.second].push_back(kv.first.first); }
  for (auto& a : adj) std::sort(a.begin(), a.end());
  {   // connectivity + radiality on the full graph
    std::vector<char> seen(n, 0);
    std::vector<int> q{slack};
    seen[slack] = 1;
    for (size_t qh = 0; qh < q.size(); ++qh)
      for (int v : adj[q[qh]]) if (!seen[v]) { seen[v] = 1; q.push_back(v); }
    if (static_cast<int>(q.size()) != n)
      return bail(fail(MAPDN_ERR_TOPOLOGY, "network is not connected to the slack bus (" +
                                               std::to_string(n - q.size()) + " unreachable buses)"));
  }
  // A radial net (|edges| = n - 1) takes the zero-fill tree solver; a meshed one the dense-LU fallback.
  const bool meshed = static_cast<int>(pairs.size()) != n - 1;
  if (meshed && n - 1 > 256)
    return bail(fail(MAPDN_ERR_TOPOLOGY, "network is meshed (" + std::to_string(pairs.size() - (n - 1)) +
                                             " loop-closing branches) and has more than 256 PQ buses: the dense "
                                             "fallback solver only covers small meshed feeders"));
  const int npq = n - 1;
  // BFS inside the PQ forest (never crossing the slack bus)
  auto bfs = [&](int src, std::vector<int>& dist, std::vector<int>& from) {
    std::vector<int> q{src};
    dist[src] = 0; from[src] = -1;
    for (size_t qh = 0; qh < q.size(); ++qh)
      for (int v : adj[q[qh]]) if (v != slack && dist[v] < 0) { dist[v] = dist[q[qh]] + 1; from[v] = q[qh]; q.push_back(v); }
    return q;
  };
  std::vector<int> roots;
  {
    std::vector<int> d0(n, -1), f0(n, -1);
    for (int s0 : adj[slack]) {                        // one tree per slack neighbour
      if (d0[s0] >= 0) continue;
      std::vector<int> comp = bfs(s0, d0, f0);
      int u = comp.back();                             // farthest from s0
      std::vector<int> d1(n, -1), f1(n, -1);
      std::vector<int> c1 = bfs(u, d1, f1);
      int v = c1.back();                               // farthest from u: u..v is a diameter
      int c = v;
      for (int k = 0; k < d1[v] / 2; ++k) c = f1[c];   // walk half-way back: the centre
      roots.push_back(c);
    }
  }
  std::vector<int> order, node_of_bus(n, -1), parent_bus(n, -1), depth(n, 0);
  order.reserve(npq);
  for (int r : roots) { node_of_bus[r] = static_cast<int>(order.size()); order.push_back(r); }
  for (size_t qh = 0; qh < order.size(); ++qh) {
    const int u = order[qh];
    for (int v : adj[u]) {
      if (v == slack || node_of_bus[v] >= 0) continue;
      node_of_bus[v] = static_cast<int>(order.size());
      parent_bus[v] = u;
      depth[v] = depth[u] + 1;
      order.push_back(v);
    }
  }
  node_of_bus[slack] = npq;
  std::vector<int> parent(npq, -1), nchild(npq, 0), height(npq, 0);
  for (int i = 0; i < npq; ++i)
    if (parent_bus[order[i]] >= 0) { parent[i] = node_of_bus[parent_bus[order[i]]]; nchild[parent[i]]++; }
  if (meshed) {   // no elimination forest: every bus is its own root, the sweeps are not used
    std::fill(parent.begin(), parent.end(), -1);
    std::fill(nchild.begin(), nchild.end(), 0);
    for (int b = 0; b < n; ++b) depth[b] = 0;
  }
  for (int i = npq - 1; i >= 0; --i)
    if (parent[i] >= 0) height[parent[i]] = std::max(height[parent[i]], height[i] + 1);
  std::vector<int> cfirst(npq + 1);
  cfirst[0] = static_cast<int>(roots.size());
  for (int i = 0; i < npq; ++i) cfirst[i + 1] = cfirst[i] + nchild[i];
  int max_h = 0;
  for (int i = 0; i < npq; ++i) max_h = std::max(max_h, height[i]);
  const int n_lev = max_h + 1;                          // = max depth + 1
  std::vector<uint16_t> elev(n_lev + 1), dlev(n_lev + 1);
  std::vector<int> eorder;
  for (int hgt = 0; hgt <= max_h; ++hgt) {
    elev[hgt] = static_cast<uint16_t>(eorder.size());
    for (int i = 0; i < npq; ++i) if (height[i] == hgt) eorder.push_back(i);
  }
  elev[n_lev] = static_cast<uint16_t>(eorder.size());
  {
    int d = 0;
    dlev[0] = 0;
    for (int i = 0; i < npq; ++i) while (depth[order[i]] > d) dlev[++d] = static_cast<uint16_t>(i);
    while (d < n_lev) dlev[++d] = static_cast<uint16_t>(npq);
  }
  int max_width = 0, max_children = 0;
  for (int l = 0; l < n_lev; ++l) max_width = std::max(max_width, elev[l + 1] - elev[l]);
  for (int i = 0; i < npq; ++i) max_children = std::max(max_children, nchild[i]);
  int G = cfg->lanes_per_env;
  if (G == 0) G = (npq <= 64) ? 8 : (npq <= 256 ? 32 : 64);      // measured on B200 (profiles/r02_sweeps.txt)
  if (meshed) G = 32;                    // the dense fallback works one warp per env     // measured on B200: 8 lanes/env for 33-bus feeders, a full warp beyond
  // Flat schedules for this G: a level wider than G takes several steps; idle lanes get the trash record.
  // Lanes follow chains: a bus is placed on the lane that handled its child (forward sweep) / its parent
  // (back sweep) in the immediately preceding step whenever that lane is free, so the dependent value can
  // stay in registers.
  const int trash = npq + 1;
  std::vector<uint64_t> esched, bsched;
  int n_wide_e = 0, n_narrow_b = 0;      // G > 32: forward steps [n_wide_e, end) and back steps [0, n_narrow_b) use warp 0 only
  {
    std::vector<int> lane_of(npq, -1), step_of(npq, -1), reg_child(npq, -1), epos(npq, -1);
    int cur = 0;
    // Multi-warp groups (G > 32): the levels near the roots hold a handful of buses. From the first level on after which no
    // level is wider than a warp ("narrow suffix" of the forward sweep / "narrow prefix" of the back sweep) only warp 0 of
    // the group works: those steps are packed into lanes 0..31 and synchronise with __syncwarp instead of a named barrier.
    int first_narrow_lev = n_lev;
    if (G > 32) { while (first_narrow_lev > 0 && elev[first_narrow_lev] - elev[first_narrow_lev - 1] <= 32) --first_narrow_lev; }
    n_wide_e = -1;
    for (int l = 0; l < n_lev; ++l) {
      const int w = elev[l + 1] - elev[l], nst = (w + G - 1) / G;
      const bool narrow = G > 32 && l >= first_narrow_lev;
      if (narrow && n_wide_e < 0) n_wide_e = cur;
      std::vector<int> slot(static_cast<size_t>(nst) * G, -1), inh(npq, -1);
      std::vector<int> rest;
      for (int k = elev[l]; k < elev[l + 1]; ++k) {
        const int i = eorder[k];
        int pick = -1;
        if (nchild[i] >= 1 && nchild[i] <= 2)
          for (int c = cfirst[i]; c < cfirst[i] + nchild[i]; ++c)
            if (step_of[c] == cur - 1 && slot[lane_of[c]] < 0 && (!narrow || lane_of[c] < 32) &&
                (pick < 0 || height[c] > height[pick])) pick = c;
        if (pick >= 0) { slot[lane_of[pick]] = i; inh[i] = pick; }
        else rest.push_back(i);
      }
      size_t pos = 0;
      for (int i : rest) { while (slot[pos] >= 0) ++pos; slot[pos] = i; }
      for (int sidx = 0; sidx < nst * G; ++sidx) {
        const int i = slot[sidx];
        if (i < 0) { esched.push_back(static_cast<uint64_t>(trash) | (static_cast<uint64_t>(npq) << 16) |
                                      (static_cast<uint64_t>(npq) << 32) | (static_cast<uint64_t>(kEschedReg0 | kEschedIdle) << 48)); continue; }
        lane_of[i] = sidx % G; step_of[i] = cur + sidx / G;
        uint64_t c0 = npq, c1 = npq, fl = kEschedLeaf;       // no child: zero update, nothing to fetch
        if (nchild[i] > 2) {
          c0 = cfirst[i]; c1 = cfirst[i] + 1; fl = static_cast<uint64_t>(std::min(nchild[i] - 2, 255)) | kEschedLoad0 | kEschedLoad1;
          if (nchild[i] - 2 > 255) return bail(fail(MAPDN_ERR_UNSUPPORTED, "a bus with more than 257 children"));
        } else if (nchild[i] >= 1) {
          const int a0 = inh[i] >= 0 ? inh[i] : cfirst[i];
          c0 = a0; fl = (inh[i] >= 0 && sidx / G == 0) ? kEschedReg0 : kEschedLoad0;
          if (fl & kEschedReg0) reg_child[i] = a0;
          if (nchild[i] == 2) { c1 = (a0 == cfirst[i]) ? cfirst[i] + 1 : cfirst[i]; fl |= kEschedLoad1; }
        }
        epos[i] = static_cast<int>(esched.size());
        esched.push_back(static_cast<uint64_t>(i) | (c0 << 16) | (c1 << 32) | (fl << 48));
      }
      cur += nst;
    }
    // a bus stores its Schur update only if its parent will fetch it from shared memory
    for (int i = 0; i < npq; ++i)
      if (parent[i] >= 0 && reg_child[parent[i]] != i) esched[epos[i]] |= static_cast<uint64_t>(kEschedStore) << 48;
    if (n_wide_e < 0) n_wide_e = cur;             // no narrow suffix
    // back sweep by depth: children inherit the lane of their parent (the child with the tallest subtree first)
    std::fill(lane_of.begin(), lane_of.end(), -1); std::fill(step_of.begin(), step_of.end(), -1);
    cur = 0;
    const int first_back_level = 1;      // the roots' dx = D^-1 r is already in place
    int last_narrow_dlev = first_back_level - 1;  // depth levels first_back_level .. last_narrow_dlev are narrow (prefix)
    if (G > 32) { while (last_narrow_dlev + 1 < n_lev && dlev[last_narrow_dlev + 2] - dlev[last_narrow_dlev + 1] <= 32) ++last_narrow_dlev; }
    n_narrow_b = 0;
    for (int l = first_back_level; l < n_lev; ++l) {
      const int w = dlev[l + 1] - dlev[l], nst = (w + G - 1) / G;
      if (G > 32 && l <= last_narrow_dlev) n_narrow_b = cur + nst;
      std::vector<int> slot(static_cast<size_t>(nst) * G, -1);
      std::vector<char> reg(npq, 0);
      std::vector<int> nodes;
      for (int i = dlev[l]; i < dlev[l + 1]; ++i) nodes.push_back(i);
      std::stable_sort(nodes.begin(), nodes.end(), [&](int a, int b) { return height[a] > height[b]; });
      std::vector<int> rest;
      for (int i : nodes) {
        const int pa = parent[i];
        if (pa >= 0 && step_of[pa] == cur - 1 && lane_of[pa] >= 0 && slot[lane_of[pa]] < 0) { slot[lane_of[pa]] = i; reg[i] = 1; }
        else rest.push_back(i);
      }
      size_t pos = 0;
      for (int i : rest) { while (slot[pos] >= 0) ++pos; slot[pos] = i; }
      for (int sidx = 0; sidx < nst * G; ++sidx) {
        const int i = slot[sidx];
        if (i < 0) {
          bsched.push_back(static_cast<uint64_t>(trash) | (static_cast<uint64_t>(npq) << 16) |
                           (static_cast<uint64_t>(kBschedRegParent | kBschedIdle) << 32));
          continue;
        }
        lane_of[i] = sidx % G; step_of[i] = cur + sidx / G;
        bsched.push_back(static_cast<uint64_t>(i) | (static_cast<uint64_t>(parent[i] >= 0 ? parent[i] : npq) << 16) |
                         (static_cast<uint64_t>((reg[i] && sidx / G == 0) ? kBschedRegParent : 0u) << 32));
      }
      cur += nst;
    }
  }
  if (getenv("MAPDN_DEBUG_SCHED")) {
    int nreg = 0, nl0 = 0, nl1 = 0, nreal = 0;
    for (uint64_t e2 : esched) { if ((e2 & 0xFFFF) == (uint64_t)trash) continue; ++nreal; unsigned fl = e2 >> 48; nreg += !!(fl & kEschedReg0); nl0 += !!(fl & kEschedLoad0); nl1 += !!(fl & kEschedLoad1); }
    int breg = 0, breal = 0;
    for (uint64_t b2 : bsched) { if ((b2 & 0xFFFF) == (uint64_t)trash) continue; ++breal; breg += (b2 >> 32) & 1; }
    fprintf(stderr, "[sched] G=%d levels=%d esteps=%zu real=%d reg0=%d load0=%d load1=%d | bsteps=%zu real=%d regp=%d\n", G, n_lev,
            esched.size() / G, nreal, nreg, nl0, nl1, bsched.size() / G, breal, breg);
  }
  if (bsched.empty())      // a forest of single buses: one all-idle step
    bsched.assign(G, static_cast<uint64_t>(trash) | (static_cast<uint64_t>(npq) << 16) |
                         (static_cast<uint64_t>(kBschedRegParent | kBschedIdle) << 32));
  const int n_esteps = static_cast<int>(esched.size()) / G, n_bsteps = static_cast<int>(bsched.size()) / G;

  // ---- 2b. bank-conflict-aware relabelling of the node records ----
  // A node record is 144 B = 9 x 16 B, so the 16-byte bank group of field f of node i is (i + f) mod 8: the eight lanes of a
  // quarter-warp (one 128-bit access wavefront) are conflict free iff their node ids differ mod 8. The passes own nodes
  // by id (conflict free by construction) but reach parents / children by pointer, and the sweeps touch whatever the
  // schedules say; ncu counted 25 % of the shared-load wavefronts as conflicts with the breadth-first ids. The ids are
  // free to choose, so pick a permutation that minimises the weighted number of extra wavefronts over every access group
  // of the kernel (simulated annealing on pairwise swaps, deterministic; identity when it does not apply).
  std::vector<int> kid0(npq, npq), kid1(npq, npq);
  for (int i = 0; i < npq; ++i) { if (nchild[i] > 0) kid0[i] = cfirst[i]; if (nchild[i] > 1) kid1[i] = cfirst[i] + 1; }
  double relabel_cost0 = 0.0, relabel_cost1 = 0.0;
  if (!meshed && max_children <= 2 && G >= 8 && npq >= 8 && !getenv("MAPDN_NO_RELABEL")) {
    struct Grp { std::vector<int> nodes; double w; };
    std::vector<Grp> groups;                                  // groups whose members do not depend on the labelling
    const double w_iter = 4.5;                                // Newton iterations per step (sweeps and passes run that often)
    auto add_quarters = [&](const std::vector<int>& per_lane, double w) {      // per_lane: node per lane of the group (-1: no access)
      for (int q = 0; q < G / 8; ++q) {
        Grp g; g.w = w;
        for (int l = 8 * q; l < 8 * q + 8; ++l) if (per_lane[l] >= 0) g.nodes.push_back(per_lane[l]);
        std::sort(g.nodes.begin(), g.nodes.end());
        g.nodes.erase(std::unique(g.nodes.begin(), g.nodes.end()), g.nodes.end());      // same address = broadcast
        if (g.nodes.size() > 1) groups.push_back(std::move(g));
      }
    };
    std::vector<int> own(G), c0v(G), c1v(G);
    for (size_t st = 0; st < esched.size() / G; ++st) {
      for (int l = 0; l < G; ++l) {
        const uint64_t ed = esched[st * G + l];
        const unsigned fl = static_cast<unsigned>(ed >> 48);
        own[l] = static_cast<int>(ed & 0xFFFFu);
        c0v[l] = (fl & kEschedLoad0) ? static_cast<int>((ed >> 16) & 0xFFFFu) : -1;
        c1v[l] = (fl & kEschedLoad1) ? static_cast<int>((ed >> 32) & 0xFFFFu) : -1;
      }
      add_quarters(own, 2.0 * w_iter);                        // own blocks: loaded (prefetch) and stored
      add_quarters(c0v, w_iter); add_quarters(c1v, w_iter);
    }
    for (size_t st = 0; st < bsched.size() / G; ++st) {
      for (int l = 0; l < G; ++l) {
        const uint64_t bd = bsched[st * G + l];
        const unsigned bfl = static_cast<unsigned>(bd >> 32);
        own[l] = static_cast<int>(bd & 0xFFFFu);
        c0v[l] = (bfl & (kBschedRegParent | kBschedIdle)) ? -1 : static_cast<int>((bd >> 16) & 0xFFFFu);
      }
      add_quarters(own, 2.0 * w_iter); add_quarters(c0v, w_iter);
    }
    for (int b0 = 0; b0 < n; b0 += G) {                       // epilogue: per-bus loop, buses b0 + lane
      for (int l = 0; l < G; ++l) own[l] = (b0 + l < n) ? node_of_bus[b0 + l] : -1;
      add_quarters(own, 1.0);
    }
    {
      std::vector<int> lf, lt;
      for (int k = 0; k < nbr; ++k) if (br_line[k]) { lf.push_back(node_of_bus[e->br_from[k]]); lt.push_back(node_of_bus[e->br_to[k]]); }
      for (size_t k0 = 0; k0 < lf.size(); k0 += G) {
        for (int l = 0; l < G; ++l) { own[l] = (k0 + l < lf.size()) ? lf[k0 + l] : -1; c0v[l] = (k0 + l < lt.size()) ? lt[k0 + l] : -1; }
        add_quarters(own, 1.0); add_quarters(c0v, 1.0);
      }
    }
    // lab[base id] = label; sentinel / trash keep their ids
    std::vector<int> lab(npq + 2), inv(npq + 2);
    for (int i = 0; i < npq + 2; ++i) lab[i] = inv[i] = i;
    auto extra = [&](const int* ids, int cnt) {               // extra wavefronts of one access: max multiplicity - 1
      int c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      int mx = 0;
      for (int k = 0; k < cnt; ++k) mx = std::max(mx, ++c[ids[k] & 7]);
      return std::max(0, mx - 1);
    };
    auto cost = [&]() {
      double tot = 0.0;
      int ids[8];
      for (const Grp& g : groups) {
        int cnt = 0;
        for (int v : g.nodes) ids[cnt++] = lab[v];
        tot += g.w * extra(ids, cnt);
      }
      // passes: label L is handled by lane L % G in round L / G; neighbours reached by pointer
      for (int L0 = 0; L0 < npq; L0 += 8) {
        int pa[8], k0[8], k1[8], np = 0, n0 = 0, n1 = 0;
        auto push_unique = [](int* a, int& cnt, int v) { for (int k = 0; k < cnt; ++k) if (a[k] == v) return; a[cnt++] = v; };
        for (int L = L0; L < std::min(npq, L0 + 8); ++L) {
          const int i = inv[L];
          push_unique(pa, np, parent[i] >= 0 ? lab[parent[i]] : npq);
          push_unique(k0, n0, lab[kid0[i]]); push_unique(k1, n1, lab[kid1[i]]);
        }
        tot += w_iter * (extra(pa, np) + extra(k0, n0) + extra(k1, n1));
      }
      return tot;
    };
    relabel_cost0 = cost();
    double cur = relabel_cost0, best = cur;
    std::vector<int> best_lab = lab;
    uint64_t rng = 0x9E3779B97F4A7C15ull;
    auto rnd = [&]() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return rng; };
    const int iters = std::min(400 * npq, 30000);
    double T = std::max(1.0, 0.02 * cur);
    const double cool = std::pow(1e-3, 1.0 / std::max(1, iters));
    for (int it = 0; it < iters && best > 0.0; ++it, T *= cool) {
      const int a = static_cast<int>(rnd() % npq), b = static_cast<int>(rnd() % npq);
      if (a == b || ((lab[a] ^ lab[b]) & 7) == 0) continue;  // same residue: no effect on any group
      std::swap(lab[a], lab[b]); inv[lab[a]] = a; inv[lab[b]] = b;
      const double c2 = cost();
      const double u = static_cast<double>(rnd() >> 11) * (1.0 / 9007199254740992.0);
      if (c2 <= cur || u < std::exp((cur - c2) / T)) {
        cur = c2;
        if (cur < best) { best = cur; best_lab = lab; }
      } else {
        std::swap(lab[a], lab[b]); inv[lab[a]] = a; inv[lab[b]] = b;
      }
    }
    lab = best_lab;
    relabel_cost1 = best;
    if (best < relabel_cost0) {
      // apply: new id of base node i is lab[i]
      std::vector<int> order2(npq), parent2(npq), nchild2(npq), k0b(npq), k1b(npq);
      for (int i = 0; i < npq; ++i) {
        const int L = lab[i];
        order2[L] = order[i];
        parent2[L] = parent[i] >= 0 ? lab[parent[i]] : -1;
        nchild2[L] = nchild[i];
        k0b[L] = lab[kid0[i]]; k1b[L] = lab[kid1[i]];
      }
      order = order2; parent = parent2; nchild = nchild2; kid0 = k0b; kid1 = k1b;
      for (int i = 0; i < npq; ++i) node_of_bus[order[i]] = i;
      auto map16 = [&](uint64_t v) { return static_cast<uint64_t>(lab[static_cast<int>(v & 0xFFFFu)]); };
      for (uint64_t& ed : esched)
        ed = (ed & 0xFFFF000000000000ull) | map16(ed) | (map16(ed >> 16) << 16) | (map16(ed >> 32) << 32);
      for (uint64_t& bd : bsched)
        bd = (bd & 0xFFFFFFFF00000000ull) | map16(bd) | (map16(bd >> 16) << 16);
    }
    if (getenv("MAPDN_DEBUG_SCHED"))
      fprintf(stderr, "[relabel] weighted extra shared-memory wavefronts per env-step: %.1f -> %.1f (%d swaps tried)\n",
              relabel_cost0, relabel_cost1, iters);
  }

  // ---- 3. element -> node maps (needed by the hot blob) ----
  const int na = npq + 2;      // + sentinel + trash records
  std::vector<uint16_t> lptr(npq + 2, 0), lidx(std::max(1, nl)), sptr(npq + 2, 0), sidx(ng), xptr(npq + 2, 0), xidx;
  {
    std::vector<std::vector<int>> ln(npq + 1), sn(npq + 1);
    for (int l = 0; l < nl; ++l) ln[node_of_bus[net->load_bus[l]]].push_back(l);
    for (int j = 0; j < ng; ++j) sn[node_of_bus[net->sgen_bus[j]]].push_back(j);
    int a = 0, b = 0;
    for (int i = 0; i <= npq; ++i) {
      lptr[i] = static_cast<uint16_t>(a); sptr[i] = static_cast<uint16_t>(b);
      xptr[i] = static_cast<uint16_t>(xidx.size());
      for (int l : ln[i]) lidx[a++] = static_cast<uint16_t>(l);
      const int bus = (i == npq) ? slack : order[i];
      for (int j : sn[i]) {
        sidx[b++] = static_cast<uint16_t>(j);
        if (net->sgen_zone[j] == net->bus_zone[bus]) xidx.push_back(static_cast<uint16_t>(j));   // reference :238-244
      }
    }
    lptr[npq + 1] = static_cast<uint16_t>(a); sptr[npq + 1] = static_cast<uint16_t>(b);
    xptr[npq + 1] = static_cast<uint16_t>(xidx.size());
  }
  // obs program (reference get_obs :232-274): per agent [P_zone | Q_zone | pv | q | vm_zone | va_zone | 0...].
  // Hot copy: double offset of the source inside the env slab. Cold copy (get_obs_kernel): kind | node.
  const int ssm = (cfg->state_space_mask & 31) ? (cfg->state_space_mask & 31) : 31;
  const bool ss_dem = ssm & 1, ss_pv = ssm & 2, ss_q = ssm & 4, ss_vm = ssm & 8, ss_va = ssm & 16;
  int obs_dim = 0;
  std::vector<std::vector<int>> zb(ng);
  for (int a = 0; a < ng; ++a) {
    for (int b = 0; b < n; ++b) if (net->bus_zone[b] == net->sgen_zone[a]) zb[a].push_back(b);
    const int nz = static_cast<int>(zb[a].size());
    obs_dim = std::max(obs_dim, nz * (2 * ss_dem + ss_vm + ss_va) + ss_pv + ss_q);
  }
  const int pvq_off2 = kNodeArrays2 * na, scratch_off2 = pvq_off2 + ng;
  if (2 * (scratch_off2 + (scratch_doubles_for(ng, nl, G, false) + 1) / 2) >= 65535)
    return bail(fail(MAPDN_ERR_UNSUPPORTED, "network too large for 16-bit slab offsets"));
  std::vector<uint16_t> obs_off(static_cast<size_t>(ng) * obs_dim);
  std::vector<unsigned> obs_src(static_cast<size_t>(ng) * obs_dim, 0u);
  std::vector<int> obs_xptr(static_cast<size_t>(ng) * obs_dim + 1, 0), obs_xidx;
  std::vector<int> agent_len(ng, 0);
  enum { K_ZERO = 0, K_P = 1, K_Q = 2, K_PV = 3, K_QSG = 4, K_VM = 5, K_VA = 6 };
  for (int a = 0; a < ng; ++a) {
    // entry list of this agent in the reference's order (:254-266), then zero padding (:270-274)
    std::vector<std::pair<unsigned, int>> ent;           // (kind, bus or sgen)
    if (ss_dem) { for (int b : zb[a]) ent.push_back({K_P, b}); for (int b : zb[a]) ent.push_back({K_Q, b}); }
    if (ss_pv) ent.push_back({K_PV, a});
    if (ss_q) ent.push_back({K_QSG, a});
    if (ss_vm) for (int b : zb[a]) ent.push_back({K_VM, b});
    if (ss_va) for (int b : zb[a]) ent.push_back({K_VA, b});
    agent_len[a] = static_cast<int>(ent.size());
    for (int k = 0; k < obs_dim; ++k) {
      const size_t idx = static_cast<size_t>(a) * obs_dim + k;
      obs_xptr[idx] = static_cast<int>(obs_xidx.size());
      unsigned kind = K_ZERO, ix = 0;
      int off = 2 * (npq * kNodeArrays2 + A_UP);               // sentinel record's UP.x: constant zero
      if (k < static_cast<int>(ent.size())) {
        kind = ent[k].first;
        const int t2 = ent[k].second;
        if (kind == K_P || kind == K_Q) {
          ix = static_cast<unsigned>(node_of_bus[t2]);
          off = 2 * (node_of_bus[t2] * kNodeArrays2 + A_OP) + (kind == K_P ? 0 : 1);
          for (int j = 0; j < ng; ++j)
            if (net->sgen_zone[j] == net->sgen_zone[a] && net->sgen_bus[j] == t2) obs_xidx.push_back(j);
        } else if (kind == K_PV) { ix = t2; off = 2 * pvq_off2 + t2; }
        else if (kind == K_QSG) { ix = t2; off = 2 * pvq_off2 + ng + t2; }
        else { ix = static_cast<unsigned>(node_of_bus[t2]); off = 2 * (node_of_bus[t2] * kNodeArrays2 + A_VV) + (kind == K_VM ? 0 : 1); }
      }
      obs_src[idx] = (kind << 28) | ix;
      obs_off[idx] = static_cast<uint16_t>(off);
    }
  }
  obs_xptr[static_cast<size_t>(ng) * obs_dim] = static_cast<int>(obs_xidx.size());
  // the same program without the padding: agent blocks back to back, the row rounded up to 4 entries (16-byte pieces of
  // fp32 rows) with reads of the zero slot
  std::vector<uint16_t> obs_compact;
  std::vector<int> agent_off(ng, 0);
  for (int a = 0; a < ng; ++a) {
    agent_off[a] = static_cast<int>(obs_compact.size());
    for (int k = 0; k < agent_len[a]; ++k) obs_compact.push_back(obs_off[static_cast<size_t>(a) * obs_dim + k]);
  }
  while (obs_compact.size() % 4) obs_compact.push_back(static_cast<uint16_t>(2 * (npq * kNodeArrays2 + A_UP)));
  // state program (reference get_state :213-230), bus-indexed
  std::vector<unsigned> state_src;
  if (ss_dem) { for (int b = 0; b < n; ++b) state_src.push_back((7u << 28) | b); for (int b = 0; b < n; ++b) state_src.push_back((8u << 28) | b); }
  if (ss_pv) for (int j = 0; j < ng; ++j) state_src.push_back((static_cast<unsigned>(K_PV) << 28) | j);
  if (ss_q) for (int j = 0; j < ng; ++j) state_src.push_back((static_cast<unsigned>(K_QSG) << 28) | j);
  if (ss_vm) for (int b = 0; b < n; ++b) state_src.push_back((static_cast<unsigned>(K_VM) << 28) | b);
  if (ss_va) for (int b = 0; b < n; ++b) state_src.push_back((9u << 28) | b);
  const int state_dim = static_cast<int>(state_src.size());

  // ---- 3a. line-loss table + scaling ----
  std::vector<double> lscale = vec_or(net->load_scaling, nl, 1.0), sscale = vec_or(net->sgen_scaling, ng, 1.0);
  std::vector<uint16_t> line_nodes;
  std::vector<double> line_c;
  for (int k = 0; k < nbr; ++k) {
    if (!br_line[k]) continue;
    const double* y = &e->ybr[8 * static_cast<size_t>(k)];
    line_nodes.push_back(static_cast<uint16_t>(node_of_bus[e->br_from[k]]));
    line_nodes.push_back(static_cast<uint16_t>(node_of_bus[e->br_to[k]]));
    // pl = Re(Sf + St) = Gff|Vf|^2 + Gtt|Vt|^2 + (Gft+Gtf) Re(Vf Vt*) + (Bft-Btf) Im(Vf Vt*)   [x baseMVA]
    line_c.push_back(y[0] * net->base_mva); line_c.push_back(y[6] * net->base_mva);
    line_c.push_back((y[2] + y[4]) * net->base_mva); line_c.push_back((y[3] - y[5]) * net->base_mva);
  }
  const int n_line = static_cast<int>(line_nodes.size() / 2);

  // PQ-PQ Ybus pattern (CSR) for the dense fallback
  std::vector<uint16_t> nbr_ptr(1, 0), nbr_idx;
  std::vector<double> nbr_y;
  if (meshed) {
    nbr_ptr.assign(npq + 1, 0);
    for (int i = 0; i < npq; ++i) {
      const int b = order[i];
      for (int v : adj[b]) {
        if (v == slack) continue;
        double g, bb;
        yoff(b, v, g, bb);
        nbr_idx.push_back(static_cast<uint16_t>(node_of_bus[v])); nbr_y.push_back(g); nbr_y.push_back(bb);
      }
      nbr_ptr[i + 1] = static_cast<uint16_t>(nbr_idx.size());
    }
  }
  // ---- 3b. hot static blob ----
  HotLayout hl{};
  int bytes_core = 0, bytes_full = 0;
  {
    int off = 0;
    auto take = [&](size_t bytes) { int o = off; off += static_cast<int>((bytes + 15) / 16 * 16); return o; };
    hl.yup = take(16 * npq); hl.ydn = take(16 * (npq + 1)); hl.yii = take(16 * npq);
    hl.ndesc = take(8 * npq); hl.esched = take(8 * esched.size()); hl.bsched = take(8 * bsched.size());
    hl.lptr = take(2 * lptr.size()); hl.lidx = take(2 * lidx.size());
    hl.sptr = take(2 * sptr.size()); hl.sidx = take(2 * sidx.size());
    hl.xptr = take(2 * xptr.size()); hl.xidx = take(2 * std::max<size_t>(1, xidx.size()));
    hl.node_of_bus = take(2 * n);
    hl.nbr_ptr = take(2 * nbr_ptr.size()); hl.nbr_idx = take(2 * std::max<size_t>(1, nbr_idx.size()));
    hl.nbr_y = take(8 * std::max<size_t>(2, nbr_y.size()));
    bytes_core = off;
    // the once-per-step tables go last: the TMA copy either includes them (hl.bytes = bytes_full) or stops before them
    if (line_nodes.empty()) { line_nodes.assign(2, 0); line_c.assign(4, 0.0); }
    hl.ysl = take(16 * npq); hl.obs_off = take(2 * obs_off.size());
    hl.line_nodes = take(2 * line_nodes.size()); hl.line_c = take(8 * line_c.size());
    bytes_full = off;
    hl.bytes = bytes_full; hl.tables_in_blob = 1;
  }
  std::vector<unsigned char> hot(bytes_full, 0);
  std::vector<double> ysl_cold(2 * static_cast<size_t>(npq), 0.0);     // Y[i,slack]: cold table, non-zero for a few buses
  std::vector<int> sl_node;
  std::vector<double> sl_y;
  {
    double* yup = reinterpret_cast<double*>(hot.data() + hl.yup); double* ydn = reinterpret_cast<double*>(hot.data() + hl.ydn);
    double* yii = reinterpret_cast<double*>(hot.data() + hl.yii);
    double* ysl = ysl_cold.data();
    uint64_t* ndesc = reinterpret_cast<uint64_t*>(hot.data() + hl.ndesc);
    for (int i = 0; i < npq; ++i) {
      const int b = order[i];
      yii[2 * i] = e->ydiag[2 * b]; yii[2 * i + 1] = e->ydiag[2 * b + 1];
      if (parent[i] >= 0) {
        yoff(b, parent_bus[b], yup[2 * i], yup[2 * i + 1]);       // Y[i,parent]
        yoff(parent_bus[b], b, ydn[2 * i], ydn[2 * i + 1]);       // Y[parent,i]
      }
      if (pairs.count({std::min(b, slack), std::max(b, slack)})) {
        yoff(b, slack, ysl[2 * i], ysl[2 * i + 1]);               // Y[i,slack]
        double g, bb;
        yoff(slack, b, g, bb);                                     // Y[slack,i]
        sl_node.push_back(i); sl_y.push_back(g); sl_y.push_back(bb);
      }
      // parent | child0 | child1 | number of further children (contiguous after child1); npq = zero slot
      const uint64_t pa = parent[i] >= 0 ? static_cast<uint64_t>(parent[i]) : npq;   // roots: sentinel, Y = 0
      const uint64_t c0 = static_cast<uint64_t>(kid0[i]), c1 = static_cast<uint64_t>(kid1[i]);   // npq = none
      const uint64_t nx = nchild[i] > 2 ? nchild[i] - 2 : 0;
      const uint64_t sl_adj = pairs.count({std::min(b, slack), std::max(b, slack)}) ? 1 : 0;
      ndesc[i] = pa | (c0 << 16) | (c1 << 32) | (nx << 48) | (sl_adj << 63);
    }
    {   // the slack injection sums over the slack's neighbours in this order: ascending bus index, so that the relabelling
        // of section 2b cannot reorder the sum when the slack has several neighbours
      std::vector<int> ks(sl_node.size());
      for (size_t k = 0; k < ks.size(); ++k) ks[k] = static_cast<int>(k);
      std::sort(ks.begin(), ks.end(), [&](int a, int b) { return order[sl_node[a]] < order[sl_node[b]]; });
      std::vector<int> node2;
      std::vector<double> y2;
      for (int k : ks) { node2.push_back(sl_node[k]); y2.push_back(sl_y[2 * k]); y2.push_back(sl_y[2 * k + 1]); }
      sl_node.swap(node2); sl_y.swap(y2);
    }
    std::memcpy(hot.data() + hl.esched, esched.data(), 8 * esched.size());
    std::memcpy(hot.data() + hl.bsched, bsched.data(), 8 * bsched.size());
    std::memcpy(hot.data() + hl.lptr, lptr.data(), 2 * lptr.size());
    if (nl) std::memcpy(hot.data() + hl.lidx, lidx.data(), 2 * static_cast<size_t>(nl));
    std::memcpy(hot.data() + hl.sptr, sptr.data(), 2 * sptr.size());
    std::memcpy(hot.data() + hl.sidx, sidx.data(), 2 * sidx.size());
    std::memcpy(hot.data() + hl.xptr, xptr.data(), 2 * xptr.size());
    if (!xidx.empty()) std::memcpy(hot.data() + hl.xidx, xidx.data(), 2 * xidx.size());
    std::memcpy(hot.data() + hl.ysl, ysl_cold.data(), 8 * ysl_cold.size());
    std::memcpy(hot.data() + hl.obs_off, obs_off.data(), 2 * obs_off.size());
    std::memcpy(hot.data() + hl.line_nodes, line_nodes.data(), 2 * line_nodes.size());
    std::memcpy(hot.data() + hl.line_c, line_c.data(), 8 * line_c.size());
    uint16_t* nob = reinterpret_cast<uint16_t*>(hot.data() + hl.node_of_bus);
    for (int b = 0; b < n; ++b) nob[b] = static_cast<uint16_t>(node_of_bus[b]);
    std::memcpy(hot.data() + hl.nbr_ptr, nbr_ptr.data(), 2 * nbr_ptr.size());
    if (!nbr_idx.empty()) {
      std::memcpy(hot.data() + hl.nbr_idx, nbr_idx.data(), 2 * nbr_idx.size());
      std::memcpy(hot.data() + hl.nbr_y, nbr_y.data(), 8 * nbr_y.size());
    }
  }

  // ---- 5. launch geometry ----
  cudaDeviceProp dp{};
  TRY_CUDA(cudaGetDeviceProperties(&dp, device));
  const size_t max_smem = dp.sharedMemPerBlockOptin;
  // envs per CTA: sub-warp groups pack 32/G envs into each of 1..4 solver warps; multi-warp groups (G = 64 / 128)
  // put 1..4 envs of G threads in a CTA. Fewer envs per CTA when that spreads the batch over all SMs.
  const int unit = (G <= 32) ? 32 / G : 1;               // envs added per step of the search
  const int n_sm = dp.multiProcessorCount;
  int stride2 = 0, epb = 0;
  bool stage_rec = false;
  // Two ways to buy shared memory when it limits the envs per SM, both with a price (measured, profiles/): (a) the four
  // once-per-step tables (Y[i,slack], obs program, line tables) stay in global memory instead of the staged blob - their
  // first touch after an L2 flush is an HBM round trip at the start of the epilogue, softened by an L2 prefetch at kernel
  // start; (b) the prologue stages the scaled loads inside the node records - index arithmetic, +1.3 k cycles per step on
  // case33. Each is used only if it lets the batch finish in fewer rounds (case322 x 1024: 4 envs per SM and 2 rounds
  // instead of 3 and 3).
  struct Plan { bool cold, rec, ok; int st2, epb; long long rounds; };
  auto smem_with = [&](bool cold, int st2, int c) {
    return static_cast<size_t>(cold ? bytes_core : bytes_full) + static_cast<size_t>(c) * (st2 * 16 + 16);   // + helper scalars
  };
  auto make_plan = [&](bool cold, bool rec) {
    Plan pl{cold, rec, false, 0, 0, 0};
    if (rec && !stage_fits_records(npq, nl)) return pl;
    pl.st2 = env_stride2_for(npq, ng, nl, G, rec);
    // measured on B200 (profiles/): two solver warps per CTA for small sub-warp groups, four for one-warp envs,
    // as many multi-warp envs as fit (<= 512 solver threads)
    int c_epb = (G <= 16) ? 2 * unit : 4 * unit;
    if (G > 32) while (c_epb > 1 && c_epb * G > 512) --c_epb;
    // Few-round batches (the BASELINE.json configs): one CTA per SM holding ceil(B / (SMs * rounds)) envs balances the
    // SMs exactly (case33 x 4096: 147 CTAs of 28 envs instead of 512 of 8, i.e. 7 instead of up to 8 solver warps on
    // the busiest SM; case141 x 2048: 2 rounds of 7). Many-round batches keep several small CTAs per SM.
    auto fits = [&](int c) { return smem_with(cold, pl.st2, c) <= max_smem && c * G <= (G <= 32 ? 256 : 512); };
    for (int r = 1; r <= 3; ++r) {
      int c = (cfg->batch + n_sm * r - 1) / (n_sm * r);
      c = (c + unit - 1) / unit * unit;
      if (fits(c)) { c_epb = std::max(c_epb, c); break; }
    }
    if (const char* ov = getenv("MAPDN_EPB")) c_epb = std::max(unit, atoi(ov) / unit * unit);   // tuning override
    while (c_epb > unit && (smem_with(cold, pl.st2, c_epb) > max_smem || (G <= 32 && c_epb * G > 256))) c_epb -= unit;
    pl.epb = c_epb;
    pl.ok = smem_with(cold, pl.st2, c_epb) <= max_smem;
    pl.rounds = (cfg->batch + static_cast<long long>(c_epb) * n_sm - 1) / (static_cast<long long>(c_epb) * n_sm);
    return pl;
  };
  bool cold_tables = false;
  size_t least_smem = SIZE_MAX;          // the smallest footprint of any plan (one step of `unit` envs): reported when none fits
  {
    const Plan plans[4] = {make_plan(false, false), make_plan(false, true), make_plan(true, false), make_plan(true, true)};   // cheapest first
    for (const Plan& pl : plans) if (pl.st2 > 0) least_smem = std::min(least_smem, smem_with(pl.cold, pl.st2, unit));
    const Plan* best = nullptr;
    for (const Plan& pl : plans) if (pl.ok && (!best || pl.rounds < best->rounds)) best = &pl;
    if (const char* ov = getenv("MAPDN_PLAN")) {             // tuning override: 0..3 = index into the list above
      const int k = atoi(ov);
      if (k >= 0 && k < 4 && plans[k].ok) best = &plans[k];
    }
    if (best) { stride2 = best->st2; epb = best->epb; stage_rec = best->rec; cold_tables = best->cold; }
  }
  hl.tables_in_blob = cold_tables ? 0 : 1;
  hl.bytes = cold_tables ? bytes_core : bytes_full;
  auto smem_for = [&](int c) { return smem_with(cold_tables, stride2, c); };
  if (epb == 0 || smem_for(epb) > max_smem)
    return bail(fail(MAPDN_ERR_UNSUPPORTED, "network too large for the shared-memory resident solver (" +
                                                std::to_string(least_smem) + " B needed, " + std::to_string(max_smem) +
                                                " B available)"));
  e->dense = meshed;
  e->G = G; e->threads = epb * G; e->epb = epb; e->smem = static_cast<int>(smem_for(epb));
  {   // helper warps (next profile rows + noise, concurrent with the Newton iteration): one per 256 Box-Muller pairs of a
      // CTA round, at most 4 -- a single warp was the critical path of case322 (197 -> 169 us with two)
    const int n_pair = (ng + 2 * nl + 1) / 2;
    e->helper_threads = 32 * std::min(4, std::max(1, (epb * n_pair + kHelperPairsPerWarp - 1) / kHelperPairsPerWarp));
  }
  if (const char* ov = getenv("MAPDN_HELPERS")) e->helper_threads = 32 * std::min(4, std::max(1, atoi(ov)));   // tuning override
  for (int mode = 0; mode < 4; ++mode) {
    KernelFn fn = kernel_for(G, mode, meshed);
    // the attribute belongs to the function, not to the handle: always allow the device maximum, so that creating a
    // second handle with a smaller footprint cannot break the launches of the first
    cudaFuncAttributes fa{};
    TRY_CUDA(cudaFuncGetAttributes(&fa, reinterpret_cast<const void*>(fn)));
    const int dyn_max = static_cast<int>(max_smem - fa.sharedSizeBytes);        // opt-in limit minus the static part
    if (e->smem > dyn_max)
      return bail(fail(MAPDN_ERR_UNSUPPORTED, "network too large for the shared-memory resident solver"));
    TRY_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_max));
  }
  {
    int per_sm = 0;
    TRY_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel_for(G, MODE_STEP, meshed), e->threads + e->helper_threads, e->smem));
    e->max_blocks = std::max(1, per_sm) * dp.multiProcessorCount;
    if (meshed) e->max_blocks = std::min(e->max_blocks, 2 * dp.multiProcessorCount);   // bounds the dense workspace
  }

  // ---- 6. upload + env state ----
  Params& P = e->base;
  P.n_bus = n; P.npq = npq; P.n_load = nl; P.n_sgen = ng; P.n_line = n_line; P.n_lev = n_lev;
  P.obs_dim = obs_dim; P.state_dim = state_dim; P.n_slack_adj = static_cast<int>(sl_node.size());
  P.n_esteps = n_esteps; P.n_bsteps = n_bsteps; P.has_extra_children = max_children > 2;
  P.n_wide_e = std::min(n_wide_e, n_esteps); P.n_narrow_b = std::min(n_narrow_b, n_bsteps);
  P.slack_bus = slack;
  P.nb = cfg->batch; P.env_stride2 = stride2; P.pvq_off2 = pvq_off2; P.scratch_off2 = scratch_off2; P.hot_layout = hl;
  P.helper_off = hl.bytes + e->epb * stride2 * 16;
  P.stage_in_records = stage_rec ? 1 : 0;
  P.obs_skip_off = -1;
  e->obs_zero_off = 2 * (npq * kNodeArrays2 + A_UP);
  TRY(dev_upload(e, obs_compact, &P.obs_compact_prog));
  P.obs_compact_len = 0;
  e->agent_len = agent_len; e->agent_off = agent_off; e->compact_row = static_cast<int>(obs_compact.size());
  {   // bus shunts by node (res_bus p/q carry the shunt power, pandapower _get_shunt_results)
    std::vector<double> sh_g(npq + 1), sh_b(npq + 1);
    bool any = false;
    for (int i = 0; i <= npq; ++i) {
      const int b = (i == npq) ? slack : order[i];
      sh_g[i] = gs[b]; sh_b[i] = bs[b];
      any = any || gs[b] != 0.0 || bs[b] != 0.0;
    }
    P.has_shunt = any;
    TRY(dev_upload(e, sh_g, &P.sh_g)); TRY(dev_upload(e, sh_b, &P.sh_b));
  }
  std::vector<int> bus_of_node(order.begin(), order.end());
  TRY(dev_upload(e, hot, &P.hot));
  TRY(dev_upload(e, bus_of_node, &P.bus_of_node));
  TRY(dev_upload(e, lscale, &P.lscale)); TRY(dev_upload(e, sscale, &P.sscale));
  TRY(dev_upload(e, sl_node, &P.sl_node)); TRY(dev_upload(e, sl_y, &P.sl_y));
  {
    const double* d_ysl = nullptr;
    TRY(dev_upload(e, ysl_cold, &d_ysl));
    P.ysl = reinterpret_cast<const double2*>(d_ysl);
    TRY(dev_upload(e, obs_off, &P.obs_off)); TRY(dev_upload(e, line_nodes, &P.line_nodes)); TRY(dev_upload(e, line_c, &P.line_c));
  }
  {
    std::vector<int> sgen_node(ng);
    for (int j = 0; j < ng; ++j) sgen_node[j] = node_of_bus[net->sgen_bus[j]];
    TRY(dev_upload(e, sgen_node, &P.sgen_node));
  }
  TRY(dev_upload(e, state_src, &P.state_src)); TRY(dev_upload(e, obs_src, &P.obs_src)); TRY(dev_upload(e, obs_xptr, &P.obs_xptr)); TRY(dev_upload(e, obs_xidx, &P.obs_xidx));
  const size_t B = static_cast<size_t>(cfg->batch);
  if (prof) {
    const size_t T = static_cast<size_t>(prof->n_rows);
    TRY(dev_upload(e, std::vector<double>(prof->s_max, prof->s_max + ng), &P.s_max));
    TRY(dev_upload(e, std::vector<double>(prof->pv_std, prof->pv_std + ng), &P.pv_std));
    TRY(dev_upload(e, std::vector<double>(prof->load_p_std, prof->load_p_std + nl), &P.lp_std));
    TRY(dev_upload(e, std::vector<double>(prof->load_q_std, prof->load_q_std + nl), &P.lq_std));
    double *dpv, *dlp, *dlq;
    TRY(dev_alloc(e, T * ng, &dpv)); TRY(dev_alloc(e, T * nl, &dlp)); TRY(dev_alloc(e, T * nl, &dlq));
    TRY_CUDA(cudaMemcpy(dpv, prof->pv, T * ng * sizeof(double), cudaMemcpyHostToDevice));
    if (nl) {
      TRY_CUDA(cudaMemcpy(dlp, prof->load_p, T * nl * sizeof(double), cudaMemcpyHostToDevice));
      TRY_CUDA(cudaMemcpy(dlq, prof->load_q, T * nl * sizeof(double), cudaMemcpyHostToDevice));
    }
    P.prof_pv = dpv; P.prof_lp = dlp; P.prof_lq = dlq;
    P.n_rows = prof->n_rows; P.steps_per_hour = prof->steps_per_hour;
    const int episode_days = cfg->episode_limit / (24 * prof->steps_per_hour) + 1;     // reference :397
    P.n_day_choices = prof->n_days - episode_days;                                     // reference :398
    if (P.n_day_choices < 1) return bail(fail(MAPDN_ERR_INVALID, "profile store shorter than one episode"));
    // the latest sampled window must fit: start_max + episode_limit rows
    const long long last = (static_cast<long long>(P.n_day_choices - 1) * 24 + 23) * prof->steps_per_hour +
                           (prof->steps_per_hour - 1) + cfg->episode_limit;
    if (last > prof->n_rows - 1) return bail(fail(MAPDN_ERR_INVALID, "profile store shorter than n_days claims"));
  }
  P.base_mva = net->base_mva; P.inv_base = 1.0 / net->base_mva;
  P.vm_init = (net->vm_init > 0) ? net->vm_init : net->slack_vm;
  P.vm0 = net->slack_vm; P.va0 = net->slack_va_deg * (3.14159265358979323846 / 180.0);
  P.e0 = P.vm0 * std::cos(P.va0); P.f0 = P.vm0 * std::sin(P.va0);
  P.ysl_g0 = e->ydiag[2 * slack]; P.ysl_b0 = e->ydiag[2 * slack + 1];
  P.tol = (cfg->tol > 0) ? cfg->tol : 1e-8;
  P.max_iter = (cfg->max_iter > 0) ? cfg->max_iter : 10;
  {
    // The first Newton iteration starts from the flat start, where S_calc and the Jacobian depend on the network only:
    // factorise J(V0) once, leaf -> root on the elimination forest, with the formulas of the kernel's edge / mismatch pass
    // and elimination step (env_kernel.cuh: nr_solve). Per node six double2: S_calc = (P, Q); M = D'^-1 J[i,parent] rows
    // 0 / 1 (what the back sweep multiplies dx_parent with); D'^-1 rows 0 / 1; J[parent,i] = (a, b).
    std::vector<double> ft(static_cast<size_t>(12) * std::max(1, npq), 0.0);
    if (!meshed) {
      const double* yup = reinterpret_cast<const double*>(hot.data() + hl.yup);
      const double* ydn = reinterpret_cast<const double*>(hot.data() + hl.ydn);
      const double* yii = reinterpret_cast<const double*>(hot.data() + hl.yii);
      // children in a labelling-independent order (first child, second child, then the contiguous extras): the node
      // relabelling of section 2b must not change a single bit of the results
      std::vector<std::vector<int>> kids(npq);
      for (int i = 0; i < npq; ++i) {
        if (kid0[i] != npq) kids[i].push_back(kid0[i]);
        if (kid1[i] != npq) kids[i].push_back(kid1[i]);
        for (int c = 2; c < nchild[i]; ++c) kids[i].push_back(kid1[i] + c - 1);      // extras follow child 1 contiguously
      }
      std::vector<int> topo;                               // parents before children
      for (int i = 0; i < npq; ++i) if (parent[i] < 0) topo.push_back(i);
      for (size_t qh = 0; qh < topo.size(); ++qh) for (int c : kids[topo[qh]]) topo.push_back(c);
      const double vi_x = P.vm_init, vi_y = 0.0;             // every PQ bus
      std::vector<double> upx(npq), upy(npq), dnx(npq), dny(npq), d01x(npq), d01y(npq), d23x(npq), d23y(npq);
      std::vector<double> s00(npq, 0.0), s01(npq, 0.0), s10(npq, 0.0), s11(npq, 0.0);     // Schur update a bus hands to its parent
      for (int i = 0; i < npq; ++i) {                      // edge terms of (i, parent); roots: Y = 0
        const double vp_x = P.vm_init, vp_y = 0.0;
        const double cc = vi_x * vp_x + vi_y * vp_y, ss = vi_y * vp_x - vi_x * vp_y;
        upx[i] = yup[2 * i] * ss - yup[2 * i + 1] * cc; upy[i] = yup[2 * i] * cc + yup[2 * i + 1] * ss;
        dnx[i] = -ydn[2 * i] * ss - ydn[2 * i + 1] * cc; dny[i] = ydn[2 * i] * cc - ydn[2 * i + 1] * ss;
      }
      for (int i = 0; i < npq; ++i) {                      // S_calc and the diagonal blocks
        const double cs0 = vi_x * P.e0 + vi_y * P.f0, sn0 = vi_y * P.e0 - vi_x * P.f0;
        double sa = ysl_cold[2 * i] * sn0 - ysl_cold[2 * i + 1] * cs0 + upx[i];
        double sb = ysl_cold[2 * i] * cs0 + ysl_cold[2 * i + 1] * sn0 + upy[i];
        for (int c : kids[i]) { sa += dnx[c]; sb += dny[c]; }
        const double vv = vi_x * vi_x + vi_y * vi_y;
        const double gv = yii[2 * i] * vv, bv = yii[2 * i + 1] * vv;
        const double Pc = gv + sb, Qc = sa - bv;
        ft[12 * i + 0] = Pc; ft[12 * i + 1] = Qc;
        d01x[i] = -Qc - bv; d01y[i] = Pc + gv; d23x[i] = Pc - gv; d23y[i] = Qc - bv;
      }
      for (size_t k = topo.size(); k-- > 0;) {              // children before parents
        const int i = topo[k];
        for (int c : kids[i]) { d01x[i] -= s00[c]; d01y[i] -= s01[c]; d23x[i] -= s10[c]; d23y[i] -= s11[c]; }
        const double idet = 1.0 / (d01x[i] * d23y[i] - d01y[i] * d23x[i]);
        const double ux = upx[i], uy = upy[i], dx = dnx[i], dy = dny[i];
        const double ma00 = d23y[i] * ux + d01y[i] * uy, ma01 = d23y[i] * uy - d01y[i] * ux;      // adj(D') J[i,parent]
        const double ma10 = -d23x[i] * ux - d01x[i] * uy, ma11 = d01x[i] * ux - d23x[i] * uy;
        ft[12 * i + 2] = ma00 * idet; ft[12 * i + 3] = ma01 * idet; ft[12 * i + 4] = ma10 * idet; ft[12 * i + 5] = ma11 * idet;
        ft[12 * i + 6] = d23y[i] * idet; ft[12 * i + 7] = -d01y[i] * idet;                         // D'^-1
        ft[12 * i + 8] = -d23x[i] * idet; ft[12 * i + 9] = d01x[i] * idet;
        ft[12 * i + 10] = dx; ft[12 * i + 11] = dy;
        s00[i] = (dx * ma00 + dy * ma10) * idet; s01[i] = (dx * ma01 + dy * ma11) * idet;         // J[parent,i] D'^-1 J[i,parent]
        s10[i] = (dx * ma10 - dy * ma00) * idet; s11[i] = (dx * ma11 - dy * ma01) * idet;
      }
    }
    const double* d_ft = nullptr;
    TRY(dev_upload(e, ft, &d_ft));
    P.first_tab = reinterpret_cast<const double2*>(d_ft);
  }
  P.barrier = cfg->barrier; P.voltage_weight = cfg->voltage_weight; P.q_weight = cfg->q_weight;
  P.line_weight = cfg->line_weight; P.use_line_weight = cfg->use_line_weight;
  P.v_upper = cfg->v_upper; P.v_lower = cfg->v_lower; P.episode_limit = cfg->episode_limit;
  P.action_low = cfg->action_low; P.action_high = cfg->action_high; P.reset_action = cfg->reset_action;
  P.seed = cfg->seed; P.env_id_offset = cfg->env_id_offset;
  TRY(dev_alloc(e, B * nl, &P.cur_pl)); TRY(dev_alloc(e, B * nl, &P.cur_ql));
  TRY(dev_alloc(e, B * ng, &P.cur_pv)); TRY(dev_alloc(e, B * ng, &P.cur_q));
  TRY(dev_alloc(e, B * n, &P.res_vm)); TRY(dev_alloc(e, B * n, &P.res_va));
  TRY(dev_alloc(e, B * n, &P.res_p)); TRY(dev_alloc(e, B * n, &P.res_q));
  TRY(dev_alloc(e, B * std::max(1, n_line), &P.res_pl));
  TRY(dev_alloc(e, B, &P.steps)); TRY(dev_alloc(e, B, &P.sum_rewards));
  TRY(dev_alloc(e, B, &P.start_row)); TRY(dev_alloc(e, B, &P.episode)); TRY(dev_alloc(e, B, &P.nr_iters));
  if (meshed) {
    const size_t m = 2 * static_cast<size_t>(npq);
    P.dense_stride = static_cast<int>(m * (m + 1));
    const size_t groups = static_cast<size_t>(e->max_blocks) * e->epb;       // one slice per resident env group
    TRY(dev_alloc(e, groups * P.dense_stride, &P.dense_ws));
  }
  // staging for the *_host entry points
  TRY(dev_alloc(e, B * ng, &e->d_stage_actions)); TRY(dev_alloc(e, B, &e->d_stage_reward)); TRY(dev_alloc(e, B, &e->d_stage_term));
  TRY(dev_alloc(e, B * MAPDN_N_INFO, &e->d_stage_info)); TRY(dev_alloc(e, B * std::max<size_t>(ng * obs_dim, e->compact_row), &e->d_stage_obs));   // compact rows round up to 4 entries

  mapdn_dims& d = e->dims;
  d.batch = cfg->batch; d.n_bus = n; d.n_branch = nbr; d.n_line = n_line; d.n_load = nl; d.n_sgen = ng;
  d.n_agents = ng; d.n_actions = 1; d.obs_dim = obs_dim; d.state_dim = P.state_dim; d.n_info = MAPDN_N_INFO;
  d.lanes_per_env = G; d.envs_per_block = e->epb; d.smem_bytes = e->smem; d.n_levels = n_lev;
  // SURVEY §8d: read p_load,q_load,p_pv,a ; write vm,va ; write obs ; reward+done+11 info
  d.algorithmic_bytes_per_env_step = 8LL * (2 * nl + 2 * ng) + 8LL * 2 * n + 8LL * ng * obs_dim + 8LL * 13;
  (void)max_width;
  // the memsets / uploads above ran on the legacy default stream: order them before any launch of the caller's
  // (possibly non-blocking) streams
  TRY_CUDA(cudaDeviceSynchronize());
  *out = e;
  return MAPDN_OK;
#undef TRY
#undef TRY_CUDA
}

mapdn_status mapdn_get_dims(const mapdn_env* e, mapdn_dims* out) {
  if (!e || !out) return fail(MAPDN_ERR_INVALID, "null argument");
  *out = e->dims;
  return MAPDN_OK;
}

int64_t mapdn_launch_count(const mapdn_env* e) { return e ? e->launches : 0; }

mapdn_status mapdn_reset(mapdn_env* e, const int32_t* start_dhi_dev, const uint8_t* mask_dev, int32_t add_noise,
                         double* obs_dev, double* state_dev, uint8_t* converged_dev, void* stream) {
  if (!e) return fail(MAPDN_ERR_INVALID, "null handle");
  if (!e->base.prof_pv) return fail(MAPDN_ERR_INVALID, "handle was created without a profile store");
  MAPDN_ON_DEVICE(e->device);
  Params p = e->base;
  p.start_dhi = start_dhi_dev; p.mask = mask_dev; p.add_noise = add_noise; p.obs = obs_dev; p.state = state_dev;
  p.reset_ok = converged_dev;
  return launch_env_kernel(e, MODE_RESET, p, static_cast<cudaStream_t>(stream));
}

mapdn_status mapdn_step(mapdn_env* e, const double* actions_dev, int32_t add_noise, double* reward_dev,
                        uint8_t* terminated_dev, double* info_dev, double* obs_dev, void* stream) {
  if (!e || !actions_dev || !reward_dev || !terminated_dev) return fail(MAPDN_ERR_INVALID, "null argument");
  if (!e->base.prof_pv) return fail(MAPDN_ERR_INVALID, "handle was created without a profile store");
  MAPDN_ON_DEVICE(e->device);
  Params p = e->base;
  p.actions = actions_dev; p.add_noise = add_noise; p.reward = reward_dev; p.term = terminated_dev;
  p.info = info_dev; p.obs = obs_dev;
  return launch_env_kernel(e, MODE_STEP, p, static_cast<cudaStream_t>(stream));
}

mapdn_status mapdn_step_host(mapdn_env* e, const double* actions_host, int32_t add_noise, double* reward_host,
                             uint8_t* terminated_host, double* info_host, double* obs_host, void* stream) {
  if (!e || !actions_host || !reward_host || !terminated_host) return fail(MAPDN_ERR_INVALID, "null argument");
  MAPDN_ON_DEVICE(e->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t B = e->dims.batch, ng = e->dims.n_sgen, od = e->dims.obs_dim;
  MAPDN_CUDA(cudaMemcpyAsync(e->d_stage_actions, actions_host, B * ng * sizeof(double), cudaMemcpyHostToDevice, st));
  mapdn_status s = mapdn_step(e, e->d_stage_actions, add_noise, e->d_stage_reward, e->d_stage_term, info_host ? e->d_stage_info : nullptr,
                              obs_host ? e->d_stage_obs : nullptr, stream);
  if (s != MAPDN_OK) return s;
  MAPDN_CUDA(cudaMemcpyAsync(reward_host, e->d_stage_reward, B * sizeof(double), cudaMemcpyDeviceToHost, st));
  MAPDN_CUDA(cudaMemcpyAsync(terminated_host, e->d_stage_term, B, cudaMemcpyDeviceToHost, st));
  if (info_host) MAPDN_CUDA(cudaMemcpyAsync(info_host, e->d_stage_info, B * MAPDN_N_INFO * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (obs_host) MAPDN_CUDA(cudaMemcpyAsync(obs_host, e->d_stage_obs, B * ng * od * sizeof(double), cudaMemcpyDeviceToHost, st));
  MAPDN_CUDA(cudaStreamSynchronize(st));
  return MAPDN_OK;
}

// device alias of a pinned host buffer (unified addressing); verified once per buffer
static mapdn_status pinned_alias(mapdn_env* e, const void* host, void** dev, const char* what) {
  *dev = const_cast<void*>(host);
  if (!host) return MAPDN_OK;
  if (std::find(e->pinned_ok.begin(), e->pinned_ok.end(), host) != e->pinned_ok.end()) return MAPDN_OK;
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, host) != cudaSuccess || at.type != cudaMemoryTypeHost || at.devicePointer != host) {
    cudaGetLastError();
    return fail(MAPDN_ERR_INVALID, std::string(what) + ": not page-locked host memory with unified addressing "
                                   "(cudaHostAlloc / cudaHostRegister it, or use mapdn_step_host)");
  }
  if (e->pinned_ok.size() < 64) e->pinned_ok.push_back(host);
  return MAPDN_OK;
}

mapdn_status mapdn_step_host_pinned(mapdn_env* e, const double* actions_host, int32_t add_noise, double* reward_host,
                                    uint8_t* terminated_host, double* info_host, void* obs_host, int32_t obs_is_f32,
                                    int32_t skip_padding, int32_t sync, void* stream) {
  if (!e || !actions_host || !reward_host || !terminated_host) return fail(MAPDN_ERR_INVALID, "null argument");
  if (!e->base.prof_pv) return fail(MAPDN_ERR_INVALID, "handle was created without a profile store");
  MAPDN_ON_DEVICE(e->device);
  void *a, *r, *t, *i, *o;
  mapdn_status s;
  if ((s = pinned_alias(e, actions_host, &a, "actions_host")) != MAPDN_OK) return s;
  if ((s = pinned_alias(e, reward_host, &r, "reward_host")) != MAPDN_OK) return s;
  if ((s = pinned_alias(e, terminated_host, &t, "terminated_host")) != MAPDN_OK) return s;
  if ((s = pinned_alias(e, info_host, &i, "info_host")) != MAPDN_OK) return s;
  if ((s = pinned_alias(e, obs_host, &o, "obs_host")) != MAPDN_OK) return s;
  Params p = e->base;
  p.actions = static_cast<const double*>(a); p.add_noise = add_noise; p.reward = static_cast<double*>(r);
  p.term = static_cast<unsigned char*>(t); p.info = static_cast<double*>(i);
  p.obs = obs_is_f32 ? nullptr : static_cast<double*>(o);
  p.obs32 = obs_is_f32 ? static_cast<float*>(o) : nullptr;
  p.obs_skip_off = skip_padding ? e->obs_zero_off : -1;
  s = launch_env_kernel(e, MODE_STEP, p, static_cast<cudaStream_t>(stream));
  if (s != MAPDN_OK) return s;
  if (sync) MAPDN_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return MAPDN_OK;
}

mapdn_status mapdn_obs_compact_layout(const mapdn_env* e, int32_t* agent_off, int32_t* agent_len, int32_t* row_len) {
  if (!e) return fail(MAPDN_ERR_INVALID, "null handle");
  for (int a = 0; a < e->dims.n_agents; ++a) {
    if (agent_off) agent_off[a] = e->agent_off[a];
    if (agent_len) agent_len[a] = e->agent_len[a];
  }
  if (row_len) *row_len = e->compact_row;
  return MAPDN_OK;
}

mapdn_status mapdn_step_host_compact(mapdn_env* e, const double* actions_host, int32_t add_noise, double* reward_host,
                                     uint8_t* terminated_host, double* info_host, void* obs_host, int32_t obs_is_f32,
                                     int32_t direct, int32_t sync, void* stream) {
  if (!e || !actions_host || !reward_host || !terminated_host || !obs_host) return fail(MAPDN_ERR_INVALID, "null argument");
  if (!e->base.prof_pv) return fail(MAPDN_ERR_INVALID, "handle was created without a profile store");
  MAPDN_ON_DEVICE(e->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  void *a, *r, *t, *i, *o;
  mapdn_status s;
  if ((s = pinned_alias(e, actions_host, &a, "actions_host")) != MAPDN_OK) return s;
  if ((s = pinned_alias(e, reward_host, &r, "reward_host")) != MAPDN_OK) return s;
  if ((s = pinned_alias(e, terminated_host, &t, "terminated_host")) != MAPDN_OK) return s;
  if ((s = pinned_alias(e, info_host, &i, "info_host")) != MAPDN_OK) return s;
  if ((s = pinned_alias(e, obs_host, &o, "obs_host")) != MAPDN_OK) return s;    // pageable memory would make the copy synchronous
  Params p = e->base;
  p.actions = static_cast<const double*>(a); p.add_noise = add_noise; p.reward = static_cast<double*>(r);
  p.term = static_cast<unsigned char*>(t); p.info = static_cast<double*>(i);
  void* dst = direct ? o : static_cast<void*>(e->d_stage_obs);
  p.obs = obs_is_f32 ? nullptr : static_cast<double*>(dst);
  p.obs32 = obs_is_f32 ? static_cast<float*>(dst) : nullptr;
  p.obs_compact_len = e->compact_row;
  s = launch_env_kernel(e, MODE_STEP, p, st);
  if (s != MAPDN_OK) return s;
  if (!direct) {
    const size_t bytes = static_cast<size_t>(e->dims.batch) * e->compact_row * (obs_is_f32 ? sizeof(float) : sizeof(double));
    MAPDN_CUDA(cudaMemcpyAsync(obs_host, e->d_stage_obs, bytes, cudaMemcpyDeviceToHost, st));
  }
  if (sync) MAPDN_CUDA(cudaStreamSynchronize(st));
  return MAPDN_OK;
}

mapdn_status mapdn_wait(mapdn_env* e, void* stream) {
  if (!e) return fail(MAPDN_ERR_INVALID, "null handle");
  MAPDN_ON_DEVICE(e->device);
  MAPDN_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return MAPDN_OK;
}

mapdn_status mapdn_step_f32obs(mapdn_env* e, const double* actions_dev, int32_t add_noise, double* reward_dev,
                               uint8_t* terminated_dev, double* info_dev, float* obs_dev, void* stream) {
  if (!e || !actions_dev || !reward_dev || !terminated_dev) return fail(MAPDN_ERR_INVALID, "null argument");
  if (!e->base.prof_pv) return fail(MAPDN_ERR_INVALID, "handle was created without a profile store");
  MAPDN_ON_DEVICE(e->device);
  Params p = e->base;
  p.actions = actions_dev; p.add_noise = add_noise; p.reward = reward_dev; p.term = terminated_dev;
  p.info = info_dev; p.obs = nullptr; p.obs32 = obs_dev;
  return launch_env_kernel(e, MODE_STEP, p, static_cast<cudaStream_t>(stream));
}

mapdn_status mapdn_step_host_f32obs(mapdn_env* e, const double* actions_host, int32_t add_noise, double* reward_host,
                                    uint8_t* terminated_host, double* info_host, float* obs_host, void* stream) {
  if (!e || !actions_host || !reward_host || !terminated_host) return fail(MAPDN_ERR_INVALID, "null argument");
  MAPDN_ON_DEVICE(e->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t B = e->dims.batch, ng = e->dims.n_sgen, od = e->dims.obs_dim;
  float* d_obs32 = reinterpret_cast<float*>(e->d_stage_obs);          // the fp64 staging buffer is large enough
  MAPDN_CUDA(cudaMemcpyAsync(e->d_stage_actions, actions_host, B * ng * sizeof(double), cudaMemcpyHostToDevice, st));
  mapdn_status s = mapdn_step_f32obs(e, e->d_stage_actions, add_noise, e->d_stage_reward, e->d_stage_term,
                                     info_host ? e->d_stage_info : nullptr, obs_host ? d_obs32 : nullptr, stream);
  if (s != MAPDN_OK) return s;
  MAPDN_CUDA(cudaMemcpyAsync(reward_host, e->d_stage_reward, B * sizeof(double), cudaMemcpyDeviceToHost, st));
  MAPDN_CUDA(cudaMemcpyAsync(terminated_host, e->d_stage_term, B, cudaMemcpyDeviceToHost, st));
  if (info_host) MAPDN_CUDA(cudaMemcpyAsync(info_host, e->d_stage_info, B * MAPDN_N_INFO * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (obs_host) MAPDN_CUDA(cudaMemcpyAsync(obs_host, d_obs32, B * ng * od * sizeof(float), cudaMemcpyDeviceToHost, st));
  MAPDN_CUDA(cudaStreamSynchronize(st));
  return MAPDN_OK;
}

mapdn_status mapdn_get_obs(mapdn_env* e, double* obs_dev, void* stream) {
  if (!e || !obs_dev) return fail(MAPDN_ERR_INVALID, "null argument");
  MAPDN_ON_DEVICE(e->device);
  Params p = e->base;
  p.obs = obs_dev;
  const long long tot = static_cast<long long>(p.nb) * p.n_sgen * p.obs_dim;
  MAPDN_LAUNCH(get_obs_kernel, static_cast<unsigned>((tot + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), p);
  MAPDN_CUDA(cudaGetLastError());
  e->launches++;
  return MAPDN_OK;
}

mapdn_status mapdn_get_state(mapdn_env* e, double* state_dev, void* stream) {
  if (!e || !state_dev) return fail(MAPDN_ERR_INVALID, "null argument");
  MAPDN_ON_DEVICE(e->device);
  Params p = e->base;
  p.state = state_dev;
  const long long tot = static_cast<long long>(p.nb) * p.state_dim;
  MAPDN_LAUNCH(get_state_kernel, static_cast<unsigned>((tot + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), p);
  MAPDN_CUDA(cudaGetLastError());
  e->launches++;
  return MAPDN_OK;
}

mapdn_status mapdn_get_field(mapdn_env* e, int32_t field, double* out_dev, void* stream) {
  if (!e || !out_dev) return fail(MAPDN_ERR_INVALID, "null argument");
  MAPDN_ON_DEVICE(e->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Params& p = e->base;
  const long long B = p.nb;
  const double* src = nullptr;
  long long cnt = 0;
  double scale = 1.0;
  switch (field) {
    case MAPDN_FIELD_VM: src = p.res_vm; cnt = B * p.n_bus; break;
    case MAPDN_FIELD_VA_DEG: src = p.res_va; cnt = B * p.n_bus; scale = 57.295779513082320876798; break;
    case MAPDN_FIELD_P_BUS: src = p.res_p; cnt = B * p.n_bus; break;
    case MAPDN_FIELD_Q_BUS: src = p.res_q; cnt = B * p.n_bus; break;
    case MAPDN_FIELD_P_SGEN: src = p.cur_pv; cnt = B * p.n_sgen; break;
    case MAPDN_FIELD_Q_SGEN: src = p.cur_q; cnt = B * p.n_sgen; break;
    case MAPDN_FIELD_LINE_LOSS: src = p.res_pl; cnt = B * p.n_line; break;
    case MAPDN_FIELD_P_LOAD: src = p.cur_pl; cnt = B * p.n_load; break;
    case MAPDN_FIELD_Q_LOAD: src = p.cur_ql; cnt = B * p.n_load; break;
    case MAPDN_FIELD_SUM_REWARDS: src = p.sum_rewards; cnt = B; break;
    case MAPDN_FIELD_STEPS:
      MAPDN_LAUNCH(int_to_double_kernel, static_cast<unsigned>((B + 255) / 256), 256, 0, st, B, p.steps, out_dev);
      MAPDN_CUDA(cudaGetLastError()); e->launches++;
      return MAPDN_OK;
    case MAPDN_FIELD_NR_ITERS:
      MAPDN_LAUNCH(int_to_double_kernel, static_cast<unsigned>((B + 255) / 256), 256, 0, st, B, p.nr_iters, out_dev);
      MAPDN_CUDA(cudaGetLastError()); e->launches++;
      return MAPDN_OK;
    case MAPDN_FIELD_START_ROW:
      MAPDN_LAUNCH(i64_to_double_kernel, static_cast<unsigned>((B + 255) / 256), 256, 0, st, B, p.start_row, out_dev);
      MAPDN_CUDA(cudaGetLastError()); e->launches++;
      return MAPDN_OK;
    default: return fail(MAPDN_ERR_INVALID, "unknown field");
  }
  if (cnt == 0) return MAPDN_OK;
  MAPDN_LAUNCH(scale_copy_kernel, static_cast<unsigned>((cnt + 255) / 256), 256, 0, st, cnt, src, scale, out_dev);
  MAPDN_CUDA(cudaGetLastError());
  e->launches++;
  return MAPDN_OK;
}

mapdn_status mapdn_solve(mapdn_env* e, int32_t nb, const double* p_load, const double* q_load, const double* p_sgen,
                         const double* q_sgen, double* vm, double* va_deg, double* p_bus, double* q_bus, double* pl,
                         int32_t* iters, uint8_t* converged, void* stream) {
  if (!e || nb < 1 || !p_sgen || !q_sgen || (e->dims.n_load > 0 && (!p_load || !q_load)))
    return fail(MAPDN_ERR_INVALID, "null argument");
  MAPDN_ON_DEVICE(e->device);
  Params p = e->base;
  p.nb = nb;
  p.in_pl = p_load; p.in_ql = q_load; p.in_pv = p_sgen; p.in_q = q_sgen;
  p.out_vm = vm; p.out_va = va_deg; p.out_p = p_bus; p.out_q = q_bus; p.out_pl = pl;
  p.out_iters = iters; p.out_conv = converged;
  return launch_env_kernel(e, MODE_SOLVE, p, static_cast<cudaStream_t>(stream));
}

mapdn_status mapdn_droop(mapdn_env* e, int32_t nb, const double* p_load, const double* q_load, const double* p_sgen,
                         const double* s_rated, const double* q_max_manual, double gain, double tol, int32_t max_ite,
                         double* vm, double* q_sgen, double* loss, int32_t* iterations, void* stream) {
  if (!e || nb < 1 || !p_sgen || !s_rated || !q_max_manual || !q_sgen || !loss || !iterations ||
      (e->dims.n_load > 0 && (!p_load || !q_load)))
    return fail(MAPDN_ERR_INVALID, "null argument");
  if (max_ite < 1 || !(gain > 0.0)) return fail(MAPDN_ERR_INVALID, "droop: need max_ite >= 1 and gain > 0");
  MAPDN_ON_DEVICE(e->device);
  Params p = e->base;
  p.nb = nb;
  p.in_pl = p_load; p.in_ql = q_load; p.in_pv = p_sgen; p.in_q = nullptr;
  p.droop_s = s_rated; p.droop_qmm = q_max_manual; p.droop_gain = gain; p.droop_tol = tol; p.droop_max_ite = max_ite;
  p.out_vm = vm; p.out_va = nullptr; p.out_p = nullptr; p.out_q = nullptr; p.out_pl = nullptr;
  p.out_iters = iterations; p.out_conv = nullptr; p.droop_q_out = q_sgen; p.droop_loss_out = loss;
  return launch_env_kernel(e, MODE_DROOP, p, static_cast<cudaStream_t>(stream));
}

mapdn_status mapdn_get_ybus_dense(mapdn_env* e, double* g_host, double* b_host) {
  if (!e || !g_host || !b_host) return fail(MAPDN_ERR_INVALID, "null argument");
  const int n = e->dims.n_bus;
  std::fill(g_host, g_host + static_cast<size_t>(n) * n, 0.0);
  std::fill(b_host, b_host + static_cast<size_t>(n) * n, 0.0);
  for (int i = 0; i < n; ++i) { g_host[static_cast<size_t>(i) * n + i] = e->ydiag[2 * i]; b_host[static_cast<size_t>(i) * n + i] = e->ydiag[2 * i + 1]; }
  for (size_t k = 0; k < e->br_from.size(); ++k) {
    const size_t f = e->br_from[k], t = e->br_to[k];
    g_host[f * n + t] += e->ybr[8 * k + 2]; b_host[f * n + t] += e->ybr[8 * k + 3];
    g_host[t * n + f] += e->ybr[8 * k + 4]; b_host[t * n + f] += e->ybr[8 * k + 5];
  }
  return MAPDN_OK;
}

}  // extern "C"
