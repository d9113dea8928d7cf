// mpc_capi.cu -- the C-ABI of include/mpc_b200.h on top of the sm_100a kernel.
//
// Boundary it replaces: MPC::MPC / MPC::solve (/root/reference/src/control/MPC.cpp:160-325) and
// Config::load (/root/reference/src/utils/Config.cpp:31-87).  No CPU fallback: every compute entry
// point fails with MPC_ENODEV / MPC_ECUDA when the device or the launch is unavailable.
#include "../../include/mpc_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <type_traits>
#include <vector>

#include "mpc_kernel.cuh"
#include "mpc_lane_kernel.cuh"
#include "mpc_rollout.cuh"
#include "mpc_sensitivity.cuh"
#include "mpc_run_logic.h"

using namespace mpcb200;

static thread_local char g_err[512] = "";

static int cuda_fail(cudaError_t e, const char *what) {
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return MPC_ECUDA;
}
#define CK(call)                                      \
  do {                                                \
    cudaError_t e__ = (call);                         \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

// device counters of a handle: [0] work queue, [1 + 2k] records parked by launch k of a lane-kernel chain,
// [2 + 2k] cursor of the coop kernel over them, [MPC_HIST0 ..] horizon histogram of a ragged batch
// [MPC_RESTART_COUNT] problems handed to the final launch without a record, [MPC_RESTART_CURSOR] its cursor over them
enum { MPC_MAX_PHASES = 6, MPC_RESTART_COUNT = 17, MPC_RESTART_CURSOR = 18, MPC_HIST0 = 20, MPC_NCOUNTER = MPC_HIST0 + MPC_NMAX + 1 };

// a kernel whose attributes a handle has set, and its CTAs per SM (coop family; 0 for the lane kernel).  Room for every
// instantiation: 4 horizons x (coop, finisher, lane kernel: cold and warm; rollout).
struct KernelAttr { const void *fn; int per_sm; };
enum { MPC_NKERNELS = 28 };

struct mpc_handle {
  mpc_config cfg;
  int device;
  int sm_count;
  int *d_counter;
  long long launches;
  int kernel_kind;      // MPC_KERNEL_AUTO / LANE / COOP
  int lane_threads;     // threads per CTA of the lane kernel
  int lane_ctas_per_sm; // CTAs per SM of the lane kernel (0 = occupancy maximum)
  int handoff_iter;     // rule 1: lane kernel parks problems still running after this many iterations (0 = never, the default)
  int park_lanes;       // tail packing: a warp with at most this many problems left parks them once the queue is empty (0 = off)
  int resume_phases;    // lane-kernel resume launches between the main launch and the final one
  int resume_min;       // a resume launch with no more than this many records to work on leaves them to the next launch
  // early copy-back (mpc_solve_batch_host): the device->host copies of a lane-kernel chain start before its final launch
  cudaStream_t stream2;
  cudaEvent_t ev_pre, ev_copy;
  bool no_early_copy;   // test switch: always copy back after the last launch
  double *d_ckpt;       // migration records, two buffers of cap_ckpt records (each launch of a chain reads one, writes the other)
  size_t cap_ckpt;      // records per buffer
  int ckpt_ns;
  bool sort_ragged;     // ragged batches (N_per given): hand the problems out longest horizon first
  int rollout_mode;     // MPC_ROLLOUT_AUTO / PER_STEP / PERSISTENT
  int *d_restart;       // indices of the problems the lane kernel handed over without a record
  size_t cap_restart;
  double *d_scratch;    // coop kernels: global scratch per lane group (watchdog backup, restoration rows)
  size_t cap_scratch;
  int *d_perm;          // ragged batches: problem order of the work queue (longest horizon first)
  size_t cap_perm;
  double *dual_lam, *dual_zl, *dual_zu;   // caller's device buffers for the multipliers (or NULL)
  const double *ws_x, *ws_lam, *ws_zl, *ws_zu;   // caller's device buffers of a warm start (ws_x NULL: cold start)
  double ws_mu;                                  // its initial barrier parameter
  // mpc_set_warm_start_one: mpc_solve_one keeps its last solution (x, lambda, zl, zu) in d_one and starts from it shifted
  bool one_warm, one_prev_ok;
  double one_mu;
  double *d_one;        // [2][x 8N-2 | lambda 6N | zl 8N-2 | zu 8N-2]: the last solution, the next start point
  int one_N;
  // staging buffers for the host-pointer entry points (grown on demand)
  double *d_in, *d_out;
  int *d_iout;
  double *h_pin;       // pinned host mirror for mpc_solve_one
  size_t cap_B;
  int cap_N;
  bool cap_w;
  double *d_run;        // device workspace of the run()/rollout entry points
  int *d_run_i;
  size_t cap_run;
  cudaStream_t stream;
  KernelAttr attr[MPC_NKERNELS];   // one device and one call in flight per handle: no lock
  int n_attr;
};

// ------------------------------------------------------------------------------------------------
// minimal JSON reader (objects, arrays, numbers, strings, true/false/null): enough for the
// config-*.json files Config::load reads (Config.cpp:34-35)
// ------------------------------------------------------------------------------------------------
namespace {
struct JVal {
  enum { NUL, NUM, STR, ARR, OBJ, BOOL } t = NUL;
  double num = 0;
  std::string str;
  std::vector<JVal> arr;
  std::map<std::string, JVal> obj;
};
struct JParser {
  const char *p;
  bool ok = true;
  explicit JParser(const char *s) : p(s) {}
  void ws() { while (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r') p++; }
  bool lit(const char *s) { size_t n = strlen(s); if (strncmp(p, s, n) == 0) { p += n; return true; } return false; }
  std::string str() {
    std::string out;
    if (*p != '"') { ok = false; return out; }
    p++;
    while (*p && *p != '"') {
      if (*p == '\\' && p[1]) { p++; char c = *p; out += (c == 'n' ? '\n' : c == 't' ? '\t' : c); }
      else out += *p;
      p++;
    }
    if (*p != '"') ok = false; else p++;
    return out;
  }
  JVal val() {
    JVal v;
    ws();
    if (*p == '{') {
      v.t = JVal::OBJ; p++; ws();
      if (*p == '}') { p++; return v; }
      while (ok) {
        ws(); std::string k = str(); ws();
        if (*p != ':') { ok = false; break; }
        p++;
        v.obj[k] = val(); ws();
        if (*p == ',') { p++; continue; }
        if (*p == '}') { p++; break; }
        ok = false;
      }
    } else if (*p == '[') {
      v.t = JVal::ARR; p++; ws();
      if (*p == ']') { p++; return v; }
      while (ok) {
        v.arr.push_back(val()); ws();
        if (*p == ',') { p++; continue; }
        if (*p == ']') { p++; break; }
        ok = false;
      }
    } else if (*p == '"') {
      v.t = JVal::STR; v.str = str();
    } else if (lit("true")) { v.t = JVal::BOOL; v.num = 1;
    } else if (lit("false")) { v.t = JVal::BOOL; v.num = 0;
    } else if (lit("null")) { v.t = JVal::NUL;
    } else {
      char *end = nullptr;
      v.num = strtod(p, &end);
      if (end == p) ok = false; else { v.t = JVal::NUM; p = end; }
    }
    return v;
  }
};
inline double mph2mps(double mph) { return mph * 1609.34 / 3600.0; }   // utils.h:11-13
inline double deg2rad(double x) { return x * M_PI / 180; }             // utils.h:69
}  // namespace

extern "C" int mpc_config_defaults(mpc_config *c) {
  if (!c) return MPC_EINVAL;
  memset(c, 0, sizeof(*c));
  // Config.cpp:5-29
  c->N = 25;
  c->max_fit_order = 4;
  c->max_fit_error = 0.5;
  c->latency_ms = 100;
  c->lookahead = 0;
  c->ipopt_timeout = 0.5;
  c->dt = 0.025;
  c->max_steering = deg2rad(25.0);
  c->max_accel = mph2mps(8);
  c->max_decel = mph2mps(-20);
  c->max_speed = mph2mps(100);
  c->Lf = 2.67;
  c->epsi_panic = 1;
  c->cte_panic = 0.6;
  c->steer_adjust_thresh = 0.6;
  c->steer_adjust_ratio = 0.025;
  const double w[8] = {100, 100, 1, 1, 1, 5000, 1, 1000};
  for (int i = 0; i < 8; i++) c->weights[i] = w[i];
  c->n_steers = 3;
  c->steers[0] = 0.1; c->steers[1] = 0.2; c->steers[2] = 0.3;
  c->n_steer_speeds = 4;
  c->steer_speeds[0] = mph2mps(80); c->steer_speeds[1] = mph2mps(65);
  c->steer_speeds[2] = mph2mps(30); c->steer_speeds[3] = mph2mps(25);
  c->max_iter = 3000;
  c->tol = 1e-8;
  c->watchdog_trigger = 10;
  c->filter_reset_trigger = 5;
  c->tiny_step_tol = 10.0 * 2.220446049250313e-16;
  return MPC_OK;
}

extern "C" int mpc_config_parse_json(const char *text, mpc_config *c) {
  if (!text || !c) return MPC_EINVAL;
  JParser jp(text);
  JVal js = jp.val();
  if (!jp.ok || js.t != JVal::OBJ) return MPC_EPARSE;
  auto has = [&](const char *k) { return js.obj.count(k) && js.obj[k].t != JVal::NUL; };
  auto num = [&](const char *k, double &out) { if (!has(k) || js.obj[k].t != JVal::NUM) return false; out = js.obj[k].num; return true; };
  auto arr = [&](const char *k, std::vector<double> &out) {
    if (!has(k) || js.obj[k].t != JVal::ARR) return false;
    out.clear();
    for (auto &e : js.obj[k].arr) { if (e.t != JVal::NUM) return false; out.push_back(e.num); }
    return true;
  };
  mpc_config_defaults(c);
  double v;
  // same keys, same order and conversions as Config.cpp:39-86
  if (!num("N", v)) return MPC_EPARSE; c->N = (int)v;
  if (!num("dt", c->dt)) return MPC_EPARSE;
  if (!num("max acceleration", v)) return MPC_EPARSE; c->max_accel = mph2mps(v);
  if (!num("max deceleration", v)) return MPC_EPARSE; c->max_decel = mph2mps(v);
  if (!num("max steering", v)) return MPC_EPARSE; c->max_steering = deg2rad(v);
  if (!num("max speed", v)) return MPC_EPARSE; c->max_speed = mph2mps(v);
  const double speed_scale = c->max_speed / mph2mps(100.0);
  if (!num("latency", v)) return MPC_EPARSE; c->latency_ms = (int)v;
  c->lookahead = c->latency_ms * 1.0E-3;
  if (!num("max polynomial fitting order", v)) return MPC_EPARSE; c->max_fit_order = (int)v;
  if (!num("max polynomial fitting error", c->max_fit_error)) return MPC_EPARSE;
  if (!num("ipopt timeout", c->ipopt_timeout)) return MPC_EPARSE;
  if (!num("Lf", c->Lf)) return MPC_EPARSE;
  if (!num("epsi panic", c->epsi_panic)) return MPC_EPARSE;
  if (!num("cte panic", c->cte_panic)) return MPC_EPARSE;
  if (!num("steer adjustment threshold", c->steer_adjust_thresh)) return MPC_EPARSE;
  if (!num("steer adjustment ratio", v)) return MPC_EPARSE;
  c->steer_adjust_ratio = v < 0.0 ? 0.0 : (v > 0.1 ? 0.1 : v);
  std::vector<double> a;
  if (!arr("weights", a) || a.size() <= 11) return MPC_EPARSE;   // assert(w.size() > WEIGHT_LARGE_CTE)
  for (int i = 0; i < MPC_NWEIGHTS; i++) c->weights[i] = a[i];
  if (!arr("steers", a) || a.size() > MPC_NTAB) return MPC_EPARSE;
  c->n_steers = (int)a.size();
  for (size_t i = 0; i < a.size(); i++) c->steers[i] = a[i];
  auto conv = [&](double s) { return speed_scale <= 1 ? std::fmin(mph2mps(s), c->max_speed) : mph2mps(s) * speed_scale; };
  if (!arr("steer speeds", a) || a.empty() || a.size() > MPC_NTAB) return MPC_EPARSE;
  c->n_steer_speeds = (int)a.size();
  for (size_t i = 0; i < a.size(); i++) c->steer_speeds[i] = conv(a[i]);
  if (!arr("yaw changes", a) || a.size() > MPC_NTAB) return MPC_EPARSE;
  c->n_yaw_changes = (int)a.size();
  for (size_t i = 0; i < a.size(); i++) c->yaw_changes[i] = a[i];
  if (!arr("yaw change speeds", a) || a.size() > MPC_NTAB) return MPC_EPARSE;
  c->n_yaw_change_speeds = (int)a.size();
  for (size_t i = 0; i < a.size(); i++) c->yaw_change_speeds[i] = conv(a[i]);
  return MPC_OK;
}

extern "C" int mpc_config_load_json(const char *path, mpc_config *c) {
  if (!path || !c) return MPC_EINVAL;
  FILE *f = fopen(path, "rb");
  if (!f) return MPC_EIO;
  std::string text;
  char buf[4096];
  size_t n;
  while ((n = fread(buf, 1, sizeof(buf), f)) > 0) text.append(buf, n);
  fclose(f);
  return mpc_config_parse_json(text.c_str(), c);
}

// The command line of the reference's controller (src/mpc_main.cpp:55-79) and what it does to the loaded
// configuration on connection (mpc_main.cpp:238-246).
extern "C" int mpc_config_from_cli(int argc, const char *const *argv, const char *config_dir, mpc_config *cfg,
                                   char *config_file_out, int config_file_cap) {
  if (!cfg || argc < 0 || (argc > 0 && !argv)) return MPC_EINVAL;
  std::string dir = config_dir ? config_dir : "..";
  std::string file = dir + "/config-stable.json";          // mpc_main.cpp:47
  double max_speed = -1;
  int latency = -1;
  for (int i = 0; i < argc; i++) {
    const std::string a = argv[i] ? argv[i] : "";
    if (a == "-config") {
      if (++i >= argc) return MPC_EINVAL;
      file = argv[i];
    } else if (a == "-speed") {
      if (++i >= argc || sscanf(argv[i], "%lf", &max_speed) != 1) return MPC_EINVAL;
    } else if (a == "-latency") {
      if (++i >= argc || sscanf(argv[i], "%d", &latency) != 1) return MPC_EINVAL;
      if (!latency) file = dir + "/config-no-latency.json";
    } else if (a == "-fast") {
      file = dir + "/config-fast.json";
    } else if (a == "-stable") {
      file = dir + "/config-stable.json";
    } else {
      return MPC_EINVAL;                                   // "Unknown option", exit(-1) in the reference
    }
  }
  if (config_file_out && config_file_cap > 0) snprintf(config_file_out, (size_t)config_file_cap, "%s", file.c_str());
  int rc = mpc_config_load_json(file.c_str(), cfg);
  if (rc) return rc;
  if (latency >= 0) cfg->latency_ms = latency;             // Config::lookahead keeps the file's value, as in the reference
  if (max_speed > 0) cfg->max_speed = mph2mps(max_speed);  // the speed tables are NOT rescaled (mpc_main.cpp:244-246)
  return MPC_OK;
}

static int check_config(const mpc_config *c) {
  if (!c) return MPC_EINVAL;
  if (c->N < 2 || c->N > MPC_NMAX) return MPC_EINVAL;
  if (c->n_steers < 0 || c->n_steers > MPC_NTAB || c->n_steer_speeds < 1 || c->n_steer_speeds > MPC_NTAB) return MPC_EINVAL;
  if (!(c->dt > 0) || !(c->Lf > 0) || c->max_iter < 0 || !(c->tol > 0)) return MPC_EINVAL;
  // the run()-level tables index fixed-size arrays on the device: keep the counts inside them
  if (c->n_yaw_changes < 0 || c->n_yaw_changes > MPC_NTAB || c->n_yaw_change_speeds < 0 || c->n_yaw_change_speeds > MPC_NTAB) return MPC_EINVAL;
  if (c->watchdog_trigger < 0 || c->filter_reset_trigger < 1 || !(c->tiny_step_tol >= 0)) return MPC_EINVAL;
  return MPC_OK;
}
// what the MPC::run-level entry points need on top: a speed-limit table to read (the reference calls .back() on an
// empty vector there, Vehicle.cpp:66-79 -- undefined behaviour; here it is an argument error) and a fit order that
// fits MPC_NCOEF coefficients
static int check_run_config(const mpc_config *c) {
  if (c->n_yaw_change_speeds < 1 || c->max_fit_order < 3 || c->max_fit_order > MPC_NCOEF) return MPC_EINVAL;
  return MPC_OK;
}

extern "C" int mpc_create(const mpc_config *cfg, int device, mpc_handle **out) {
  if (!out) return MPC_EINVAL;
  *out = nullptr;
  int rc = check_config(cfg);
  if (rc) return rc;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    snprintf(g_err, sizeof(g_err), "no CUDA device: %s", cudaGetErrorString(e));
    (void)cudaGetLastError();
    return MPC_ENODEV;
  }
  if (device < 0 || device >= ndev) return MPC_ENODEV;
  CK(cudaSetDevice(device));
  mpc_handle *h = new (std::nothrow) mpc_handle();
  if (!h) return MPC_ENOMEM;
  memset(h, 0, sizeof(*h));
  h->cfg = *cfg;
  h->device = device;
  cudaDeviceProp prop;
  cudaError_t ce = cudaGetDeviceProperties(&prop, device);
  h->sm_count = prop.multiProcessorCount;
  // work-queue counter, per launch of a chain: records written / taken; horizon histogram
  if (ce == cudaSuccess) ce = cudaMalloc(&h->d_counter, MPC_NCOUNTER * sizeof(int));
  if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (ce != cudaSuccess) { mpc_destroy(h); return cuda_fail(ce, "mpc_create"); }
  h->kernel_kind = MPC_KERNEL_AUTO;
  h->lane_threads = 0;
  h->lane_ctas_per_sm = 0;
  h->handoff_iter = 0;
  h->sort_ragged = true;
  h->park_lanes = MPC_PARK_LANES_DEFAULT;
  h->resume_phases = MPC_RESUME_PHASES_DEFAULT;
  h->resume_min = MPC_RESUME_MIN_DEFAULT;
  *out = h;
  return MPC_OK;
}

extern "C" void mpc_destroy(mpc_handle *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->d_counter);
  cudaFree(h->d_ckpt);
  cudaFree(h->d_perm);
  cudaFree(h->d_restart);
  cudaFree(h->d_scratch);
  cudaFree(h->d_in);
  cudaFree(h->d_out);
  cudaFree(h->d_iout);
  cudaFreeHost(h->h_pin);
  cudaFree(h->d_run);
  cudaFree(h->d_run_i);
  cudaFree(h->d_one);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->stream2) cudaStreamDestroy(h->stream2);
  if (h->ev_pre) cudaEventDestroy(h->ev_pre);
  if (h->ev_copy) cudaEventDestroy(h->ev_copy);
  delete h;
}

extern "C" int mpc_set_config(mpc_handle *h, const mpc_config *cfg) {
  if (!h) return MPC_EINVAL;
  int rc = check_config(cfg);
  if (rc) return rc;
  h->cfg = *cfg;
  h->one_prev_ok = false;   // a solution of another problem definition is no start point
  return MPC_OK;
}

// The lane kernel keeps everything in registers and thread-private memory: no shared memory, so
// the whole unified L1 is cache for the per-stage arrays.  One CTA per SM (its warps run the slots of a
// trip in step), sized so that every lane gets the same number of problems: with
// r = ceil(B / (SMs * 256)) problems per lane, ceil(B / (SMs * r)) lanes per SM -- otherwise the lanes
// without a last problem idle through the final round while their warps still issue every instruction.
// ---- ragged batches: hand the problems out longest horizon first.  Lanes of a warp fetch neighbouring queue
// entries, so they hold horizons of similar length (every sweep of a warp runs to the longest N among its lanes),
// and the longest problems start first.  Counting sort by N: histogram, descending exclusive scan, scatter.
__global__ void mpc_horizon_hist_kernel(const int *N_pp, int B, int *hist) {
  __shared__ int sh[MPC_NMAX + 1];
  for (int k = threadIdx.x; k <= MPC_NMAX; k += blockDim.x) sh[k] = 0;
  __syncthreads();
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    int n = N_pp[b];
    n = n < 0 ? 0 : (n > MPC_NMAX ? MPC_NMAX : n);
    atomicAdd(&sh[n], 1);
  }
  __syncthreads();
  for (int k = threadIdx.x; k <= MPC_NMAX; k += blockDim.x) if (sh[k]) atomicAdd(&hist[k], sh[k]);
}
__global__ void mpc_horizon_scan_kernel(int *hist) {
  int acc = 0;
  for (int k = MPC_NMAX; k >= 0; k--) { const int c = hist[k]; hist[k] = acc; acc += c; }
}
__global__ void mpc_horizon_scatter_kernel(const int *N_pp, int B, int *cursor, int *perm) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    int n = N_pp[b];
    n = n < 0 ? 0 : (n > MPC_NMAX ? MPC_NMAX : n);
    perm[atomicAdd(&cursor[n], 1)] = b;
  }
}

// Global scratch of the coop kernels (one block per resident lane group) and the restart list of a chain.
template <int NS>
static int ensure_coop_scratch(mpc_handle *h, KParams &kp, long long groups_total) {
  const size_t per = (size_t)Lane<NS, true>::SC_SIZE;
  const size_t need = per * (size_t)groups_total;
  if (!h->d_scratch || h->cap_scratch < need) {
    cudaFree(h->d_scratch);
    h->d_scratch = nullptr; h->cap_scratch = 0;
    CK(cudaMalloc(&h->d_scratch, need * sizeof(double)));
    h->cap_scratch = need;
  }
  kp.scratch = h->d_scratch; kp.scratch_stride = (long long)per;
  return MPC_OK;
}
static int ensure_restart(mpc_handle *h, KParams &kp) {
  if (!h->d_restart || h->cap_restart < (size_t)kp.B) {
    cudaFree(h->d_restart);
    h->d_restart = nullptr; h->cap_restart = 0;
    CK(cudaMalloc(&h->d_restart, (size_t)kp.B * sizeof(int)));
    h->cap_restart = kp.B;
  }
  kp.restart_list = h->d_restart;
  kp.restart_count = h->d_counter + MPC_RESTART_COUNT;
  kp.restart_cursor = h->d_counter + MPC_RESTART_CURSOR;
  return MPC_OK;
}

// Calls f(std::integral_constant<int, NS>()) with the horizon capacity NS of the kernels that solve horizon N.
template <class F>
static int with_horizon(int N, F f) {
  if (N <= 10) return f(std::integral_constant<int, 10>());
#ifndef MPC_DEV_N10
  if (N <= 20) return f(std::integral_constant<int, 20>());
  if (N <= 32) return f(std::integral_constant<int, 32>());
  return f(std::integral_constant<int, MPC_NMAX>());
#else
  return MPC_EINVAL;   // development build (-DMPC_DEV_N10, a third of the compile time): N <= 10 only
#endif
}

// Sets the attributes of kernel `fn` through set(&per_sm) the first time this handle launches it; *per_sm: its CTAs
// per SM, as `set` stored it.
template <class Set>
static int kernel_attrs(mpc_handle *h, const void *fn, int *per_sm, Set set) {
  for (int i = 0; i < h->n_attr; i++)
    if (h->attr[i].fn == fn) { *per_sm = h->attr[i].per_sm; return MPC_OK; }
  const int rc = set(per_sm);
  if (rc) return rc;
  if (h->n_attr < MPC_NKERNELS) h->attr[h->n_attr++] = {fn, *per_sm};
  return MPC_OK;
}

// The coop-family kernels (mpc_coop_kernel, mpc_coop_resume_kernel, mpc_rollout_kernel): one problem per group of 16
// or 32 lanes, per-stage rows in shared memory, CTAs of 128 threads -- as many as fit on the SMs, but no more groups
// than `work` problems -- and a block of global scratch per group.
template <int NS, class Kernel, class... Args>
static int launch_coop_family(mpc_handle *h, Kernel kernel, const char *name, KParams &kp, long long work,
                              cudaStream_t st, const Args &...args) {
  const int threads = 128, groups = threads / (NS <= 16 ? 16 : 32);
  const size_t smem = (size_t)groups * NS * ST_ROW_SH * sizeof(double);
  int per_sm = 0;
  int rc = kernel_attrs(h, (const void *)kernel, &per_sm, [&](int *n) {
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, kernel, threads, smem));
    return MPC_OK;
  });
  if (rc) return rc;
  if (per_sm < 1) { snprintf(g_err, sizeof(g_err), "%s does not fit on an SM (smem %zu)", name, smem); return MPC_ECUDA; }
  long long want = (work + groups - 1) / groups, grid = (long long)h->sm_count * per_sm;
  if (grid > want) grid = want;
  if (grid < 1) grid = 1;
  rc = ensure_coop_scratch<NS>(h, kp, grid * groups);
  if (rc) return rc;
  kernel<<<(unsigned)grid, threads, smem, st>>>(kp, args...);
  CK(cudaGetLastError());
  h->launches++;
  return MPC_OK;
}

// What the early copy-back of mpc_solve_batch_host needs from a lane-kernel chain: whether h->ev_pre was recorded
// before the chain's final launch, and that launch's parameters (its record list = the outputs still to come), record
// size and offset of the problem index in a record.
struct PreFinisher {
  bool recorded;
  KParams kp;
  int rec, cki;
};

// The lane kernel and the launches that finish its tail, all on one stream with no host round trip:
//   main launch            fresh problems from the work queue; parks by rule 1 (iterations) and rule 2 (sparse warp)
//   resume launches        the parked problems, 32 to a warp; park by rule 2 into the other buffer
//   final launch           the coop kernel (one problem per lane group, rows in shared memory, every branch of the
//                          algorithm): the records that are left, then the problems handed over without a record
// pre: NULL, or where to report the event recorded before the final launch.
template <int NS, bool WARM>
static int launch_lane(mpc_handle *h, KParams &kp, cudaStream_t st, PreFinisher *pre) {
  int unused;
  int rc = kernel_attrs(h, (const void *)mpc_lane_kernel<NS, false, WARM>, &unused, [&](int *per_sm) {
    CK(cudaFuncSetAttribute(mpc_lane_kernel<NS, false, WARM>, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
    CK(cudaFuncSetAttribute(mpc_lane_kernel<NS, true, WARM>, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
    *per_sm = 0;
    return MPC_OK;
  });
  if (rc) return rc;
  int threads = h->lane_threads;           // 0 = automatic
  if (threads <= 0) {
    const long long max_lanes = (long long)h->sm_count * LANE_MAX_THREADS;
    const long long rounds = (kp.B + max_lanes - 1) / max_lanes;
    const long long lanes_per_sm = (kp.B + rounds * h->sm_count - 1) / (rounds * h->sm_count);
    threads = (int)((lanes_per_sm + 31) / 32) * 32;
    if (threads < 32) threads = 32;
    if (threads > LANE_MAX_THREADS) threads = LANE_MAX_THREADS;
  }
  long long want = ((long long)kp.B + threads - 1) / threads;
  long long grid = (long long)h->sm_count * (h->lane_ctas_per_sm > 0 ? h->lane_ctas_per_sm : 1);
  if (grid > want) grid = want;
  if (grid < 1) grid = 1;
  // rule 1 (off by default; profiles/r01_handoff_sweep.txt and r01_tail_packing_sweep.txt: 13% on the 64K batch of
  // config-stable at 13 iterations, but a loss on workloads with a wider spread of iteration counts, and nothing on
  // top of rule 2): needs the coop kernel
  const bool rule1 = h->handoff_iter > 0 && kp.B >= MPC_LANE_MIN_BATCH && kp.B <= MPC_HANDOFF_MAX_BATCH;
  const int park = kp.B >= MPC_TAIL_MIN_BATCH ? h->park_lanes : 0;
  const int phases = park > 0 ? h->resume_phases : 0;
  int *cnt = h->d_counter + 1;   // [2k] records written by launch k of the chain, [2k + 1] cursor of the coop kernel
  kp.handoff_iter = INT_MAX;
  kp.ckpt_count = cnt; kp.ckpt_next = cnt + 1; kp.ckpt_in_count = cnt;
  rc = ensure_restart(h, kp);
  if (rc) return rc;
  CK(cudaMemsetAsync(kp.counter, 0, MPC_HIST0 * sizeof(int), st));
  // The lane kernel hands every problem that needs a rare branch of the algorithm (restoration phase, watchdog, a
  // large filter, tiny steps) to the coop kernel: as a record where a slot is free, else through the restart list.
  // So a chain always ends with a launch of the coop kernel; it returns at once when it has nothing to do.
  const size_t rec = Lane<NS, false>::CK_SIZE;
  size_t cap = (size_t)kp.B / 8;
  const size_t sparse = (size_t)grid * threads * (park > 0 ? park : 0) / 32 + 1024;
  if (cap < sparse) cap = sparse;
  if (cap > 32768) cap = 32768;
  if (cap > (size_t)kp.B) cap = kp.B;
  if (!h->d_ckpt || h->cap_ckpt < cap || h->ckpt_ns != NS) {
    cudaFree(h->d_ckpt);
    h->d_ckpt = nullptr; h->cap_ckpt = 0;
    // no memory for the record buffers (2.6 GB for the largest case, NS = 64): run without tail handling
    while (cap >= 1024 && cudaMalloc(&h->d_ckpt, 2 * cap * rec * sizeof(double)) != cudaSuccess) {
      (void)cudaGetLastError();
      h->d_ckpt = nullptr;
      cap /= 4;
    }
    if (h->d_ckpt) { h->cap_ckpt = cap; h->ckpt_ns = NS; }
  }
  if (!h->d_ckpt) {
    // no record buffers at all: one launch, hand-overs go through the restart list
    mpc_lane_kernel<NS, false, WARM><<<(unsigned)grid, threads, 0, st>>>(kp);
    CK(cudaGetLastError());
    h->launches++;
    return launch_coop_family<NS>(h, mpc_coop_resume_kernel<NS, WARM>, "finisher", kp, kp.B, st);
  }
  cap = h->cap_ckpt;
  double *buf[2] = {h->d_ckpt, h->d_ckpt + h->cap_ckpt * rec};
  kp.ckpt_cap = (int)cap;
  kp.ckpt = buf[0]; kp.ckpt_count = cnt;
  kp.park_lanes = park; kp.handoff_iter = rule1 ? h->handoff_iter : INT_MAX;
  kp.chain_counts = cnt; kp.chain_buf0 = buf[0]; kp.chain_buf1 = buf[1];
  kp.chain_pos = 0; kp.chain_last = phases + 1; kp.resume_min = h->resume_min;
  mpc_lane_kernel<NS, false, WARM><<<(unsigned)grid, threads, 0, st>>>(kp);
  CK(cudaGetLastError());
  h->launches++;
  // resume launches: enough lanes for a full buffer in one pass, dealt over all SMs.  Each works out on the device
  // which buffer holds the live records (chain_resolve) and returns at once if there are too few to be worth a pass.
  int rthreads = (int)(((cap + h->sm_count - 1) / h->sm_count + 31) / 32) * 32;
  if (rthreads > LANE_MAX_THREADS) rthreads = LANE_MAX_THREADS;
  long long rgrid = ((long long)cap + rthreads - 1) / rthreads;
  if (rgrid > h->sm_count) rgrid = h->sm_count;
  kp.handoff_iter = INT_MAX;
  kp.perm = nullptr;
  kp.ckpt = nullptr; kp.ckpt_count = nullptr;
  for (int k = 1; k <= phases; k++) {
    kp.chain_pos = k;
    mpc_lane_kernel<NS, true, WARM><<<(unsigned)rgrid, rthreads, 0, st>>>(kp);
    CK(cudaGetLastError());
    h->launches++;
  }
  kp.chain_pos = phases + 1;
  kp.park_lanes = 0;
  if (pre) {
    // from here on only the final launch writes outputs, and only those of the problems in its record list
    CK(cudaEventRecord(h->ev_pre, st));
    pre->recorded = true;
    pre->kp = kp;
    pre->rec = (int)Lane<NS, false>::CK_SIZE; pre->cki = (int)Lane<NS, false>::CK_I;
  }
  return launch_coop_family<NS>(h, mpc_coop_resume_kernel<NS, WARM>, "finisher", kp,
                                (long long)kp.B < (long long)cap * 2 ? kp.B : (long long)cap * 2, st);
}

// The coop kernel: one problem per group of 16 or 32 lanes, per-stage rows in shared memory.
template <int NS, bool WARM>
static int launch_coop(mpc_handle *h, KParams &kp, cudaStream_t st) {
  kp.handoff_iter = INT_MAX; kp.ckpt_count = h->d_counter + 1; kp.ckpt_next = h->d_counter + 2;
  if (kp.counter) CK(cudaMemsetAsync(kp.counter, 0, sizeof(int), st));
  return launch_coop_family<NS>(h, mpc_coop_kernel<NS, WARM>, "coop kernel", kp, kp.B, st);
}

extern "C" int mpc_set_dual_outputs(mpc_handle *h, double *lambda, double *zl, double *zu) {
  if (!h || ((lambda != nullptr) != (zl != nullptr)) || ((lambda != nullptr) != (zu != nullptr))) return MPC_EINVAL;
  h->dual_lam = lambda; h->dual_zl = zl; h->dual_zu = zu;
  return MPC_OK;
}

extern "C" int mpc_set_warm_start(mpc_handle *h, const double *x0, const double *lambda0, const double *zl0,
                                  const double *zu0, double mu_init) {
  if (!h || !(mu_init >= 0.0) || mu_init == INFINITY) return MPC_EINVAL;
  h->ws_x = x0;
  h->ws_lam = x0 ? lambda0 : nullptr; h->ws_zl = x0 ? zl0 : nullptr; h->ws_zu = x0 ? zu0 : nullptr;
  h->ws_mu = mu_init > 0.0 ? mu_init : 0.1;   // Ipopt's mu_init default
  return MPC_OK;
}

// Receding-horizon shift, one thread per problem: every block of stages of the layouts of `full` and of the multiplier
// outputs moves one stage earlier.  The new last stage of a state block continues with the increment of the old last
// stage (the model's step with the last stage's rates held: the shift needs neither the polynomial nor dt, and uses
// only additions, so that a CPU restatement gives the same bits); actuations and multipliers repeat their last stage.
__global__ void mpc_warm_start_shift_kernel(int B, int N, const double *x, const double *lam, const double *zl,
                                            const double *zu, double *x0, double *lam0, double *zl0, double *zu0) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const size_t sB = (size_t)B;
  auto shift = [&](const double *in, double *out, int r0, int n, bool extrapolate) {
    for (int i = 0; i + 1 < n; i++) out[(size_t)(r0 + i) * sB + b] = in[(size_t)(r0 + i + 1) * sB + b];
    const double last = in[(size_t)(r0 + n - 1) * sB + b];
    out[(size_t)(r0 + n - 1) * sB + b] = extrapolate ? __dadd_rn(last, __dsub_rn(last, in[(size_t)(r0 + n - 2) * sB + b])) : last;
  };
  // x, y, psi, v, cte, epsi: N stages from row k*N; delta, a: N-1 stages from rows 6N, 7N-1 (MPC.cpp:189-196)
  for (int k = 0; k < 6; k++) shift(x, x0, k * N, N, true);
  shift(x, x0, 6 * N, N - 1, false);
  shift(x, x0, 7 * N - 1, N - 1, false);
  if (lam)
    for (int k = 0; k < 6; k++) shift(lam, lam0, k * N, N, false);
  const double *zin[2] = {zl, zu};
  double *zout[2] = {zl0, zu0};
  for (int j = 0; j < 2; j++) {
    if (!zin[j]) continue;
    for (int k = 0; k < 6; k++) shift(zin[j], zout[j], k * N, N, false);
    shift(zin[j], zout[j], 6 * N, N - 1, false);
    shift(zin[j], zout[j], 7 * N - 1, N - 1, false);
  }
}

extern "C" int mpc_warm_start_shift(mpc_handle *h, int B, const double *x, const double *lambda, const double *zl,
                                    const double *zu, double *x0, double *lambda0, double *zl0, double *zu0,
                                    void *cuda_stream) {
  if (!h || B < 0 || !x || !x0 || (!lambda != !lambda0) || (!zl != !zl0) || (!zu != !zu0)) return MPC_EINVAL;
  if (B == 0) return MPC_OK;
  CK(cudaSetDevice(h->device));
  mpc_warm_start_shift_kernel<<<(B + 255) / 256, 256, 0, (cudaStream_t)cuda_stream>>>(B, h->cfg.N, x, lambda, zl, zu,
                                                                                      x0, lambda0, zl0, zu0);
  CK(cudaGetLastError());
  h->launches++;
  return MPC_OK;
}

extern "C" int mpc_set_handoff(mpc_handle *h, int iterations) {
  if (!h || iterations < 0) return MPC_EINVAL;
  h->handoff_iter = iterations;
  return MPC_OK;
}

extern "C" int mpc_set_tail(mpc_handle *h, int park_lanes, int resume_launches, int resume_min_records, int flags) {
  if (!h || park_lanes < 0 || park_lanes > 31 || resume_launches < 0 || resume_launches > MPC_MAX_PHASES || resume_min_records < 0) return MPC_EINVAL;
  h->park_lanes = park_lanes;
  h->resume_phases = resume_launches;
  h->resume_min = resume_min_records;
  h->sort_ragged = (flags & MPC_TAIL_SORT_RAGGED) != 0;
  h->no_early_copy = (flags & MPC_TAIL_LATE_COPY) != 0;
  return MPC_OK;
}

extern "C" int mpc_set_kernel(mpc_handle *h, int kind, int lane_threads, int lane_ctas_per_sm) {
  if (!h || (kind != MPC_KERNEL_AUTO && kind != MPC_KERNEL_LANE && kind != MPC_KERNEL_COOP)) return MPC_EINVAL;
  if (lane_threads != 0 && (lane_threads < 32 || lane_threads > LANE_MAX_THREADS || lane_threads % 32)) return MPC_EINVAL;
  h->kernel_kind = kind;
  h->lane_threads = lane_threads;
  h->lane_ctas_per_sm = lane_ctas_per_sm < 0 ? 0 : lane_ctas_per_sm;
  return MPC_OK;
}

// the configuration part of the launch parameters
static void fill_kparams(const mpc_config &c, int B, KParams &kp) {
  memset(&kp, 0, sizeof(kp));
  kp.B = B; kp.Nmax = c.N; kp.max_iter = c.max_iter; kp.n_steers = c.n_steers; kp.n_steer_speeds = c.n_steer_speeds;
  kp.dt = c.dt; kp.Lf = c.Lf; kp.cte_panic = c.cte_panic; kp.epsi_panic = c.epsi_panic;
  kp.max_speed = c.max_speed; kp.max_steering = c.max_steering; kp.max_accel = c.max_accel; kp.max_decel = c.max_decel;
  kp.tol = c.tol;
  kp.watchdog_trigger = c.watchdog_trigger; kp.filter_reset_trigger = c.filter_reset_trigger; kp.tiny_step_tol = c.tiny_step_tol;
  memcpy(kp.weights, c.weights, sizeof(kp.weights));
  memcpy(kp.steers, c.steers, sizeof(kp.steers));
  memcpy(kp.steer_speeds, c.steer_speeds, sizeof(kp.steer_speeds));
}

// a warm start is defined for the whole horizon of every problem: not with per-problem horizons
static int check_warm_start(const mpc_handle *h, const int *N_per) { return h->ws_x && N_per ? MPC_EINVAL : MPC_OK; }

// What one solve_batch call needs beyond the problem arrays.
struct SolveCall {
  const double *ws_x, *ws_lam, *ws_zl, *ws_zu;   // warm start (ws_x NULL: cold start)
  double ws_mu;
  double *dual_lam, *dual_zl, *dual_zu;           // multiplier outputs, or NULL
  bool one_shot;                                  // one problem per lane group, no work queue (single solves)
  PreFinisher *pre;                               // early copy-back: record h->ev_pre before a chain's final launch, or NULL
};

// A call with the handle's bound settings: its multiplier outputs, and its warm start if `warm` (the C-ABI's batch
// entry points; the single solve and the MPC::run-level entry points start where the reference does).
static SolveCall bound_call(const mpc_handle *h, bool warm) {
  SolveCall call = {};
  call.dual_lam = h->dual_lam; call.dual_zl = h->dual_zl; call.dual_zu = h->dual_zu;
  if (warm && h->ws_x) {
    call.ws_x = h->ws_x; call.ws_lam = h->ws_lam; call.ws_zl = h->ws_zl; call.ws_zu = h->ws_zu; call.ws_mu = h->ws_mu;
  }
  return call;
}

static int solve_batch(mpc_handle *h, const SolveCall &call, int B, const double *state, const double *coeffs,
                       const double *yaw_lo, const double *yaw_hi, const double *weights, const int *N_per,
                       const double *dt_per, double *result, double *traj_x, double *traj_y, double *full, int *status,
                       int *iters, void *cuda_stream) {
  if (!h || B < 0 || !state || !coeffs || !yaw_lo || !yaw_hi || !result) return MPC_EINVAL;
  if (call.ws_x && N_per) return MPC_EINVAL;
  if (B == 0) return MPC_OK;
  CK(cudaSetDevice(h->device));
  const mpc_config &c = h->cfg;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  KParams kp;
  fill_kparams(c, B, kp);
  kp.state = state; kp.coeffs = coeffs; kp.yaw_lo = yaw_lo; kp.yaw_hi = yaw_hi; kp.weights_pp = weights;
  kp.N_pp = N_per; kp.dt_pp = dt_per;
  kp.result = result; kp.traj_x = traj_x; kp.traj_y = traj_y; kp.full = full; kp.status = status; kp.iters = iters;
  kp.counter = h->d_counter;
  kp.dual_lam = call.dual_lam; kp.dual_zl = call.dual_zl; kp.dual_zu = call.dual_zu;
  kp.ws_x = call.ws_x; kp.ws_lam = call.ws_lam; kp.ws_zl = call.ws_zl; kp.ws_zu = call.ws_zu; kp.ws_mu = call.ws_mu;
  // Kernel choice (crossovers measured on B200, profiles/r01_kernel_crossover.txt): below MPC_LANE_MIN_BATCH
  // problems there are fewer problems than lanes and the time is set by the longest-running problem, so the
  // coop kernel (one problem per group of 16/32 lanes) wins; above it the lane kernel (one problem per lane)
  // has the throughput.
  int kind = h->kernel_kind;
  if (kind == MPC_KERNEL_AUTO) {
    if (c.N > 32) kind = B <= MPC_COOP_MAX_BATCH_LONG ? MPC_KERNEL_COOP : MPC_KERNEL_LANE;
    else kind = B >= MPC_LANE_MIN_BATCH ? MPC_KERNEL_LANE : MPC_KERNEL_COOP;
  }
  const bool coop = kind == MPC_KERNEL_COOP;
  if (coop && call.one_shot) kp.counter = nullptr;
  if (!coop && N_per && B >= MPC_TAIL_MIN_BATCH && h->sort_ragged) {
    if (!h->d_perm || h->cap_perm < (size_t)B) {
      cudaFree(h->d_perm);
      h->d_perm = nullptr;
      CK(cudaMalloc(&h->d_perm, (size_t)B * sizeof(int)));
      h->cap_perm = B;
    }
    int *hist = h->d_counter + MPC_HIST0;
    CK(cudaMemsetAsync(hist, 0, (MPC_NMAX + 1) * sizeof(int), st));
    const int sg = (B + 255) / 256 < 4 * h->sm_count ? (B + 255) / 256 : 4 * h->sm_count;
    mpc_horizon_hist_kernel<<<sg, 256, 0, st>>>(N_per, B, hist);
    mpc_horizon_scan_kernel<<<1, 1, 0, st>>>(hist);
    mpc_horizon_scatter_kernel<<<sg, 256, 0, st>>>(N_per, B, hist, h->d_perm);
    CK(cudaGetLastError());
    h->launches += 3;
    kp.perm = h->d_perm;
  }
  // warm-started launches run their own instantiations of the kernels (Lane::init)
  auto launch = [&](auto ns, auto warm) {
    constexpr int NS = decltype(ns)::value;
    constexpr bool WARM = decltype(warm)::value;
    return coop ? launch_coop<NS, WARM>(h, kp, st) : launch_lane<NS, WARM>(h, kp, st, call.pre);
  };
  return with_horizon(c.N, [&](auto ns) {
    return kp.ws_x ? launch(ns, std::true_type()) : launch(ns, std::false_type());
  });
}

extern "C" int mpc_solve_batch(mpc_handle *h, int B, const double *state, const double *coeffs,
                               const double *yaw_lo, const double *yaw_hi, const double *weights,
                               const int *N_per, const double *dt_per, double *result, double *traj_x,
                               double *traj_y, double *full, int *status, int *iters, void *cuda_stream) {
  if (!h) return MPC_EINVAL;
  return solve_batch(h, bound_call(h, true), B, state, coeffs, yaw_lo, yaw_hi, weights, N_per, dt_per, result, traj_x,
                     traj_y, full, status, iters, cuda_stream);
}

extern "C" int mpc_solution_sensitivity(mpc_handle *h, int B, const double *state, const double *coeffs,
                                        const double *yaw_lo, const double *yaw_hi, const double *weights,
                                        const double *dt_per, const double *full, const double *lambda, const double *zl,
                                        const double *zu, const int *status, double *dresult, double *dfull,
                                        void *cuda_stream) {
  if (!h || B < 0 || !state || !coeffs || !yaw_lo || !yaw_hi || !full || !lambda || !zl || !zu || !dresult)
    return MPC_EINVAL;
  if (B == 0) return MPC_OK;
  CK(cudaSetDevice(h->device));
  KParams kp;
  fill_kparams(h->cfg, B, kp);
  kp.state = state; kp.coeffs = coeffs; kp.yaw_lo = yaw_lo; kp.yaw_hi = yaw_hi; kp.weights_pp = weights; kp.dt_pp = dt_per;
  const SensArgs A = {full, lambda, zl, zu, status, dresult, dfull};
  return with_horizon(h->cfg.N, [&](auto ns) {
    mpc_sensitivity_kernel<decltype(ns)::value><<<(B + 127) / 128, 128, 0, (cudaStream_t)cuda_stream>>>(kp, A);
    CK(cudaGetLastError());
    h->launches++;
    return MPC_OK;
  });
}

// Early copy-back: the outputs of the problems the final launch of a chain finished, written again -- straight into
// the caller's (pinned, device-mapped) host arrays -- after the bulk copies that ran beside that launch.  Column b of
// every output array, all rows, for every record of the final launch's list.
struct PatchArrays {
  const double *src[4]; double *dst[4]; int rows[4];     // result, traj_x, traj_y, full
  const int *isrc[2]; int *idst[2];                      // status, iters
};
__global__ void mpc_patch_outputs_kernel(const KParams P, int rec_size, int cki, const PatchArrays A) {
  const ChainIO io = chain_resolve(P);
  const size_t B = (size_t)P.B;
  const int R = A.rows[0] + A.rows[1] + A.rows[2] + A.rows[3] + 2;
  int n_restart = *P.restart_count;   // problems the final launch solved from the start (no record)
  if (n_restart > P.B) n_restart = P.B;
  const int n_all = io.n + n_restart;
  const long long total = (long long)n_all * R;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(idx % n_all);
    int r = (int)(idx / n_all);
    const int b = k < io.n ? (int)io.in[(size_t)k * rec_size + cki] : P.restart_list[k - io.n];
    if (r >= R - 2) {
      const int a = r - (R - 2);
      if (A.idst[a]) A.idst[a][b] = A.isrc[a][b];
      continue;
    }
    for (int a = 0; a < 4; a++) {
      if (r < A.rows[a]) { A.dst[a][(size_t)r * B + b] = A.src[a][(size_t)r * B + b]; break; }
      r -= A.rows[a];
    }
  }
}

// ---- host-pointer entry points -------------------------------------------------------------------
// the device staging arrays of a batch of horizon N, each at stride cap_B
struct Staging {
  double *state, *coef, *ylo, *yhi, *w, *dt;   // inputs
  double *res, *tx, *ty, *full;                // outputs
  int *status, *iters, *N;
};
static int ensure_staging(mpc_handle *h, size_t B, int N, bool with_w, Staging *s) {
  if (!h->d_in || h->cap_B < B || h->cap_N < N || (!h->cap_w && with_w)) {
    cudaFree(h->d_in); cudaFree(h->d_out); cudaFree(h->d_iout); cudaFreeHost(h->h_pin);
    h->d_in = h->d_out = nullptr; h->d_iout = nullptr; h->h_pin = nullptr;
    h->cap_B = 0; h->cap_N = 0; h->cap_w = false;   // a failed allocation below must not leave a capacity behind
    size_t cap = B < 256 ? 256 : B;
    size_t nin = (6 + 5 + 2 + 12 + 1) * cap;            // state, coeffs, yaw, weights, dt
    size_t nout = (9 + 2 * (size_t)N + (8 * (size_t)N - 2)) * cap;
    CK(cudaMalloc(&h->d_in, nin * sizeof(double)));
    CK(cudaMalloc(&h->d_out, nout * sizeof(double)));
    CK(cudaMalloc(&h->d_iout, 3 * cap * sizeof(int)));
    CK(cudaMallocHost(&h->h_pin, 64 * sizeof(double) + (9 + 2 * (size_t)MPC_NMAX) * sizeof(double)));
    h->cap_B = cap; h->cap_N = N; h->cap_w = true;
  }
  if (s) {
    const size_t cap = h->cap_B;
    s->state = h->d_in; s->coef = s->state + 6 * cap; s->ylo = s->coef + 5 * cap; s->yhi = s->ylo + cap;
    s->w = s->yhi + cap; s->dt = s->w + 12 * cap;
    s->res = h->d_out; s->tx = s->res + 9 * cap; s->ty = s->tx + (size_t)N * cap; s->full = s->ty + (size_t)N * cap;
    s->status = h->d_iout; s->iters = s->status + cap; s->N = s->iters + cap;
  }
  return MPC_OK;
}

extern "C" int mpc_solve_batch_host(mpc_handle *h, int B, const double *state, const double *coeffs,
                                    const double *yaw_lo, const double *yaw_hi, const double *weights,
                                    const int *N_per, const double *dt_per, double *result, double *traj_x,
                                    double *traj_y, double *full, int *status, int *iters) {
  if (!h || B < 0 || !state || !coeffs || !yaw_lo || !yaw_hi || !result || check_warm_start(h, N_per)) return MPC_EINVAL;
  if (B == 0) return MPC_OK;
  CK(cudaSetDevice(h->device));
  const int N = h->cfg.N;
  Staging d;
  int rc = ensure_staging(h, (size_t)B, N, weights != nullptr, &d);
  if (rc) return rc;
  cudaStream_t st = h->stream;
  const size_t sB = (size_t)B * sizeof(double);
  // inputs are [k][B] with stride B on the host and on the device.  An input that lies in pinned (page-locked,
  // device-mapped) host memory is not copied: the kernels read each value once, at the start of its problem, straight
  // over PCIe -- measured free (4.61 against 4.60 ms for the 64K batch) where the copies cost 0.15 ms.  Outputs are
  // always staged: written from the kernels they are scattered 8-byte PCIe writes (+0.76 ms), the copy is 0.3 ms.
  auto stage = [&](const void *host, void *dev, size_t bytes, const void **use) -> cudaError_t {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
      *use = at.devicePointer;
      return cudaSuccess;
    }
    (void)cudaGetLastError();
    *use = dev;
    return cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st);
  };
  const void *u_state, *u_coef, *u_ylo, *u_yhi, *u_w = nullptr, *u_dt = nullptr, *u_N = nullptr;
  CK(stage(state, d.state, 6 * sB, &u_state));
  CK(stage(coeffs, d.coef, 5 * sB, &u_coef));
  CK(stage(yaw_lo, d.ylo, sB, &u_ylo));
  CK(stage(yaw_hi, d.yhi, sB, &u_yhi));
  if (weights) CK(stage(weights, d.w, 12 * sB, &u_w));
  if (dt_per) CK(stage(dt_per, d.dt, sB, &u_dt));
  if (N_per) CK(stage(N_per, d.N, (size_t)B * sizeof(int), &u_N));
  // Early copy-back.  In a lane-kernel chain the final launch (the finisher) works for a quarter of the step on a few
  // thousand long-running problems; every other result is final before it starts.  If all output arrays are pinned
  // and device-mapped, the device->host copies run on a second stream beside the finisher, and a small kernel then
  // rewrites the finisher's problems (columns of the output arrays) straight into the host arrays.
  PatchArrays pa;
  memset(&pa, 0, sizeof(pa));
  auto mapped = [&](void *host) -> void * {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) return at.devicePointer;
    (void)cudaGetLastError();
    return nullptr;
  };
  bool early = !h->no_early_copy;
  {
    double *hostp[4] = {result, traj_x, traj_y, full};
    const double *devp[4] = {d.res, d.tx, d.ty, d.full};
    const int rows[4] = {9, N, N, 8 * N - 2};
    for (int a = 0; a < 4 && early; a++) {
      if (!hostp[a]) continue;
      pa.dst[a] = (double *)mapped(hostp[a]); pa.src[a] = devp[a]; pa.rows[a] = rows[a];
      if (!pa.dst[a]) early = false;
    }
    int *hosti[2] = {status, iters};
    const int *devi[2] = {d.status, d.iters};
    for (int a = 0; a < 2 && early; a++) {
      if (!hosti[a]) continue;
      pa.idst[a] = (int *)mapped(hosti[a]); pa.isrc[a] = devi[a];
      if (!pa.idst[a]) early = false;
    }
  }
  if (early && !h->stream2) {
    CK(cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_pre, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_copy, cudaEventDisableTiming));
  }
  if (N_per) {
    // ragged batch: rows at or beyond a problem's horizon are left untouched by the kernels, and the copies back
    // are whole arrays -- so the staging buffers start as copies of the caller's arrays
    if (traj_x) CK(cudaMemcpyAsync(d.tx, traj_x, (size_t)N * sB, cudaMemcpyHostToDevice, st));
    if (traj_y) CK(cudaMemcpyAsync(d.ty, traj_y, (size_t)N * sB, cudaMemcpyHostToDevice, st));
    if (full) CK(cudaMemcpyAsync(d.full, full, (8 * (size_t)N - 2) * sB, cudaMemcpyHostToDevice, st));
  }
  PreFinisher pre = {};
  SolveCall call = bound_call(h, true);
  if (early) call.pre = &pre;
  rc = solve_batch(h, call, B, (const double *)u_state, (const double *)u_coef, (const double *)u_ylo, (const double *)u_yhi,
                   (const double *)u_w, (const int *)u_N, (const double *)u_dt, d.res, traj_x ? d.tx : nullptr,
                   traj_y ? d.ty : nullptr, full ? d.full : nullptr, d.status, d.iters, st);
  if (rc) return rc;
  cudaStream_t cs = pre.recorded ? h->stream2 : st;
  if (pre.recorded) CK(cudaStreamWaitEvent(cs, h->ev_pre, 0));
  CK(cudaMemcpyAsync(result, d.res, 9 * sB, cudaMemcpyDeviceToHost, cs));
  if (traj_x) CK(cudaMemcpyAsync(traj_x, d.tx, (size_t)N * sB, cudaMemcpyDeviceToHost, cs));
  if (traj_y) CK(cudaMemcpyAsync(traj_y, d.ty, (size_t)N * sB, cudaMemcpyDeviceToHost, cs));
  if (full) CK(cudaMemcpyAsync(full, d.full, (8 * (size_t)N - 2) * sB, cudaMemcpyDeviceToHost, cs));
  if (status) CK(cudaMemcpyAsync(status, d.status, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, cs));
  if (iters) CK(cudaMemcpyAsync(iters, d.iters, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, cs));
  if (pre.recorded) {
    CK(cudaEventRecord(h->ev_copy, cs));
    CK(cudaStreamWaitEvent(st, h->ev_copy, 0));
    mpc_patch_outputs_kernel<<<h->sm_count, 256, 0, st>>>(pre.kp, pre.rec, pre.cki, pa);
    CK(cudaGetLastError());
    h->launches++;
  }
  CK(cudaStreamSynchronize(st));
  return MPC_OK;
}

// ---- several devices, one host thread ----------------------------------------------------------------------------
struct mpc_multi {
  int n;
  mpc_handle *h[64];
};

extern "C" int mpc_create_multi(const mpc_config *cfg, const int *devices, int n_devices, mpc_multi **out) {
  if (!out) return MPC_EINVAL;
  *out = nullptr;
  if (!devices || n_devices < 1 || n_devices > 64) return MPC_EINVAL;
  mpc_multi *m = new (std::nothrow) mpc_multi();
  if (!m) return MPC_ENOMEM;
  m->n = 0;
  for (int g = 0; g < n_devices; g++) {
    const int rc = mpc_create(cfg, devices[g], &m->h[g]);
    if (rc) { mpc_destroy_multi(m); return rc; }
    m->n = g + 1;
  }
  *out = m;
  return MPC_OK;
}

extern "C" void mpc_destroy_multi(mpc_multi *m) {
  if (!m) return;
  for (int g = 0; g < m->n; g++) mpc_destroy(m->h[g]);
  delete m;
}

extern "C" int mpc_multi_device_count(const mpc_multi *m) { return m ? m->n : 0; }
extern "C" mpc_handle *mpc_multi_handle(mpc_multi *m, int g) { return (m && g >= 0 && g < m->n) ? m->h[g] : nullptr; }

extern "C" int mpc_solve_batch_multi(mpc_multi *m, int B, const double *state, const double *coeffs,
                                     const double *yaw_lo, const double *yaw_hi, const double *weights,
                                     const int *N_per, const double *dt_per, double *result, double *traj_x,
                                     double *traj_y, double *full, int *status, int *iters) {
  if (!m || m->n < 1 || B < 0 || !state || !coeffs || !yaw_lo || !yaw_hi || !result) return MPC_EINVAL;
  for (int g = 0; g < m->n; g++)
    if (check_warm_start(m->h[g], N_per)) return MPC_EINVAL;
  if (B == 0) return MPC_OK;
  const int G = m->n;
  const int N = m->h[0]->cfg.N;
  const size_t pitchB = (size_t)B * sizeof(double);
  // queue every shard: copies in, launches, copies out -- nothing here waits for a device
  auto queue_shard = [&](int g) -> int {
    const long long lo = (long long)B * g / G, hi = (long long)B * (g + 1) / G;
    const int Bs = (int)(hi - lo);
    if (Bs == 0) return MPC_OK;
    mpc_handle *h = m->h[g];
    CK(cudaSetDevice(h->device));
    Staging d;
    int rc = ensure_staging(h, (size_t)Bs, N, weights != nullptr, &d);
    if (rc) return rc;
    cudaStream_t st = h->stream;
    const size_t w = (size_t)Bs * sizeof(double);
    // a shard of a [rows][B] array is `rows` runs of Bs values: one strided copy per array
    auto in2d = [&](double *dst, const double *src, int rows) {
      return cudaMemcpy2DAsync(dst, w, src + lo, pitchB, w, (size_t)rows, cudaMemcpyHostToDevice, st);
    };
    auto out2d = [&](double *dst, const double *src, int rows) {
      return cudaMemcpy2DAsync(dst + lo, pitchB, src, w, w, (size_t)rows, cudaMemcpyDeviceToHost, st);
    };
    CK(in2d(d.state, state, 6));
    CK(in2d(d.coef, coeffs, 5));
    CK(in2d(d.ylo, yaw_lo, 1));
    CK(in2d(d.yhi, yaw_hi, 1));
    if (weights) CK(in2d(d.w, weights, 12));
    if (dt_per) CK(in2d(d.dt, dt_per, 1));
    if (N_per) {
      CK(cudaMemcpyAsync(d.N, N_per + lo, (size_t)Bs * sizeof(int), cudaMemcpyHostToDevice, st));
      // rows at or beyond a problem's horizon stay as the caller left them (see mpc_solve_batch_host)
      if (traj_x) CK(in2d(d.tx, traj_x, N));
      if (traj_y) CK(in2d(d.ty, traj_y, N));
      if (full) CK(in2d(d.full, full, 8 * N - 2));
    }
    rc = solve_batch(h, bound_call(h, true), Bs, d.state, d.coef, d.ylo, d.yhi, weights ? d.w : nullptr,
                     N_per ? d.N : nullptr, dt_per ? d.dt : nullptr, d.res, traj_x ? d.tx : nullptr,
                     traj_y ? d.ty : nullptr, full ? d.full : nullptr, d.status, d.iters, st);
    if (rc) return rc;
    CK(out2d(result, d.res, 9));
    if (traj_x) CK(out2d(traj_x, d.tx, N));
    if (traj_y) CK(out2d(traj_y, d.ty, N));
    if (full) CK(out2d(full, d.full, 8 * N - 2));
    if (status) CK(cudaMemcpyAsync(status + lo, d.status, (size_t)Bs * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (iters) CK(cudaMemcpyAsync(iters + lo, d.iters, (size_t)Bs * sizeof(int), cudaMemcpyDeviceToHost, st));
    return MPC_OK;
  };
  int first_error = MPC_OK, queued = 0;
  for (; queued < G && first_error == MPC_OK; queued++) first_error = queue_shard(queued);
  // wait for every device that has work queued -- also after an error, so that no copy into the caller's arrays is
  // still in flight when this call returns
  for (int g = 0; g < queued; g++) {
    if (cudaSetDevice(m->h[g]->device) != cudaSuccess || cudaStreamSynchronize(m->h[g]->stream) != cudaSuccess) {
      if (first_error == MPC_OK) { snprintf(g_err, sizeof(g_err), "device %d: %s", m->h[g]->device, cudaGetErrorString(cudaGetLastError())); first_error = MPC_ECUDA; }
    }
  }
  return first_error;
}

extern "C" int mpc_set_warm_start_one(mpc_handle *h, int on, double mu_init) {
  if (!h || !(mu_init >= 0.0) || mu_init == INFINITY) return MPC_EINVAL;
  h->one_warm = on != 0;
  h->one_prev_ok = false;
  h->one_mu = mu_init;
  return MPC_OK;
}

// One problem, host pointers.
extern "C" int mpc_solve_one(mpc_handle *h, const double *state, const double *coeffs, double yaw_lo,
                             double yaw_hi, double *result, double *traj_x, double *traj_y, int *status,
                             int *iters) {
  if (!h || !state || !coeffs || !result) return MPC_EINVAL;
  CK(cudaSetDevice(h->device));
  const int N = h->cfg.N;
  int rc = ensure_staging(h, 1, N, false, nullptr);
  if (rc) return rc;
  cudaStream_t st = h->stream;
  double *hp = h->h_pin;                       // [13 inputs | 9 + 2N outputs | 2 ints]
  for (int k = 0; k < 6; k++) hp[k] = state[k];
  for (int k = 0; k < MPC_NCOEF; k++) hp[6 + k] = coeffs[k];
  hp[11] = yaw_lo; hp[12] = yaw_hi;
  // The kernel reads the inputs from and writes the outputs to the pinned staging block directly (unified
  // virtual addressing makes cudaMallocHost memory device-accessible under the same pointer): one launch and
  // one synchronisation, no copy calls -- a single solve is latency-bound and every API call counts.
  double *ho = hp + 16;
  int *hi = reinterpret_cast<int *>(hp + 16 + 9 + 2 * (size_t)N);
  double *full = nullptr;
  SolveCall call = bound_call(h, false);   // cold; the bound multiplier outputs unless the single-solve warm start is on
  call.one_shot = true;
  if (h->one_warm) {
    // the last solution and the next start point, each [x 8N-2 | lambda 6N | zl 8N-2 | zu 8N-2] (B = 1): the solve
    // writes the first, the shift turns it into the second
    const size_t nx = 8 * (size_t)N - 2, per = 3 * nx + 6 * (size_t)N;
    if (!h->d_one || h->one_N != N) {
      cudaFree(h->d_one);
      h->d_one = nullptr; h->one_N = 0; h->one_prev_ok = false;
      CK(cudaMalloc(&h->d_one, 2 * per * sizeof(double)));
      CK(cudaMemsetAsync(h->d_one, 0, 2 * per * sizeof(double), st));   // bound multipliers of unbounded variables stay 0
      h->one_N = N;
    }
    double *sol = h->d_one, *nxt = h->d_one + per;
    full = sol;
    call.dual_lam = sol + nx; call.dual_zl = sol + nx + 6 * N; call.dual_zu = sol + 2 * nx + 6 * N;
    if (h->one_prev_ok) {
      rc = mpc_warm_start_shift(h, 1, sol, sol + nx, sol + nx + 6 * N, sol + 2 * nx + 6 * N, nxt, nxt + nx,
                                nxt + nx + 6 * N, nxt + 2 * nx + 6 * N, st);
      if (rc) return rc;
      call.ws_x = nxt; call.ws_lam = nxt + nx; call.ws_zl = nxt + nx + 6 * N; call.ws_zu = nxt + 2 * nx + 6 * N;
      call.ws_mu = h->one_mu > 0.0 ? h->one_mu : 0.1;
    }
  }
  rc = solve_batch(h, call, 1, hp, hp + 6, hp + 11, hp + 12, nullptr, nullptr, nullptr, ho, ho + 9, ho + 9 + N, full, hi,
                   hi + 1, st);
  if (rc) return rc;
  CK(cudaStreamSynchronize(st));
  if (h->one_warm) h->one_prev_ok = hi[0] == MPC_STATUS_SUCCESS;   // a failed solve is no start point
  for (int k = 0; k < 9; k++) result[k] = ho[k];
  if (traj_x) for (int k = 0; k < N; k++) traj_x[k] = ho[9 + k];
  if (traj_y) for (int k = 0; k < N; k++) traj_y[k] = ho[9 + N + k];
  if (status) *status = hi[0];
  if (iters) *iters = hi[1];
  return MPC_OK;
}

// Native latency of mpc_solve_one: reps calls, problem k % n of the given set each, timed one by one on the host
// clock around the call (what a C++ caller of MPC::solve sees; the Python binding adds its own argument marshalling).
extern "C" int mpc_measure_solve_latency(mpc_handle *h, int n, const double *state, const double *coeffs,
                                         const double *yaw_lo, const double *yaw_hi, int reps, int warmup,
                                         double *p50_us, double *p99_us) {
  if (!h || n < 1 || !state || !coeffs || !yaw_lo || !yaw_hi || reps < 1 || warmup < 0 || !p50_us || !p99_us) return MPC_EINVAL;
  std::vector<double> t;
  t.reserve(reps);
  double res[9];
  int status = 0, iters = 0;
  for (int k = 0; k < warmup + reps; k++) {
    const int i = k % n;
    const auto t0 = std::chrono::steady_clock::now();
    int rc = mpc_solve_one(h, state + 6 * (size_t)i, coeffs + MPC_NCOEF * (size_t)i, yaw_lo[i], yaw_hi[i], res, nullptr, nullptr,
                           &status, &iters);
    const auto t1 = std::chrono::steady_clock::now();
    if (rc) return rc;
    if (k >= warmup) t.push_back(std::chrono::duration<double, std::micro>(t1 - t0).count());
  }
  std::sort(t.begin(), t.end());
  *p50_us = t[t.size() / 2];
  *p99_us = t[(size_t)((t.size() - 1) * 0.99)];
  return MPC_OK;
}

// ---- the simulator protocol without the socket: src/mpc_main.cpp:26-36 (hasData), 81-222 (onMessage) ----------
extern "C" int mpc_telemetry_parse(const char *msg, mpc_telemetry *out) {
  if (!msg || !out) return MPC_EINVAL;
  memset(out, 0, sizeof(*out));
  const std::string sdata(msg);
  if (!(sdata.size() > 2 && sdata[0] == '4' && sdata[1] == '2')) { out->kind = MPC_MSG_IGNORED; return MPC_OK; }
  // hasData(): "null" anywhere means no data; otherwise from the first '[' to the last "}]"
  std::string s;
  const size_t b1 = sdata.find_first_of("["), b2 = sdata.rfind("}]");
  if (sdata.find("null") == std::string::npos && b1 != std::string::npos && b2 != std::string::npos) s = sdata.substr(b1, b2 - b1 + 2);
  if (s.empty()) { out->kind = MPC_MSG_MANUAL; return MPC_OK; }
  JParser jp(s.c_str());
  JVal j = jp.val();
  if (!jp.ok || j.t != JVal::ARR || j.arr.size() < 2 || j.arr[0].t != JVal::STR) return MPC_EPARSE;
  if (j.arr[0].str != "telemetry") { out->kind = MPC_MSG_IGNORED; return MPC_OK; }
  JVal &d = j.arr[1];
  if (d.t != JVal::OBJ) return MPC_EPARSE;
  auto num = [&](const char *k, double &v) { if (!d.obj.count(k) || d.obj[k].t != JVal::NUM) return false; v = d.obj[k].num; return true; };
  if (!num("x", out->x) || !num("y", out->y) || !num("psi", out->psi) || !num("speed", out->speed_mph) ||
      !num("steering_angle", out->steering_angle)) return MPC_EPARSE;
  if (!d.obj.count("ptsx") || !d.obj.count("ptsy") || d.obj["ptsx"].t != JVal::ARR || d.obj["ptsy"].t != JVal::ARR) return MPC_EPARSE;
  const size_t n = d.obj["ptsx"].arr.size();
  if (n != d.obj["ptsy"].arr.size() || n < 3 || n > MPC_MAX_WAYPOINTS) return MPC_EPARSE;
  for (size_t i = 0; i < n; i++) { out->ptsx[i] = d.obj["ptsx"].arr[i].num; out->ptsy[i] = d.obj["ptsy"].arr[i].num; }
  out->npts = (int)n;
  out->kind = MPC_MSG_TELEMETRY;
  return MPC_OK;
}

extern "C" int mpc_telemetry_step(mpc_handle *h, const char *msg, double *throttle_prev, double tau_solve,
                                  int with_trajectory, char *reply, int reply_cap) {
  if (!h || !msg || !throttle_prev || !reply || reply_cap < 32) return MPC_EINVAL;
  reply[0] = 0;
  mpc_telemetry t;
  int rc = mpc_telemetry_parse(msg, &t);
  if (rc) return rc;
  if (t.kind == MPC_MSG_IGNORED) return MPC_OK;
  if (t.kind == MPC_MSG_MANUAL) { snprintf(reply, (size_t)reply_cap, "42[\"manual\",{}]"); return MPC_OK; }
  const mpc_config &c = h->cfg;
  double x = t.x, y = t.y;
  double psi = mpcrun::normalize_angle(t.psi);                  // mpc_main.cpp:127
  double v = mph2mps(t.speed_mph);                              // :129
  const double steer = -t.steering_angle;                       // :131
  const double accel_est = (*throttle_prev - v / 50.0) * 6;     // :156
  if (c.latency_ms) mpcrun::vehicle_move(&x, &y, &psi, &v, steer, accel_est, c.Lf, c.lookahead + tau_solve);   // :157-159
  const double pose[4] = {x, y, psi, v};
  double state[6], coeffs[MPC_NCOEF], ylo, yhi, res[9], out8[8], tx[MPC_NMAX], ty[MPC_NMAX];
  mpc_run_aux aux;
  rc = mpc_run_prepare(&c, pose, steer, t.ptsx, t.ptsy, t.npts, state, coeffs, &ylo, &yhi, &aux);
  if (rc) return rc;
  int status = 0, iters = 0;
  rc = mpc_solve_one(h, state, coeffs, ylo, yhi, res, tx, ty, &status, &iters);
  if (rc) return rc;
  if (status != MPC_STATUS_SUCCESS) printf("Ipopt failed with %d\n", status);   // MPC.cpp:301
  mpc_run_finish(&c, &aux, v, res, out8);
  const double steer_value = -out8[4];                          // :172
  const double throttle = mpcrun::compute_throttle(out8[5], out8[3], c.max_accel, c.max_decel, c.max_speed);   // :174
  *throttle_prev = throttle;
  // the reply object, keys in nlohmann's (sorted) order; without PLOT_TRAJECTORY the reference assigns NULL,
  // which nlohmann stores as the integer 0 (mpc_main.cpp:189-199)
  std::string js = "{";
  auto arr = [](const double *a, int n) { std::string s = "["; char b[40]; for (int i = 0; i < n; i++) { snprintf(b, sizeof(b), "%s%.15g", i ? "," : "", a[i]); s += b; } return s + "]"; };
  char b[64];
  js += "\"mpc_x\":" + (with_trajectory ? arr(tx, c.N) : std::string("0"));
  js += ",\"mpc_y\":" + (with_trajectory ? arr(ty, c.N) : std::string("0"));
  js += ",\"next_x\":" + (with_trajectory ? arr(t.ptsx, t.npts) : std::string("0"));
  js += ",\"next_y\":" + (with_trajectory ? arr(t.ptsy, t.npts) : std::string("0"));
  snprintf(b, sizeof(b), ",\"steering_angle\":%.15g", steer_value); js += b;
  snprintf(b, sizeof(b), ",\"throttle\":%.15g}", throttle); js += b;
  const std::string out = "42[\"steer\"," + js + "]";
  if ((int)out.size() + 1 > reply_cap) return MPC_EINVAL;
  memcpy(reply, out.c_str(), out.size() + 1);
  return MPC_OK;
}

// ---- whole control steps on the device ------------------------------------------------------------
// workspace: state 6, coeffs 5, yaw 2, aux 4, result 9 doubles per vehicle; status, iters ints
static int ensure_run_ws(mpc_handle *h, size_t B) {
  if (h->d_run && h->cap_run >= B) return MPC_OK;
  cudaFree(h->d_run); cudaFree(h->d_run_i);
  h->d_run = nullptr; h->d_run_i = nullptr;
  h->cap_run = 0;
  size_t cap = B < 1024 ? 1024 : B;
  CK(cudaMalloc(&h->d_run, 26 * cap * sizeof(double)));
  CK(cudaMalloc(&h->d_run_i, 2 * cap * sizeof(int)));
  h->cap_run = cap;
  return MPC_OK;
}

extern "C" int mpc_run_batch(mpc_handle *h, int B, const double *pose, const double *steering, const double *ptsx,
                             const double *ptsy, int npts, double *out8, double *traj_x, double *traj_y,
                             double *coeffs_out, double *ptsx_v, double *ptsy_v, int *status, int *iters,
                             void *cuda_stream) {
  if (!h || B < 0 || !pose || !ptsx || !ptsy || !out8 || npts < 3 || npts > MPC_MAX_WAYPOINTS) return MPC_EINVAL;
  if (check_run_config(&h->cfg)) return MPC_EINVAL;
  if (B == 0) return MPC_OK;
  CK(cudaSetDevice(h->device));
  int rc = ensure_run_ws(h, (size_t)B);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  double *w = h->d_run;               // packed at stride B: state 6, yaw 2, aux 4, result 9, coeffs 5
  RunBatch R;
  R.B = B; R.npts = npts; R.pose = pose; R.steering = steering; R.ptsx = ptsx; R.ptsy = ptsy;
  R.ptsx_v = ptsx_v; R.ptsy_v = ptsy_v;
  R.state = w; R.yaw_lo = w + 6 * (size_t)B; R.yaw_hi = R.yaw_lo + B; R.aux = R.yaw_hi + B;
  double *result = R.aux + 4 * (size_t)B;
  R.coeffs = coeffs_out ? coeffs_out : result + 9 * (size_t)B;
  int *d_status = status ? status : h->d_run_i, *d_iters = iters ? iters : h->d_run_i + B;
  const int thr = 128, grid = (B + thr - 1) / thr;
  mpc_run_pre_kernel<<<grid, thr, 0, st>>>(h->cfg, R);
  CK(cudaGetLastError());
  rc = solve_batch(h, bound_call(h, false), B, R.state, R.coeffs, R.yaw_lo, R.yaw_hi, nullptr, nullptr, nullptr, result,
                   traj_x, traj_y, nullptr, d_status, d_iters, st);
  if (rc) return rc;
  mpc_run_post_kernel<<<grid, thr, 0, st>>>(h->cfg, B, R.aux, result, out8);
  CK(cudaGetLastError());
  h->launches += 2;
  return MPC_OK;
}

// the closed loop as one launch of mpc_rollout_kernel: a lane group per vehicle, all T steps
template <int NS>
static int launch_rollout(mpc_handle *h, const LoopArgs &A, int T, cudaStream_t st) {
  KParams kp;
  fill_kparams(h->cfg, A.V, kp);
  kp.state = A.state; kp.coeffs = A.coeffs; kp.yaw_lo = A.yaw_lo; kp.yaw_hi = A.yaw_hi;
  kp.result = A.result; kp.status = const_cast<int *>(A.status); kp.iters = const_cast<int *>(A.iters);
  kp.handoff_iter = INT_MAX;
  return launch_coop_family<NS>(h, mpc_rollout_kernel<NS>, "rollout kernel", kp, A.V, st, h->cfg, A, T);
}

extern "C" int mpc_set_rollout_mode(mpc_handle *h, int mode) {
  if (!h || mode < MPC_ROLLOUT_AUTO || mode > MPC_ROLLOUT_PERSISTENT) return MPC_EINVAL;
  h->rollout_mode = mode;
  return MPC_OK;
}

extern "C" int mpc_rollout(mpc_handle *h, int V, int T, const double *track_x, const double *track_y, int n_track,
                           double *veh, int *seg, double *pending, double dt_ctrl, double tau_solve, double *rec,
                           void *cuda_stream) {
  if (!h || V < 0 || T < 0 || !track_x || !track_y || n_track < 6 || !veh || !seg || !(dt_ctrl > 0)) return MPC_EINVAL;
  if (h->cfg.latency_ms && !pending) return MPC_EINVAL;
  if (check_run_config(&h->cfg)) return MPC_EINVAL;
  if (V == 0 || T == 0) return MPC_OK;
  CK(cudaSetDevice(h->device));
  int rc = ensure_run_ws(h, (size_t)V);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  double *w = h->d_run;
  LoopArgs A;
  A.V = V; A.n_track = n_track; A.track_x = track_x; A.track_y = track_y; A.veh = veh; A.seg = seg; A.pending = pending;
  A.dt_ctrl = dt_ctrl; A.tau_solve = tau_solve; A.rec = rec;
  A.state = w; A.coeffs = w + 6 * (size_t)V; A.yaw_lo = w + 11 * (size_t)V; A.yaw_hi = w + 12 * (size_t)V;
  A.aux = w + 13 * (size_t)V; A.result = w + 17 * (size_t)V;
  int *d_status = h->d_run_i, *d_iters = h->d_run_i + V;
  A.status = d_status; A.iters = d_iters;
  const bool persistent = h->rollout_mode == MPC_ROLLOUT_PERSISTENT || (h->rollout_mode == MPC_ROLLOUT_AUTO && V <= MPC_ROLLOUT_PERSISTENT_MAX);
  if (persistent) {
    A.step = 0;
    return with_horizon(h->cfg.N, [&](auto ns) { return launch_rollout<decltype(ns)::value>(h, A, T, st); });
  }
  const int thr = 128, grid = (V + thr - 1) / thr;
  for (int k = 0; k < T; k++) {
    A.step = k;
    mpc_loop_pre_kernel<<<grid, thr, 0, st>>>(h->cfg, A);
    rc = solve_batch(h, bound_call(h, false), V, A.state, A.coeffs, A.yaw_lo, A.yaw_hi, nullptr, nullptr, nullptr,
                     A.result, nullptr, nullptr, nullptr, d_status, d_iters, st);
    if (rc) return rc;
    mpc_loop_post_kernel<<<grid, thr, 0, st>>>(h->cfg, A);
    h->launches += 2;
  }
  CK(cudaGetLastError());
  return MPC_OK;
}

// ---- FP64 FMA peak micro-benchmark (roofline denominator) -----------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double *out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int j = 0; j < 8; j++) {
      x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
      x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
  }
  double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
  if (s == 123.456) out[0] = s;   // keep the chains alive
}

extern "C" int mpc_measure_fp64_peak(int device, double *tflops) {
  if (!tflops) return MPC_EINVAL;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) { (void)cudaGetLastError(); return MPC_ENODEV; }
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  double *d = nullptr;
  CK(cudaMalloc(&d, 8));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  double best = 0;
  for (int rep = 0; rep < 5; rep++) {
    CK(cudaEventRecord(e0));
    dfma_peak_kernel<<<blocks, threads>>>(d, iters, 0.999999, 1e-9);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    double fl = 2.0 * 64.0 * iters * (double)blocks * threads;
    double tf = fl / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *tflops = best;
  return MPC_OK;
}

// records parked by launch k = 0, 1, ... of the last lane-kernel chain (synchronises the device)
extern "C" int mpc_tail_counts(mpc_handle *h, int *parked, int n) {
  if (!h || !parked || n < 0) return MPC_EINVAL;
  int host[MPC_HIST0];
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(host, h->d_counter, sizeof(host), cudaMemcpyDeviceToHost));
  for (int k = 0; k < n; k++) parked[k] = (1 + 2 * k < MPC_HIST0) ? host[1 + 2 * k] : 0;
  return MPC_OK;
}

extern "C" long long mpc_launch_count(const mpc_handle *h) { return h ? h->launches : 0; }
extern "C" const char *mpc_last_error(void) { return g_err; }
extern "C" const char *mpc_version(void) { return "mpc_b200 0.3 (sm_100a, fp64 interior point with restoration phase and watchdog; lane and coop kernels, explicit fma)"; }
