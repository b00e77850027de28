// C ABI of the dsx sampler (include/dsx.h): handle, weight loading, schedule, workspace, and the host
// side of the sampling loops.  The K-step loops run as a fixed sequence of kernel launches on the
// caller's stream -- no host synchronisation and no PyTorch op inside the loop
// (usr/diff/shallow_diffusion_tts.py:261-270 is a Python loop of ~300 ATen launches per step).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "dsx_internal.h"

namespace dsx {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int dev_alloc(dsx_handle* h, void** p, size_t bytes, bool model_owned) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? DSX_E_NOMEM : DSX_E_CUDA;
  }
  if (model_owned) h->owned.push_back(q);
  *p = q;
  return DSX_OK;
}

static void free_ws(Workspace& w) {
  void* ptrs[] = {w.X, w.SKIP, w.CONDF, w.G1, w.Zf, w.Y, w.CONDH, w.CP, w.S16, w.Z, w.DTAB, w.EMB, w.TVALS, w.EPS, w.XTMP, w.XSTATE};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  w = Workspace();
}

// Grow-only workspace: every buffer keeps its byte capacity; a call with a new (B, T) that fits re-uses the allocations
// (only the tensor maps are re-encoded, see tc_prepare_maps), so utterance lengths that change from call to call cost no
// cudaFree / cudaMalloc (cudaFree synchronises the device).  New allocations are zeroed on the caller's stream.
int ensure_workspace(dsx_handle* h, const Geom& g, int rows, cudaStream_t s) {
  Workspace& w = h->ws;
  const ModelDev& m = h->m;
  const bool tc = h->precision != DSX_PREC_FP32_SIMT;
  const size_t nf = g.frames_padded();
  bool moved = false;
  auto need = [&](void** p, size_t& cap, size_t bytes) -> int {
    if (cap >= bytes && *p) return DSX_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    w.bytes -= cap;
    cap = 0;
    const size_t grow = bytes + bytes / 8;      // headroom: slightly longer utterances next time do not reallocate
    DSX_TRY(dev_alloc(h, p, grow, false));
    DSX_CUDA(cudaMemsetAsync(*p, 0, grow, s));
    cap = grow;
    w.bytes += grow;
    moved = true;
    return DSX_OK;
  };
#define NEED(field, bytes) DSX_TRY(need(reinterpret_cast<void**>(&w.field), w.cap_##field, (bytes)))
  NEED(X, nf * m.C * 4);
  NEED(SKIP, nf * m.C * 4);
  if (tc) {
    const void* cond_before[2] = {w.CONDH, w.CP};
    NEED(Y, nf * m.C * 2 * 4);
    NEED(CONDH, nf * m.H * 2 * 2);
    NEED(S16, nf * m.C * 2 * 2);
    NEED(Z, static_cast<size_t>(m.L) * nf * m.C * 2);
    NEED(CP, static_cast<size_t>(m.L) * g.tiles * 2 * 256 * kTile * 4);
    if (cond_before[0] != w.CONDH || cond_before[1] != w.CP) h->cond_ready = false;
  } else {
    const void* cond_before = w.CONDF;
    NEED(G1, nf * 2 * m.C * 4);
    NEED(Zf, nf * m.C * 4);
    NEED(CONDF, nf * m.H * 4);
    if (cond_before != w.CONDF) h->cond_ready = false;
  }
  if (w.rows_cap < rows) {
    const int keep_rows = std::max(rows, w.rows_cap + w.rows_cap / 2);
    NEED(DTAB, static_cast<size_t>(keep_rows) * m.L * m.C * 4);
    NEED(EMB, static_cast<size_t>(keep_rows) * m.C * 4);
    NEED(TVALS, static_cast<size_t>(keep_rows) * 8);
    w.rows_cap = keep_rows;
  }
  const size_t mel = static_cast<size_t>(g.B) * m.M * g.T;
  NEED(EPS, 5 * mel * 4);
  NEED(XTMP, mel * 4);
  NEED(XSTATE, mel * 4);
#undef NEED
  if (moved) h->ws_epoch++;
  w.g = g;
  return DSX_OK;
}

int check_status(dsx_handle* h, cudaStream_t s, const char* what) {
  DSX_CUDA(cudaMemcpyAsync(h->status_host, h->status_dev, sizeof(int), cudaMemcpyDeviceToHost, s));
  DSX_CUDA(cudaStreamSynchronize(s));
  if (*h->status_host != 0) {
    int code = *h->status_host;
    cudaMemsetAsync(h->status_dev, 0, sizeof(int), s);
    // the tiles of the aborted launch stopped at different layers: their publish counters are no longer in lockstep.
    // Zero them and forget the geometry so the next stack launch starts from a clean state (the handle stays usable).
    reset_flags(h);
    set_error("%s: in-kernel watchdog tripped (code %d: 1xx producer, 2xx MMA issuer, 3xx epilogue wait)", what, code);
    return DSX_E_KERNEL;
  }
  return DSX_OK;
}

void reset_flags(dsx_handle* h) {
  if (h->flags_dev) cudaMemset(h->flags_dev, 0, static_cast<size_t>(h->flags_cap) * sizeof(unsigned int));
  h->flag_count = 0;
  h->flags_geom_b = 0;
  h->flags_geom_t = 0;
  h->flags_kind = 0;
}

// DSX_OPT_PROFILE: when `mode` is the selected one, record the start of a (start, stop) pair of CUDA events; *stop is the
// event the caller records to end it (null otherwise).
static int prof_start(dsx_handle* h, int mode, cudaStream_t s, cudaEvent_t* stop) {
  *stop = nullptr;
  if (h->profile != mode) return DSX_OK;
  while (h->prof_events.size() < h->prof_used + 2) {
    cudaEvent_t e;
    DSX_CUDA(cudaEventCreate(&e));
    h->prof_events.push_back(e);
  }
  *stop = h->prof_events[h->prof_used + 1];
  DSX_CUDA(cudaEventRecord(h->prof_events[h->prof_used], s));
  h->prof_used += 2;
  return DSX_OK;
}

static dsx_strides contiguous_mel(int M, int T) {
  dsx_strides xs;
  xs.b = static_cast<int64_t>(M) * T;
  xs.c = T;
  xs.t = 1;
  return xs;
}

// The head of DSX_PREC_FP32_SIMT as CUDA-core launches, the flags read as by k_tc_head.  eps goes to ha.eps, else to the
// history slot of the PNDM step, else to scratch slot 4 of ws.EPS.
static int simt_head(dsx_handle* h, const Geom& g, const HeadArgs& ha, cudaStream_t s) {
  const size_t mel = static_cast<size_t>(g.B) * h->m.M * g.T;
  const PlmsFuse* pl = ha.plms;
  float* eps = ha.eps ? ha.eps : (pl && pl->eps_store) ? pl->eps_store : h->ws.EPS + 4 * mel;
  float* x = ha.x;
  dsx_strides xs = ha.xs;
  if (ha.flags & TC_HEAD) DSX_TRY(launch_head(h, g, eps, s));
  if (ha.flags & TC_UPDATE) DSX_TRY(launch_ddpm_update(h, x, eps, ha.noise, ha.seed, ha.offset, ha.c, mel, g.T, s));
  if (ha.flags & TC_PLMS) {
    if (pl->x_out) { x = pl->x_out; xs = contiguous_mel(h->m.M, g.T); }
    DSX_TRY(launch_plms_update(h, x, ha.x, eps, pl->h1, pl->h2, pl->h3, pl->c, mel, s));
  }
  if (ha.flags & TC_INPROJ) DSX_TRY(launch_inproj(h, x, xs, g, s));
  return DSX_OK;
}

// Input projection of a call's first evaluation (table row (row0, row_per_b)); every later one runs in the head of the
// evaluation before it (TC_INPROJ).
static int start_eval(dsx_handle* h, const Geom& g, float* x, dsx_strides xs, int row0, int row_per_b, cudaStream_t s) {
  if (h->precision == DSX_PREC_FP32_SIMT) return launch_inproj(h, x, xs, g, s);
  HeadArgs ha;
  ha.flags = TC_INPROJ; ha.x = x; ha.xs = xs; ha.next_row0 = row0; ha.row_per_b = row_per_b;
  return launch_tc_head(h, g, ha, s);
}

// One evaluation: residual layers [0, nl) of table row (row0, row_per_b), then the head `ha` describes (none when ha.flags
// is 0).  The stack kernel runs both in one launch where it can take the call; otherwise the head is a launch of its own:
// k_tc_head, or the CUDA-core kernels of DSX_PREC_FP32_SIMT.  Weight set of DSX_PREC_FP16S: row j of a loop uses set j % R.
static int run_step(dsx_handle* h, const Geom& g, int row0, int row_per_b, int nl, const HeadArgs& ha, cudaStream_t s) {
  const bool fp32 = h->precision == DSX_PREC_FP32_SIMT;
  bool fused = false;
  cudaEvent_t stop;
  DSX_TRY(prof_start(h, 1, s, &stop));     // DSX_OPT_PROFILE = 1: one bracket per evaluation, around the residual stack
  if (fp32) {
    for (int l = 0; l < nl; ++l) DSX_TRY(launch_simt_layer(h, l, g, row0, row_per_b, s));
  } else if (tc_stack_usable(h, g)) {
    fused = ha.flags && h->fused_head && nl == h->m.L && h->profile != 2;
    DSX_TRY(launch_tc_stack(h, nl, g, row0, row_per_b, row0, s, fused ? &ha : nullptr));
  } else {
    DSX_TRY(launch_tc_layers(h, 0, nl, g, row0, row_per_b, s));
  }
  if (stop) DSX_CUDA(cudaEventRecord(stop, s));
  if (!ha.flags || fused) return DSX_OK;
  DSX_TRY(prof_start(h, 2, s, &stop));     // DSX_OPT_PROFILE = 2: around the separate head
  DSX_TRY(fp32 ? simt_head(h, g, ha, s) : launch_tc_head(h, g, ha, s));
  if (stop) DSX_CUDA(cudaEventRecord(stop, s));
  return DSX_OK;
}

// One DiffNet evaluation: x (any strides) -> eps (contiguous [B,1,M,T]).  Under dsx_debug_set_layer_limit only the first
// layers run, and no head.
static int run_eval(dsx_handle* h, const float* x, dsx_strides xs, const Geom& g, int row0, int row_per_b, float* eps,
                    cudaStream_t s) {
  const int nl = (h->layer_limit >= 0) ? std::min(h->layer_limit, h->m.L) : h->m.L;
  HeadArgs ha;
  ha.flags = nl == h->m.L ? TC_HEAD | TC_WRITE_EPS : 0;
  ha.x = const_cast<float*>(x);          // (read only with these flags)
  ha.xs = xs; ha.eps = eps;
  DSX_TRY(start_eval(h, g, ha.x, xs, row0, row_per_b, s));
  return run_step(h, g, row0, row_per_b, nl, ha, s);
}

// Workspace + tensor maps for (B, T) and, when `cond` is given, the conditioner pack and its hoisted projection (the
// step-independent part of every residual layer).  cond == NULL re-uses what the last call with a conditioner left behind
// (dsx_set_cond or any entry point): callers that drive the sampling loop themselves, one p_sample / DiffNet.forward per
// call, pay the pack + projection once per utterance batch instead of once per step.
static int prepare(dsx_handle* h, const float* cond, dsx_strides cs, int B, int T, int rows, Geom& g, cudaStream_t s) {
  DSX_CHECK(h && h->loaded, DSX_E_STATE, "dsx_load_diffnet has not been called");
  DSX_CHECK(B > 0 && T > 0, DSX_E_INVALID, "B and T must be positive (got %d, %d)", B, T);
  DSX_CUDA(cudaSetDevice(h->device));
  g.set(B, T);
  DSX_TRY(ensure_workspace(h, g, rows, s));
  if (h->precision != DSX_PREC_FP32_SIMT) DSX_TRY(tc_prepare_maps(h, g));
  if (!cond) {
    DSX_CHECK(h->cond_ready && h->cond_geom.B == B && h->cond_geom.T == T, DSX_E_STATE,
              "cond == NULL needs a conditioner set for the same (B, T) by dsx_set_cond or an earlier call (have %s %dx%d, asked %dx%d)",
              h->cond_ready ? "one for" : "none;", h->cond_geom.B, h->cond_geom.T, B, T);
    return DSX_OK;
  }
  h->cond_ready = false;
  DSX_TRY(launch_pack_cond(h, cond, cs, g, s));
  if (h->precision != DSX_PREC_FP32_SIMT) DSX_TRY(launch_tc_condproj(h, g, s));
  h->cond_ready = true;
  h->cond_geom = g;
  return DSX_OK;
}

static int sample_ddpm_impl(dsx_handle* h, float* x, const Geom& g, int t_start, int n_steps, const float* noise,
                            uint64_t seed, cudaStream_t s) {
  const size_t mel = static_cast<size_t>(g.B) * h->m.M * g.T;
  std::vector<int64_t> tv(n_steps);
  for (int j = 0; j < n_steps; ++j) tv[j] = t_start - 1 - j;
  DSX_CUDA(cudaMemcpyAsync(h->ws.TVALS, tv.data(), n_steps * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  DSX_CUDA(cudaStreamSynchronize(s));   // tv is a stack-owned staging buffer
  DSX_TRY(launch_embed_table(h, h->ws.TVALS, n_steps, s));
  const dsx_strides xs = contiguous_mel(h->m.M, g.T);
  DSX_TRY(start_eval(h, g, x, xs, 0, 0, s));
  for (int j = 0; j < n_steps; ++j) {
    const int t = t_start - 1 - j;
    HeadArgs ha;
    ha.flags = TC_HEAD | TC_UPDATE | (j + 1 < n_steps ? TC_INPROJ : 0);
    ha.x = x; ha.xs = xs; ha.seed = seed; ha.offset = static_cast<uint64_t>(j); ha.next_row0 = j + 1;
    ha.noise = noise ? noise + static_cast<size_t>(j) * mel : nullptr;
    ha.c.A = h->sched[DSX_SCH_SQRT_RECIP_ALPHAS_CUMPROD][t];
    ha.c.Bc = h->sched[DSX_SCH_SQRT_RECIPM1_ALPHAS_CUMPROD][t];
    ha.c.c1 = h->sched[DSX_SCH_POSTERIOR_MEAN_COEF1][t];
    ha.c.c2 = h->sched[DSX_SCH_POSTERIOR_MEAN_COEF2][t];
    ha.c.sigma = (t == 0) ? 0.f : expf(0.5f * h->sched[DSX_SCH_POSTERIOR_LOG_VARIANCE_CLIPPED][t]);
    DSX_TRY(run_step(h, g, j, 0, h->m.L, ha, s));
  }
  return DSX_OK;
}

// get_x_pred coefficients (usr/diff/shallow_diffusion_tts.py:174-185), fp32 op by op
static void plms_coefs(const dsx_handle* h, int t, int interval, PlmsCoef& c) {
  const std::vector<float>& ac = h->sched[DSX_SCH_ALPHAS_CUMPROD];
  const float a_t = ac[t];
  const float a_prev = (t < interval) ? 1.0f : ac[std::max(t - interval, 0)];
  const float a_t_sq = sqrtf(a_t), a_prev_sq = sqrtf(a_prev);
  c.a_diff = a_prev - a_t;
  c.kx = 1.0f / (a_t_sq * (a_t_sq + a_prev_sq));
  c.ke = 1.0f / (a_t_sq * (sqrtf((1.0f - a_prev) * a_t) + sqrtf((1.0f - a_t) * a_prev)));
}

// Linear multistep weights (shallow_diffusion_tts.py:188-197) of dsx_plms_update's `mode`: 0 = eps_t alone (the warm-up's
// x'), 1 = (eps_t + eps'') / 2 (the warm-up's update), 2..4 = Adams-Bashforth over eps_t and the 1..3 previous eps.
static void plms_weights(int mode, PlmsCoef& c) {
  static const float w[5][5] = {{1, 0, 0, 0, 1}, {1, 1, 0, 0, 2}, {3, -1, 0, 0, 2}, {23, -16, 5, 0, 12}, {55, -59, 37, -9, 24}};
  c.w0 = w[mode][0]; c.w1 = w[mode][1]; c.w2 = w[mode][2]; c.w3 = w[mode][3]; c.denom = w[mode][4];
}

static int sample_plms_impl(dsx_handle* h, float* x, const Geom& g, int t_start, int interval, cudaStream_t s) {
  const size_t mel = static_cast<size_t>(g.B) * h->m.M * g.T;
  std::vector<int> steps;
  for (int t = 0; t < t_start; t += interval) steps.push_back(t);
  std::reverse(steps.begin(), steps.end());
  const int n = static_cast<int>(steps.size());
  DSX_CHECK(n > 0, DSX_E_INVALID, "empty PLMS schedule");
  // table rows: 0..n-1 = the steps, row n = the extra warm-up evaluation at max(t0 - interval, 0)
  std::vector<int64_t> tv(n + 1);
  for (int j = 0; j < n; ++j) tv[j] = steps[j];
  tv[n] = std::max(steps[0] - interval, 0);
  DSX_CUDA(cudaMemcpyAsync(h->ws.TVALS, tv.data(), (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  DSX_CUDA(cudaStreamSynchronize(s));
  DSX_TRY(launch_embed_table(h, h->ws.TVALS, n + 1, s));
  const dsx_strides xs = contiguous_mel(h->m.M, g.T);
  DSX_TRY(start_eval(h, g, x, xs, 0, 0, s));
  // history ring of eps_t in ws.EPS slots 0..3: hist[0] = the most recent, nh of them filled
  const float* hist[3] = {nullptr, nullptr, nullptr};
  int nh = 0;
  for (int j = 0; j < n; ++j) {
    float* e0 = h->ws.EPS + static_cast<size_t>(j % 4) * mel;
    const int next = (j + 1 < n) ? TC_INPROJ : 0;
    PlmsFuse pf{};
    plms_coefs(h, steps[j], interval, pf.c);
    HeadArgs ha;
    ha.x = x; ha.xs = xs; ha.plms = &pf;
    if (nh == 0) {
      // x' = phi(x, eps_t, t) -> XTMP; eps'' = net(x', max(t - interval, 0)); eps* = (eps_t + eps'') / 2; x = phi(x, eps*, t)
      PlmsFuse p1 = pf;
      plms_weights(0, p1.c);
      p1.eps_store = e0; p1.x_out = h->ws.XTMP;
      ha.flags = TC_HEAD | TC_PLMS | TC_INPROJ; ha.plms = &p1; ha.next_row0 = n;
      DSX_TRY(run_step(h, g, j, 0, h->m.L, ha, s));
      plms_weights(1, pf.c);
      pf.h1 = e0;
      ha.flags = TC_HEAD | TC_PLMS | next; ha.plms = &pf; ha.next_row0 = j + 1;
      DSX_TRY(run_step(h, g, n, 0, h->m.L, ha, s));
    } else {
      plms_weights(nh + 1, pf.c);
      pf.h1 = hist[0];
      pf.h2 = nh >= 2 ? hist[1] : nullptr;
      pf.h3 = nh >= 3 ? hist[2] : nullptr;
      pf.eps_store = e0;
      ha.flags = TC_HEAD | TC_PLMS | next; ha.next_row0 = j + 1;
      DSX_TRY(run_step(h, g, j, 0, h->m.L, ha, s));
    }
    hist[2] = hist[1]; hist[1] = hist[0]; hist[0] = e0;
    nh = std::min(nh + 1, 3);
  }
  return DSX_OK;
}

}  // namespace dsx

using namespace dsx;

extern "C" {

int dsx_version(void) { return DSX_VERSION; }
const char* dsx_last_error(void) { return g_err; }

int dsx_create(int device, dsx_handle** out) {
  DSX_CHECK(out, DSX_E_INVALID, "out is NULL");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error("no CUDA device available (%s); dsx has no CPU fallback", cudaGetErrorString(e));
    return DSX_E_CUDA;
  }
  DSX_CHECK(device >= 0 && device < ndev, DSX_E_INVALID, "device %d out of range (%d devices)", device, ndev);
  DSX_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  DSX_CUDA(cudaGetDeviceProperties(&prop, device));
  dsx_handle* h = new dsx_handle();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  h->tc_group = 2;
  if (prop.major != 10) {
    // the tcgen05 kernels are sm_100a-only; other devices can still run the fp32 path
    h->tc_group = 0;
  }
  if (cudaMalloc(&h->status_dev, sizeof(int)) != cudaSuccess ||
      cudaMallocHost(&h->status_host, sizeof(int)) != cudaSuccess) {
    set_error("status word allocation failed");
    delete h;
    return DSX_E_CUDA;
  }
  cudaMemset(h->status_dev, 0, sizeof(int));
  *h->status_host = 0;
  *out = h;
  return DSX_OK;
}

static void free_model(dsx_handle* h) {
  for (void* p : h->owned) cudaFree(p);
  h->owned.clear();
  h->loaded = false;
}

void dsx_destroy(dsx_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  free_model(h);
  free_ws(h->ws);
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  for (void* p : h->stage)
    if (p) cudaFree(p);
  if (h->trace_dev) cudaFree(h->trace_dev);
  if (h->flags_dev) cudaFree(h->flags_dev);
  if (h->ll_dev) cudaFree(h->ll_dev);
  if (h->status_dev) cudaFree(h->status_dev);
  if (h->status_host) cudaFreeHost(h->status_host);
  delete h;
}

int dsx_load_diffnet(dsx_handle* h, const dsx_diffnet_params* p, int M, int C, int H, int L, int dilation_cycle,
                     int precision, void* stream) {
  DSX_CHECK(h && p, DSX_E_INVALID, "null handle or params");
  DSX_CHECK(M > 0 && C > 0 && H > 0 && L > 0 && dilation_cycle > 0, DSX_E_INVALID, "bad model dimensions");
  DSX_CHECK(C % 16 == 0 && H % 16 == 0 && M % 16 == 0, DSX_E_INVALID, "M, C, H must be multiples of 16 (got %d %d %d)", M, C, H);
  DSX_CHECK(precision == DSX_PREC_FP32_SIMT || precision == DSX_PREC_FP16 || precision == DSX_PREC_FP16X2 ||
                precision == DSX_PREC_FP16X3 || precision == DSX_PREC_FP16S,
            DSX_E_INVALID, "unknown precision %d", precision);
  DSX_CUDA(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  free_model(h);
  free_ws(h->ws);
  h->ws_epoch++;
  h->cond_ready = false;
  h->tm_geom = Geom();
  memset(&h->m, 0, sizeof(h->m));
  h->m.M = M; h->m.C = C; h->m.H = H; h->m.L = L; h->m.cycle = dilation_cycle;
  h->precision = precision;
  if (precision != DSX_PREC_FP32_SIMT) {
    DSX_CHECK(h->tc_group != 0, DSX_E_INVALID, "tcgen05 precisions need an sm_100 device");
    DSX_CHECK(tc_supported(h), DSX_E_INVALID, "tcgen05 path needs residual_channels == hidden_size == 256");
    DSX_CHECK(dilation_cycle <= 4, DSX_E_INVALID,
              "tcgen05 path supports dilations up to 8 (dilation_cycle_length <= 4, got %d); use DSX_PREC_FP32_SIMT", dilation_cycle);
  }
  DSX_TRY(simt_pack_model(h, p, s));
  if (precision != DSX_PREC_FP32_SIMT) DSX_TRY(tc_pack_model(h, s));
  DSX_CUDA(cudaStreamSynchronize(s));
  h->loaded = true;
  return DSX_OK;
}

int dsx_set_schedule(dsx_handle* h, const float* const* bufs, int T) {
  DSX_CHECK(h && bufs && T > 0, DSX_E_INVALID, "bad schedule arguments");
  for (int i = 0; i < DSX_SCH_COUNT; ++i) {
    DSX_CHECK(bufs[i], DSX_E_INVALID, "schedule buffer %d is NULL", i);
    h->sched[i].assign(bufs[i], bufs[i] + T);
  }
  h->sched_T = T;
  return DSX_OK;
}

int dsx_diffnet_forward(dsx_handle* h, const float* x, dsx_strides xs, const int64_t* t, const float* cond,
                        dsx_strides cs, float* eps, int B, int T, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSX_CHECK(x && t && eps, DSX_E_INVALID, "null tensor pointer");
  Geom g;
  DSX_TRY(prepare(h, cond, cs, B, T, B, g, s));
  DSX_TRY(launch_embed_table(h, t, B, s));
  h->want_taps = 1;                      // dsx_debug_read may follow
  DSX_TRY(run_eval(h, x, xs, g, 0, 1, eps, s));
  return check_status(h, s, "dsx_diffnet_forward");
}

int dsx_set_cond(dsx_handle* h, const float* cond, dsx_strides cs, int B, int T, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSX_CHECK(cond, DSX_E_INVALID, "null tensor pointer");
  Geom g;
  DSX_TRY(prepare(h, cond, cs, B, T, 1, g, s));
  return check_status(h, s, "dsx_set_cond");
}

int dsx_plms_update(dsx_handle* h, float* x_out, const float* x_in, const float* const* eps, int mode, int t, int interval,
                    int B, int T, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSX_CHECK(h && h->loaded, DSX_E_STATE, "dsx_load_diffnet has not been called");
  DSX_CHECK(h->sched_T > 0, DSX_E_STATE, "dsx_set_schedule has not been called");
  DSX_CHECK(x_out && x_in && eps && eps[0], DSX_E_INVALID, "null tensor pointer");
  DSX_CHECK(mode >= 0 && mode <= 4 && interval > 0 && t >= 0 && t < h->sched_T && B > 0 && T > 0, DSX_E_INVALID,
            "bad dsx_plms_update arguments (mode %d, t %d, interval %d)", mode, t, interval);
  static const int n_eps[5] = {1, 2, 2, 3, 4};
  for (int i = 0; i < n_eps[mode]; ++i) DSX_CHECK(eps[i], DSX_E_INVALID, "mode %d needs %d eps tensors", mode, n_eps[mode]);
  DSX_CUDA(cudaSetDevice(h->device));
  PlmsCoef c{};
  plms_coefs(h, t, interval, c);
  plms_weights(mode, c);
  const size_t mel = static_cast<size_t>(B) * h->m.M * T;
  return launch_plms_update(h, x_out, x_in, eps[0], n_eps[mode] > 1 ? eps[1] : nullptr, n_eps[mode] > 2 ? eps[2] : nullptr,
                            n_eps[mode] > 3 ? eps[3] : nullptr, c, mel, s);
}

int dsx_sample_ddpm(dsx_handle* h, float* x_inout, const float* cond, dsx_strides cs, int B, int T, int t_start,
                    int n_steps, const float* noise, uint64_t seed, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSX_CHECK(x_inout, DSX_E_INVALID, "null tensor pointer");
  DSX_CHECK(h && h->sched_T > 0, DSX_E_STATE, "dsx_set_schedule has not been called");
  DSX_CHECK(n_steps > 0 && t_start <= h->sched_T && t_start - n_steps >= 0, DSX_E_INVALID,
            "steps t_start=%d n_steps=%d outside schedule of %d", t_start, n_steps, h->sched_T);
  Geom g;
  DSX_TRY(prepare(h, cond, cs, B, T, n_steps + 1, g, s));
  h->want_taps = 0;
  DSX_TRY(sample_ddpm_impl(h, x_inout, g, t_start, n_steps, noise, seed, s));
  return check_status(h, s, "dsx_sample_ddpm");
}

int dsx_sample_plms(dsx_handle* h, float* x_inout, const float* cond, dsx_strides cs, int B, int T, int t_start,
                    int interval, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSX_CHECK(x_inout, DSX_E_INVALID, "null tensor pointer");
  DSX_CHECK(h && h->sched_T > 0, DSX_E_STATE, "dsx_set_schedule has not been called");
  DSX_CHECK(interval > 0 && t_start > 0 && t_start <= h->sched_T, DSX_E_INVALID, "bad PLMS arguments");
  Geom g;
  const int rows = (t_start + interval - 1) / interval + 2;
  DSX_TRY(prepare(h, cond, cs, B, T, rows, g, s));
  h->want_taps = 0;
  DSX_TRY(sample_plms_impl(h, x_inout, g, t_start, interval, s));
  return check_status(h, s, "dsx_sample_plms");
}

int dsx_infer(dsx_handle* h, const float* cond, dsx_strides cs, const float* fs2_mel, const float* start_noise,
              const float* x_start, const float* step_noise, uint64_t seed, const int64_t* mel2ph,
              const float* spec_min, const float* spec_max, int B, int T, int K_step, int pndm_interval,
              float* mel_out, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSX_CHECK(cond && mel_out && spec_min && spec_max, DSX_E_INVALID, "null tensor pointer");
  DSX_CHECK(fs2_mel || x_start, DSX_E_INVALID, "need fs2_mel (shallow start) or x_start (gaussian start)");
  DSX_CHECK(h && h->sched_T > 0, DSX_E_STATE, "dsx_set_schedule has not been called");
  DSX_CHECK(K_step > 0 && K_step <= h->sched_T, DSX_E_INVALID, "K_step %d outside schedule of %d", K_step, h->sched_T);
  Geom g;
  const int rows = pndm_interval > 0 ? (K_step + pndm_interval - 1) / pndm_interval + 2 : K_step + 1;
  DSX_TRY(prepare(h, cond, cs, B, T, rows, g, s));
  h->want_taps = 0;
  const int M = h->m.M;
  const size_t mel = static_cast<size_t>(B) * M * T;
  float* x = h->ws.XSTATE;   // x_t, [B,1,M,T]
  int rc = DSX_OK;
  if (x_start) {
    cudaError_t e = cudaMemcpyAsync(x, x_start, mel * 4, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) { set_error("copy of x_start failed: %s", cudaGetErrorString(e)); rc = DSX_E_CUDA; }
  } else {
    rc = launch_prologue(h, x, fs2_mel, start_noise, seed ^ 0x9E3779B97F4A7C15ull, spec_min, spec_max,
                         h->sched[DSX_SCH_SQRT_ALPHAS_CUMPROD][K_step - 1],
                         h->sched[DSX_SCH_SQRT_ONE_MINUS_ALPHAS_CUMPROD][K_step - 1], B, T, M, s);
  }
  if (rc == DSX_OK)
    rc = pndm_interval > 0 ? sample_plms_impl(h, x, g, K_step, pndm_interval, s)
                           : sample_ddpm_impl(h, x, g, K_step, K_step, step_noise, seed, s);
  if (rc == DSX_OK) rc = launch_epilogue(h, x, mel2ph, spec_min, spec_max, mel_out, B, T, M, s);
  if (rc == DSX_OK) rc = check_status(h, s, "dsx_infer");
  return rc;
}

int dsx_infer_host(dsx_handle* h, const float* cond_host, dsx_strides cs, const float* fs2_mel_host,
                   const float* x_start_host, uint64_t seed, const int64_t* mel2ph_host, const float* spec_min_host,
                   const float* spec_max_host, int B, int T, int K_step, int pndm_interval, float* mel_out_host,
                   void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSX_CHECK(h && h->loaded, DSX_E_STATE, "dsx_load_diffnet has not been called");
  DSX_CHECK(cond_host && mel_out_host && spec_min_host && spec_max_host, DSX_E_INVALID, "null host pointer");
  DSX_CUDA(cudaSetDevice(h->device));
  const int M = h->m.M, H = h->m.H;
  const size_t mel = static_cast<size_t>(B) * M * T;
  // the host cond tensor must be dense in some permutation of [B,H,T]; copy its full extent.  Device staging
  // buffers live in the handle (grow-only) so a call costs copies, not cudaMalloc / cudaFree.
  const size_t cond_elems = static_cast<size_t>(B) * H * T;
  DSX_CHECK(B > 0 && T > 0, DSX_E_INVALID, "B and T must be positive (got %d, %d)", B, T);
  DSX_CHECK(cs.b > 0 && cs.c > 0 && cs.t > 0 &&
                static_cast<size_t>((B - 1) * cs.b + (H - 1) * cs.c + (T - 1) * cs.t) + 1 == cond_elems,
            DSX_E_INVALID, "dsx_infer_host: cond_host must be a dense permutation of a contiguous [B,H,T] block (strides %lld %lld %lld)",
            static_cast<long long>(cs.b), static_cast<long long>(cs.c), static_cast<long long>(cs.t));
  int rc = DSX_OK;
  auto up = [&](int slot, const void* src, size_t bytes) -> void* {
    if (rc != DSX_OK || !src) return nullptr;
    if (h->stage_cap[slot] < bytes) {
      if (h->stage[slot]) cudaFree(h->stage[slot]);
      h->stage[slot] = nullptr;
      h->stage_cap[slot] = 0;
      rc = dev_alloc(h, &h->stage[slot], bytes, false);
      if (rc != DSX_OK) return nullptr;
      h->stage_cap[slot] = bytes;
    }
    if (src != reinterpret_cast<const void*>(1) &&
        cudaMemcpyAsync(h->stage[slot], src, bytes, cudaMemcpyHostToDevice, s) != cudaSuccess) {
      set_error("host->device copy failed");
      rc = DSX_E_CUDA;
    }
    return h->stage[slot];
  };
  float* d_cond = static_cast<float*>(up(0, cond_host, cond_elems * 4));
  float* d_fs2 = static_cast<float*>(up(1, fs2_mel_host, mel * 4));
  float* d_x = static_cast<float*>(up(2, x_start_host, mel * 4));
  float* d_min = static_cast<float*>(up(3, spec_min_host, M * 4));
  float* d_max = static_cast<float*>(up(4, spec_max_host, M * 4));
  int64_t* d_m2p = static_cast<int64_t*>(up(5, mel2ph_host, static_cast<size_t>(B) * T * 8));
  float* d_out = static_cast<float*>(up(6, reinterpret_cast<const void*>(1), mel * 4));   // output buffer only
  if (rc == DSX_OK)
    rc = dsx_infer(h, d_cond, cs, d_fs2, nullptr, d_x, nullptr, seed, d_m2p, d_min, d_max, B, T, K_step, pndm_interval,
                   d_out, stream);
  if (rc == DSX_OK && cudaMemcpyAsync(mel_out_host, d_out, mel * 4, cudaMemcpyDeviceToHost, s) != cudaSuccess) {
    set_error("device->host copy failed");
    rc = DSX_E_CUDA;
  }
  cudaStreamSynchronize(s);
  return rc;
}

int dsx_get_info(dsx_handle* h, int what, int64_t* out) {
  DSX_CHECK(h && out, DSX_E_INVALID, "null argument");
  switch (what) {
    case DSX_INFO_PRECISION: *out = h->precision; break;
    case DSX_INFO_KERNEL_LAUNCHES: *out = h->launches; break;
    case DSX_INFO_WORKSPACE_BYTES: *out = static_cast<int64_t>(h->ws.bytes); break;
    case DSX_INFO_SM_COUNT: *out = h->sm_count; break;
    case DSX_INFO_TC_CTA_GROUP: *out = h->tc_group; break;
    case DSX_INFO_LAYER_KERNEL_LAUNCHES: *out = static_cast<int64_t>(h->prof_used / 2); break;
    case DSX_INFO_STACK_MODE: *out = h->stack_mode; break;
    case DSX_INFO_CLUSTER_OCCUPANCY: *out = h->cluster_occ; break;
    case DSX_INFO_STACK_KERNEL_LAUNCHES: *out = h->stack_launches; break;
    case DSX_INFO_STACK_ROWS: *out = h->stack_rows_used; break;
    case DSX_INFO_LAYER_KERNEL_NS: {
      double total_ms = 0;
      for (size_t i = 0; i + 1 < h->prof_used; i += 2) {
        float ms = 0.f;
        DSX_CUDA(cudaEventSynchronize(h->prof_events[i + 1]));
        DSX_CUDA(cudaEventElapsedTime(&ms, h->prof_events[i], h->prof_events[i + 1]));
        total_ms += ms;
      }
      *out = static_cast<int64_t>(total_ms * 1e6);
      break;
    }
    default: set_error("unknown info %d", what); return DSX_E_INVALID;
  }
  return DSX_OK;
}

int dsx_set_option(dsx_handle* h, int what, int64_t value) {
  DSX_CHECK(h, DSX_E_INVALID, "null handle");
  switch (what) {
    case DSX_OPT_TC_CTA_GROUP:
      DSX_CHECK(value == 2, DSX_E_INVALID, "the residual-layer kernel is cta_group::2 only (cta_group::1 is exercised by dsx_selftest)");
      DSX_CHECK(h->tc_group != 0, DSX_E_INVALID, "no tcgen05 on this device");
      h->tc_group = static_cast<int>(value);
      break;
    case DSX_OPT_CP_PREFETCH: h->cp_prefetch = static_cast<int>(value); break;
    case DSX_OPT_STACK_MODE: h->stack_mode = static_cast<int>(value); break;
    case DSX_OPT_STACK_KERNEL: h->stack_kernel = static_cast<int>(value); break;
    case DSX_OPT_GATE_APPROX: h->gate_approx = static_cast<int>(value); break;
    case DSX_OPT_FUSED_HEAD: h->fused_head = static_cast<int>(value); break;
    case DSX_OPT_STACK_ROWS:
      DSX_CHECK(value == 0 || value == 64 || value == 128, DSX_E_INVALID, "DSX_OPT_STACK_ROWS must be 0 (automatic), 64 or 128");
      h->stack_rows = static_cast<int>(value);
      break;
    case DSX_OPT_BATCH_OFFSET:
      DSX_CHECK(value >= 0 && value < (1ll << 30), DSX_E_INVALID, "DSX_OPT_BATCH_OFFSET out of range");
      h->batch_offset = static_cast<int>(value);
      break;
    case DSX_OPT_SR_SETS:
      DSX_CHECK(value >= 1 && value <= 1024, DSX_E_INVALID, "DSX_OPT_SR_SETS must be in [1, 1024]");
      h->sr_sets = static_cast<int>(value);
      break;
    case DSX_OPT_PROFILE:
      h->profile = static_cast<int>(value);
      h->prof_used = 0;
      break;
    default: set_error("unknown option %d", what); return DSX_E_INVALID;
  }
  return DSX_OK;
}

int dsx_debug_read(dsx_handle* h, int which, float* out, int B, int T, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSX_CHECK(h && out && h->ws.X, DSX_E_STATE, "no workspace");
  DSX_CHECK(B == h->ws.g.B && T == h->ws.g.T, DSX_E_INVALID, "geometry mismatch");
  const float* src = which == 0 ? h->ws.X : h->ws.SKIP;
  const int C = h->m.C;
  DSX_CUDA(cudaMemcpy2DAsync(out, static_cast<size_t>(T) * C * 4, src, static_cast<size_t>(h->ws.g.Tp) * C * 4,
                             static_cast<size_t>(T) * C * 4, B, cudaMemcpyDeviceToDevice, s));
  return DSX_OK;
}

int dsx_debug_trace(dsx_handle* h, int enable, int64_t* out_host) {
  DSX_CHECK(h, DSX_E_INVALID, "null handle");
  DSX_CUDA(cudaSetDevice(h->device));
  const size_t bytes = 10 * 256 * sizeof(long long);       // [2][3][256] role stamps, then [256][4] per-CTA entry / exit
  if (out_host && h->trace_dev) {
    DSX_CUDA(cudaDeviceSynchronize());
    DSX_CUDA(cudaMemcpy(out_host, h->trace_dev, (enable == 2 ? 10 : 6) * 256 * sizeof(long long), cudaMemcpyDeviceToHost));
  }
  if (enable && !h->trace_dev) {
    DSX_CUDA(cudaMalloc(&h->trace_dev, bytes));
    DSX_CUDA(cudaMemset(h->trace_dev, 0, bytes));
  } else if (!enable && h->trace_dev) {
    DSX_CUDA(cudaDeviceSynchronize());
    cudaFree(h->trace_dev);
    h->trace_dev = nullptr;
  }
  return DSX_OK;
}

int dsx_debug_set_layer_limit(dsx_handle* h, int n_layers) {
  DSX_CHECK(h, DSX_E_INVALID, "null handle");
  h->layer_limit = n_layers;
  return DSX_OK;
}

}  // extern "C"
