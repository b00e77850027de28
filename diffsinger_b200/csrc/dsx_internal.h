// Internal declarations shared by the dsx translation units (not part of the C ABI).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/dsx.h"

namespace dsx {

void set_error(const char* fmt, ...);
#define DSX_CUDA(expr)                                                                        \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      ::dsx::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return DSX_E_CUDA;                                                                      \
    }                                                                                         \
  } while (0)
#define DSX_CHECK(cond, code, ...)     \
  do {                                 \
    if (!(cond)) {                     \
      ::dsx::set_error(__VA_ARGS__);   \
      return (code);                   \
    }                                  \
  } while (0)
#define DSX_TRY(expr)          \
  do {                         \
    int _r = (expr);           \
    if (_r != DSX_OK) return _r; \
  } while (0)

constexpr int kTile = 128;  // frames per tile (= UMMA M per CTA)
constexpr int kStackRowsPerLayer = 64 * 256;      // rows per layer of the stack kernel's hi / lo weight pack (fp16 / fp16x2)
constexpr int kStackSetRowsPerLayer = 32 * 256;   // rows (of 64 fp16) per layer of one stochastically rounded weight set

// Geometry of one call: B utterances of T frames, stored frames-major with the frame axis
// padded to a multiple of the tile so tiles never straddle utterances.
struct Geom {
  int B = 0, T = 0, Tp = 0, tiles_per_utt = 0, tiles = 0;
  void set(int b, int t) {
    B = b;
    T = t;
    tiles_per_utt = (t + kTile - 1) / kTile;
    Tp = tiles_per_utt * kTile;
    tiles = B * tiles_per_utt;
  }
  size_t frames_padded() const { return static_cast<size_t>(B) * Tp; }
};

// Device-side model description handed to kernels.
struct ModelDev {
  int M, C, H, L, cycle;
  // fp32, SIMT layouts
  const float* in_w;   // [C][M]
  const float* in_b;   // [C]
  const float* mlp0_w; // [4C][C]
  const float* mlp0_b;
  const float* mlp2_w; // [C][4C]
  const float* mlp2_b;
  const float* dif_w;  // [L][C][C]
  const float* dif_b;  // [L][C]
  const float* w1f;    // [L][2C][3C+H]   k = tap*C + c | 3C + h
  const float* b1f;    // [L][2C]         dil_b + cond_b
  const float* w2f;    // [L][2C][C]
  const float* b2f;    // [L][2C]
  const float* skip_w; // [C][C]
  const float* skip_b;
  const float* fin_w;  // [M][C]
  const float* fin_b;
  // tcgen05 packs (fp16, 128-byte rows of 64 k-values; see dsx_tc.cu for the tile order)
  const __half* wpack; // [L][20480 rows][64]
  const float* b1p;    // [L][2 chunks][256]  gate(128) | filter(128) per chunk
  const __half* whead; // [32 tiles][128 rows][64]: skip_projection, output_projection, input_projection packs
  const float* bskip;  // [L][256] prefix sums over layers of the skip-half biases of output_projection (stack kernel)
  const __half* wstk;  // [L][16384 rows][64] hi / lo planes in the stack kernel's row order (DSX_PREC_FP16 / FP16X2), or nullptr
  const __half* wsr;   // [R][L][8192 rows][64] stochastically rounded weight sets (DSX_PREC_FP16S), or nullptr
  int wsr_sets;        // R
};

struct Workspace {
  Geom g;               // capacity geometry (B, Tp) currently allocated
  int rows_cap = 0;     // step-table rows
  float* X = nullptr;       // [B][Tp][C] residual stream
  float* SKIP = nullptr;    // [B][Tp][C]
  float* CONDF = nullptr;   // [B][Tp][H] fp32 (SIMT path)
  float* G1 = nullptr;      // [B][Tp][2C] SIMT GEMM output scratch
  float* Zf = nullptr;      // [B][Tp][C]  SIMT gate output
  __half* Y = nullptr;      // [2 buffers][2 planes][B][Tp][C]
  __half* CONDH = nullptr;  // [2 planes][B][Tp][H]
  float* CP = nullptr;      // [L][tiles][2][64][128][4] conditioner projection + bias of every layer (tcgen05 path)
  __half* S16 = nullptr;    // [2 planes][B][Tp][C] skip_sum / sqrt(L), operand of the head GEMM
  __half* Z = nullptr;      // [L][B][Tp][C] gate outputs z of every layer (stack kernel: A operand of the deferred skip GEMM)
  float* DTAB = nullptr;    // [rows][L][C]
  float* EMB = nullptr;     // [rows][C] scratch (mlp output)
  int64_t* TVALS = nullptr; // [rows]
  float* EPS = nullptr;     // [5][B][M][T] current + PLMS history ring
  float* XTMP = nullptr;    // [B][M][T] PLMS warm-up state
  float* XSTATE = nullptr;  // [B][M][T] mel state of dsx_infer
  size_t bytes = 0;
  // byte capacities (grow-only)
  size_t cap_X = 0, cap_SKIP = 0, cap_CONDF = 0, cap_G1 = 0, cap_Zf = 0, cap_Y = 0, cap_CONDH = 0, cap_CP = 0, cap_S16 = 0, cap_Z = 0,
         cap_DTAB = 0, cap_EMB = 0, cap_TVALS = 0, cap_EPS = 0, cap_XTMP = 0, cap_XSTATE = 0;
};

}  // namespace dsx

struct dsx_handle {
  int device = 0;
  int sm_count = 0;
  bool loaded = false;
  int precision = DSX_PREC_FP32_SIMT;
  int tc_group = 1;
  int layer_limit = -1;
  int64_t launches = 0;
  int64_t stack_launches = 0;   // launches of k_tc_stack (dsx_stack.cu)
  dsx::ModelDev m{};
  std::vector<void*> owned;   // device allocations of the model
  int sched_T = 0;
  std::vector<float> sched[DSX_SCH_COUNT];
  dsx::Workspace ws;
  int* status_dev = nullptr;   // kernel watchdog / self-check word
  int* status_host = nullptr;  // pinned mirror
  CUtensorMap tm_w{}, tm_y[2][2]{}, tm_yh[2]{}, tm_ye[2]{}, tm_cond[2]{}, tm_s16[2]{}, tm_whead{}, tm_wsr{}, tm_wstk{}, tm_z{};
  CUtensorMap tm_y0s[2]{}, tm_zs[2]{}, tm_s16s[2][2]{}, tm_xst[2]{}, tm_y0st[2]{};   // stack kernel, [0]: 128 rows per CTA, [1]: 64 rows per CTA
  dsx::Geom tm_geom;           // geometry the activation maps were built for
  int profile = 0;
  void* stage[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // dsx_infer_host device staging
  size_t stage_cap[7] = {0, 0, 0, 0, 0, 0, 0};
  unsigned int* flags_dev = nullptr;   // per-tile publish counters of the stack kernel
  int flags_cap = 0;
  int flags_geom_b = 0, flags_geom_t = 0;   // geometry of the last stack launch
  unsigned int flag_count = 0;         // value of every counter before the next stack launch
  void* ll_dev = nullptr;              // halo packets of the stack kernel (dsx_stack.cu)
  size_t ll_cap = 0;
  unsigned int ll_seq = 1;             // next sequence number (monotonic, never 0)
  int flags_kind = 0;                  // which kernel's counting convention the counters follow (1: k_tc_layer, 2: k_tc_stack)
  int stack_kernel = 1;                // DSX_OPT_STACK_KERNEL: 1 = register-resident stack kernel (dsx_stack.cu) where it applies
  int stack_occ[2][2] = {};            // co-resident CTA pairs of k_tc_stack<WP, R> [WP - 1][R == 64] (0 unknown, -1 none)
  bool attr_stack[2][2] = {};
  int fused_head = 1;                  // DSX_OPT_FUSED_HEAD: the head / sampler update / next input projection run inside the stack launch
  int stack_rows = 0;                  // DSX_OPT_STACK_ROWS: 0 = automatic, 64 / 128 forced
  int stack_rows_used = 0;             // rows per CTA of the last stack launch
  int sr_sets = 64;                    // DSX_OPT_SR_SETS: weight sets of DSX_PREC_FP16S (takes effect at the next dsx_load_diffnet)
  unsigned long long sr_seed = 0x5DEECE66Dull;
  unsigned long long ws_epoch = 0;     // bumped whenever a workspace buffer moves (tensor maps are rebuilt)
  unsigned long long tm_epoch = ~0ull;
  bool cond_ready = false;             // CONDH / CP (or CONDF) hold the conditioner of dsx_set_cond for geometry cond_geom
  dsx::Geom cond_geom;
  int gate_approx = -1;                // DSX_OPT_GATE_APPROX: -1 = default (tanh.approx gate), 0 / 1 forced
  int want_taps = 1;                   // the next stack launches write X / SKIP back (dsx_diffnet_forward: yes, sampling loops: no)
  int batch_offset = 0;                // DSX_OPT_BATCH_OFFSET: global index of utterance 0 in the Philox noise counters
  bool attr_layer[3] = {false, false, false}, attr_head[2] = {false, false}, attr_cond = false;
  int occ_cache[3][17] = {};
  int cluster_occ = 0;              // max co-resident utterance clusters reported by the driver (last launch)
  int cp_prefetch = 1;              // tuning knob (DSX_OPT_CP_PREFETCH)
  int stack_mode = 1;               // 1: all residual layers of an evaluation in one cluster-per-utterance launch
  int trace_seq = 0;                // debug: running index of traced launches
  long long* trace_dev = nullptr;   // debug timeline buffer (dsx_debug_trace)
  std::vector<cudaEvent_t> prof_events;   // pairs (start, stop), prof_used of them recorded
  size_t prof_used = 0;
};

namespace dsx {

// ---- dsx_simt.cu -------------------------------------------------------------------------
int simt_pack_model(dsx_handle* h, const dsx_diffnet_params* p, cudaStream_t s);
int launch_embed_table(dsx_handle* h, const int64_t* t_dev, int rows, cudaStream_t s);
int launch_pack_cond(dsx_handle* h, const float* cond, dsx_strides cs, const Geom& g, cudaStream_t s);
int launch_inproj(dsx_handle* h, const float* x, dsx_strides xs, const Geom& g, cudaStream_t s);
int launch_simt_layer(dsx_handle* h, int layer, const Geom& g, int row0, int row_per_b, cudaStream_t s);
int launch_head(dsx_handle* h, const Geom& g, float* eps, cudaStream_t s);
struct DdpmCoef { float A, Bc, c1, c2, sigma; };
int launch_ddpm_update(dsx_handle* h, float* x, const float* eps, const float* noise, uint64_t seed,
                       uint64_t offset, DdpmCoef c, size_t n, int T, cudaStream_t s);
struct PlmsCoef { float kx, ke, a_diff, denom, w0, w1, w2, w3; };   // see k_plms_update
int launch_plms_update(dsx_handle* h, float* x_out, const float* x_in, const float* e0, const float* e1,
                       const float* e2, const float* e3, PlmsCoef c, size_t n, cudaStream_t s);
int launch_prologue(dsx_handle* h, float* x, const float* fs2_mel, const float* start_noise, uint64_t seed,
                    const float* spec_min, const float* spec_max, float sa, float s1a, int B, int T, int M,
                    cudaStream_t s);
int launch_epilogue(dsx_handle* h, const float* x, const int64_t* mel2ph, const float* spec_min,
                    const float* spec_max, float* mel_out, int B, int T, int M, cudaStream_t s);

// ---- dsx_tc.cu ---------------------------------------------------------------------------
int tc_pack_model(dsx_handle* h, cudaStream_t s);
int tc_prepare_maps(dsx_handle* h, const Geom& g);
int launch_tc_condproj(dsx_handle* h, const Geom& g, cudaStream_t s);
int launch_tc_layers(dsx_handle* h, int l0, int l1, const Geom& g, int row0, int row_per_b, cudaStream_t s);
// What follows the residual stack in a diffusion step: TC_HEAD = head (skip -> eps), TC_WRITE_EPS = write eps, TC_UPDATE = DDPM
// update of x, TC_PLMS = PNDM update of x (PlmsFuse), TC_INPROJ = input projection of x (after the update if any) for the
// evaluation that uses table row (next_row0, row_per_b).
enum { TC_HEAD = 1, TC_WRITE_EPS = 2, TC_UPDATE = 4, TC_INPROJ = 8, TC_PLMS = 16 };
// PNDM update fused into the head kernel (TC_PLMS): eps' = (w0 eps_t + w1 h1 + w2 h2 + w3 h3) / denom, x_out = phi(x, eps', t)
// (usr/diff/shallow_diffusion_tts.py:174-199); eps_t is also stored to `eps_store` (history ring) when non-null.
struct PlmsFuse {
  PlmsCoef c;
  const float* h1;
  const float* h2;
  const float* h3;   // earlier eps, most recent first, contiguous [B][M][T] (or null)
  float* eps_store;  // this evaluation's eps -> history ring slot (or null)
  float* x_out;      // result; null: in place
};
// The same description serves the head fused into k_tc_stack, k_tc_head and the fp32 path's separate launches
struct HeadArgs {
  int flags = 0;            // TC_* (0: no head)
  float* x = nullptr;       // mel state
  dsx_strides xs{};
  float* eps = nullptr;     // TC_WRITE_EPS
  const float* noise = nullptr;
  uint64_t seed = 0, offset = 0;
  DdpmCoef c{};
  int next_row0 = 0, row_per_b = 0;   // FiLM table row of the NEXT evaluation (TC_INPROJ)
  const PlmsFuse* plms = nullptr;
};
int launch_tc_head(dsx_handle* h, const Geom& g, const HeadArgs& ha, cudaStream_t s);
bool tc_supported(const dsx_handle* h);
int ensure_flags(dsx_handle* h, int n);
int make_map_2d(CUtensorMap* m, const void* base, uint64_t rows, uint32_t box_rows);
void reset_flags(dsx_handle* h);

// ---- dsx_stack.cu ------------------------------------------------------------------------
int tc_stack_pack(dsx_handle* h, cudaStream_t s);
bool tc_stack_usable(dsx_handle* h, const Geom& g);
int launch_tc_stack(dsx_handle* h, int nl, const Geom& g, int row0, int row_per_b, int wset, cudaStream_t s,
                    const HeadArgs* head = nullptr);

int dev_alloc(dsx_handle* h, void** p, size_t bytes, bool model_owned);
int ensure_workspace(dsx_handle* h, const Geom& g, int rows, cudaStream_t s);
int check_status(dsx_handle* h, cudaStream_t s, const char* what);

}  // namespace dsx
