// k_tc_stack<WP>: all residual layers of one DiffNet evaluation (usr/diff/net.py:58-78,121-126) in one persistent launch,
// with the residual stream in REGISTERS and the conv input y in SHARED MEMORY for the whole stack.  Per 128-frame tile
// (one CTA; two CTAs form a cta_group::2 pair, UMMA M = 256, N = 256) and layer l:
//
//   GEMM1   D1[:, chunk h] = [y(t-d) | y(t) | y(t+d)] (K = 768) . W1(h)^T      -> TMEM F0 (h = 0), F1 (h = 1); the centre
//                                                                                  taps of both chunks first, the halo taps last
//   epi1    z(chunk h) = sigmoid(D1 gate + CP) * tanh(D1 filter + CP) -> fp16, swizzled K-major rows in shared memory
//           (chunk 0 drains F0 under chunk 1's MMAs)
//   GEMM2r  D2res = z (K = 256) . W2res^T                                        -> F0 (k-blocks 0, 1 under epi1 of chunk 1)
//   epi2    x <- (x + D2res + b) / sqrt2   (x: 128 fp32 registers per epilogue thread = one frame row x 128 channels)
//           y_{l+1} = fp16(x + d_{l+1})    -> straight into the next layer's A-operand tiles in shared memory; the 8 first /
//                                              last rows of the tile are also sent to the neighbour tiles (halo rows of the
//                                              dilated taps) as self-validating {data, sequence} packets, see below
//   z_l     -> HBM by TMA store (64 KB per tile and layer)
// and after the last layer ONE deferred GEMM for the skip path (net.py:126 sums the skip halves of all layers, which is a
// single contraction over K = L * 256):
//   SKIP    = [z_0 | z_1 | ... | z_{L-1}] (K = 20 * 256) . [W2skip_0; ...; W2skip_{L-1}]^T   -> F1, read once
// so the per-layer critical path carries no skip work at all (no accumulator, no epilogue, no red.add traffic).
//
// Compared with the round-1 layer kernel (dsx_tc.cu, k_tc_layer) this removes, per layer and tile, the fp32 read-modify-
// write of x through L2 (256 KB), the skip red.add (128 KB), the y round trip through L2 (64 KB + 144 KB of TMA loads) and
// the transposing staging pass; the layer hand-over inside a tile is a shared-memory barrier instead of a global flag round
// trip.  Halo exchange between neighbouring tiles (different CTA pairs): every 16-byte packet in global memory carries 8
// bytes of fp16 data and two copies of a per-layer sequence number (the scheme NCCL's LL protocol uses); the receiving
// epilogue warps poll the packets themselves right after their own epi2, so there is no publish counter, no fence and no
// second round trip, and the ~2k cycles of latency hide under the centre-tap MMAs of the next layer.
//
// Shared memory: [W ring 5 x 16 KB | y: 4 k-blocks x (8 halo + 128 + 8 halo rows) x 128 B | z: 4 k-blocks x 16 KB |
//                 per-layer bias / FiLM vectors (1 KB per epilogue warp) | barriers]; the deferred skip GEMM streams its A
// tiles (z of every layer) through the z and y areas.
// TMEM: F0, F1 (256 columns each).
// Small batches run the same kernel with 64 rows per CTA (UMMA M = 128: twice the CTAs; the accumulators then take 128 TMEM
// columns each, so the skip half gets a third accumulator and is summed inside the layers instead of deferred), see StackCfg.
//
// Scheduling (what the clock64 timelines in profiles/ led to): the next layer's centre taps and GEMM2's k-block 2 start
// half an epilogue phase early (yhalf / zhalf: an epilogue warp finishes its first 64-channel k-block, signals, then does its
// second); the L2 prefetch of the conditioner stream is PACED over the layer and every CTA prefetches its share of the weight
// block two layers ahead, so that the first weight tiles of a layer do not queue at HBM behind a 33 MB prefetch burst; the
// epilogue warps load x only after the producers' first TMA loads are on their way.
// Roles (384 threads): warp 0 lane 0 = activation producer (layer-0 slots, z stores, CP prefetch, A tiles of the skip GEMM),
// warps 2, 3 lane 0 = weight producers, warp 1 lane 0 of the pair leader = MMA issuer, warps 4-11 = epilogue (thread = frame
// row = TMEM lane, two warps per lane quadrant split the 256 columns).  setmaxnreg moves registers from warps 0-3 to the
// epilogue warps (x lives there).
//
// Weight tiles: WP = 2 reads the hi and lo planes of the round-1 pack (fp16x2 parity mode); WP = 1 reads one plane -- either
// the round-to-nearest hi plane (fp16 fast mode) or one of R stochastically rounded weight sets, a different one at every
// diffusion step (fp16s mode: the rounding error of the weights then decorrelates across steps instead of accumulating).
#include <cuda.h>
#include <string.h>

#include <algorithm>

#include "dsx_internal.h"
#include "dsx_ptx.cuh"
#include "dsx_rng.cuh"
#include "dsx_tc_common.cuh"
#include "dsx_update.cuh"

namespace dsx {

// Rows per CTA.  R = 128: UMMA M = 256, accumulator lane = frame row, column = N index.  R = 64 (small batches: twice the CTAs,
// half the MMA and epilogue time per layer): UMMA M = 128, whose cta_group::2 accumulator holds the FIRST half of N in lanes
// 0-63 and the SECOND half in lanes 64-127 (columns 0 .. N/2-1).  The weight rows of GEMM1 are ordered so that a channel's
// gate and filter land in the same lane either way: N index = g * 128 + j with j < 64 -> gate of chunk-channel g * 64 + j,
// j >= 64 -> filter of chunk-channel g * 64 + j - 64 (k_pack_wstk / k_pack_wsr).
template <int R>
struct StackCfg {
  static constexpr int UNIT = R * 128;                      // one A k-block tile of this CTA: R rows x 64 fp16
  static constexpr int YSLOT = (R + 16) * 128;              // [8 halo | R centre | 8 halo] rows of 64 channels
  static constexpr int WSLOTS = (R == 128) ? 5 : 8;
  static constexpr int W_BYTES = WSLOTS * kUnitBytes;       // weight tiles are 128 rows x 64 per CTA in both modes
  static constexpr int Y_BYTES = 4 * YSLOT;
  static constexpr int Z_BYTES = 4 * UNIT;
  static constexpr int ASLOTS = 8;                          // A ring of the skip GEMM: 4 units in the z area + 4 in the y area
  static constexpr int TAB_BYTES = kEpiWarps * 1024;       // per epilogue warp: [bias | d_next] fp32 of its channels
  static constexpr int BAR_BYTES = 512;
  static constexpr int SMEM_BYTES = 1024 + W_BYTES + Y_BYTES + Z_BYTES + TAB_BYTES + BAR_BYTES;
  static constexpr int REGS_LOW = 56, REGS_HIGH = 224;     // setmaxnreg targets: 128 * 56 + 256 * 224 = 64512 = 384 * 168 (the
                                                            // CTA's register pool is its launch allocation)
  static constexpr int F1_COL = (R == 128) ? 256 : 128;     // TMEM column of the second accumulator
  // The skip-sum accumulator.  R = 128: F1 itself (TMEM is full: two N = 256 accumulators of 256 columns), so the skip GEMM is
  // DEFERRED to one K = L * 256 contraction after the last layer.  R = 64: an N = 256 accumulator takes 128 columns, columns
  // 256-383 are free -- the skip half of every layer accumulates there right after its GEMM2, in the tensor pipe's idle time
  // under the residual epilogue: no deferred GEMM (54 k of 491 k cycles per launch at B = 1, T = 512) and no z round trip.
  static constexpr int SKIP_COL = 256;
  static constexpr bool SKIP_IN_LAYER = (R == 64);
  static constexpr int NCH = R;                             // channels (N indices) per epilogue thread in epi2 / exit
  static constexpr int NSP = R / 16;                        // gate sub-passes (8 channels each) per chunk and thread
  static_assert(R == 128 || R == 64, "rows per CTA");
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
  static_assert(YSLOT % 1024 == 0 && UNIT % 1024 == 0, "tiles must keep the 1024-byte swizzle atoms aligned");
  static_assert(Y_BYTES >= 4 * UNIT, "A ring units in the y area");
  static_assert(W_BYTES + Y_BYTES + Z_BYTES >= 12 * UNIT, "exit tiles of the fused head (8 fp32 + 4 fp16 units) over the W / y / z areas");
};

struct TcStackParams {
  CUtensorMap tm_w;        // weight tiles, 2D [rows][64], box 64 x 128 rows
  CUtensorMap tm_y0;       // Y buffer 0 (written by the input projection), box 64 ch x (R + 16) frames: layer 0 incl. halos
  CUtensorMap tm_z;        // Z [L * B][T][256] fp16, box 64 ch x R frames: z of every layer (store per layer, load for the skip GEMM)
  CUtensorMap tm_s16[2];   // S16 hi / lo planes [B][T][256], box 64 ch x R frames (TMA store at exit)
  float* X;                // [B][Tp][256] residual stream: read at entry, written back at exit (taps)
  float* SKIP;             // [B][Tp][256] skip sum (debug tap / fp32 copy), written at exit (taps)
  uint4* ll;               // halo packets [tiles][2 layer parities][2 sides: first / last 8 rows][512] x 16 B:
                           // {fp16 x2, seq, fp16 x2, seq}, packet = 4 channels of one row (row * 64 + channel / 4)
  unsigned int seq_base;   // sequence number of layer l's y: seq_base + l (monotonic over the handle's lifetime, never 0)
  const float* CP;         // [L][128-frame tiles][2 chunks][64 column groups][128 rows][4] conditioner projection + biases
  int cp_tiles;            // 128-frame tiles of the call (CP stride)
  int cp_prefetch;
  const float* b2;         // [L][512] output_projection bias (residual half | skip half)
  const float* bskip;      // [L][256] prefix sums over layers of the skip-half biases
  const float* dtab;       // FiLM rows of this evaluation: [L][256], utterance b at + b * d_row_stride
  int d_row_stride;
  int T, Tp, tiles_per_utt, B;   // tiles_per_utt: R-frame tiles per utterance (Tp / R)
  int tile0, tile_end;     // this launch covers tiles [tile0, tile_end) (whole utterances); CTA i -> tile tile0 + i
  int nl, L, cycle;        // layers [0, nl); dilation of layer l = 1 << (l % cycle)
  const void* wbase;       // the array behind tm_w (rows of 64 fp16): L2 prefetch of the next layer's tiles
  int w_row0;              // first row of this evaluation's weight set in tm_w
  int w_layer_rows;        // rows per layer
  int w_sr;                // 0: hi / lo planes (64 tiles per layer); 1: single-plane stochastically rounded set (32 tiles per layer)
  float inv_sqrt_l;
  int fast_act;            // 1: tanh.approx gate
  int taps;                // 1: write the residual stream and the fp32 skip sum back to X / SKIP at exit (debug taps of
                           // dsx_diffnet_forward); the sampling loops do not need them
  // ---- fused head (head_flags != 0; flags as for k_tc_head): skip / output projections (net.py:115-118, 126-130), the sampler
  //      update on the mel state (shallow_diffusion_tts.py:134-204) and the next evaluation's input projection -- the rest of
  //      the diffusion step runs in this launch too: ONE kernel per step ----
  int head_flags;
  CUtensorMap tm_wh;       // whead tiles [32][128 rows][64]: skip_projection, output_projection, input_projection packs
  CUtensorMap tm_xst;      // X fp32 [B][T][256], box 32 ch x R frames, SWIZZLE_128B: store of the next evaluation's x0
  CUtensorMap tm_y0st;     // Y buffer 0 fp16, box 64 ch x R frames: store of the next evaluation's layer-0 conv input
  float* xmel;             // mel state [B,1,M,T] through xs (in / out)
  dsx_strides xs;
  float* eps_out;          // TC_WRITE_EPS: [B][M][T]
  const float* noise;      // [B][M][T] for this step, or nullptr -> Philox
  unsigned long long seed, offset;
  int b_off;
  DdpmCoef c;
  PlmsFuse pl;
  const float* bs;         // skip_projection.bias [256]
  const float* bf;         // output_projection.bias [M]
  const float* bin;        // input_projection.bias [256]
  const float* d0;         // FiLM vector of layer 0 for the NEXT evaluation, utterance b at + b * d0_row_stride
  int d0_row_stride;
  int M;
  int* status;
  unsigned long long budget_ns;
  long long* trace;        // debug: [2 CTAs][3 roles][256] clock64 stamps, or nullptr
};

#define DSX_STRACE(role, slot)                                                         \
  do {                                                                                 \
    if (p.trace && blockIdx.x < 2 && (slot) < 256)                                      \
      p.trace[(blockIdx.x * 3 + (role)) * 256 + (slot)] = clock64();                   \
  } while (0)

template <int WP, int R>
__global__ void __launch_bounds__(kThreads, 1) k_tc_stack(const __grid_constant__ TcStackParams p) {
  using Cfg = StackCfg<R>;
  if (p.trace && threadIdx.x == 0 && blockIdx.x < 256) {      // debug timeline: per-CTA entry (wall clock ns, SM cycles)
    p.trace[6 * 256 + blockIdx.x * 4] = static_cast<long long>(globaltimer_ns());
    p.trace[6 * 256 + blockIdx.x * 4 + 1] = clock64();
  }
  constexpr int G = kG;
  constexpr int WS = Cfg::WSLOTS;
  constexpr int AS = Cfg::ASLOTS;
  constexpr int UNIT = Cfg::UNIT;
  extern __shared__ uint8_t smem_raw[];
  // (pointer arithmetic on the __shared__ array, not an integer round trip: keeps the address space visible to the compiler,
  //  which otherwise emits generic LD / ST for every table load and tile store of the epilogues)
  uint8_t* wring = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* yslots = wring + Cfg::W_BYTES;
  uint8_t* zbuf = yslots + Cfg::Y_BYTES;
  float* tab = reinterpret_cast<float*>(zbuf + Cfg::Z_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(tab) + Cfg::TAB_BYTES);
  uint64_t* full = bars;            // [WS] weight tile landed (both CTAs' halves; leader's barrier)
  uint64_t* empty = full + WS;      // [WS] weight tile consumed (tcgen05.commit, both CTAs)
  uint64_t* tfull = empty + WS;     // [2] accumulator F0 / F1 complete -> epilogue
  uint64_t* tempty = tfull + 2;     // [2] epilogue phase on F0 / F1 done (drained, its z / y written), 8 warps x 2 CTAs -> leader
  uint64_t* y0full = tempty + 2;    // layer 0: the whole y slots landed by TMA (leader's barrier)
  uint64_t* yhalo = y0full + 1;     // halo rows of the layer received and written by the epilogue warps, 8 warps x 2 CTAs -> leader
  uint64_t* zdone = yhalo + 1;      // this CTA's 8 epilogue warps have written z of the layer (local)
  uint64_t* zfree = zdone + 1;      // the TMA store of z has finished reading it (local)
  uint64_t* lfin = zfree + 1;       // every MMA of the layers complete: z / y areas become the A ring of the skip GEMM
  uint64_t* afull = lfin + 1;       // [AS] A tile of the skip GEMM landed (leader's barrier)
  uint64_t* aempty = afull + AS;    // [AS]
  uint64_t* sdone = aempty + AS;    // exit: this CTA's 8 epilogue warps have written the S16 tiles (local)
  uint64_t* yhalf = sdone + 1;      // R = 128: k-blocks 0 and 2 of y_{l+1} written (first half of epi2), 8 warps x 2 CTAs -> leader
  uint64_t* zhalf = yhalf + 1;      // R = 128: z k-block 2 written (first half of chunk 1's gate epilogue), 8 warps x 2 CTAs -> leader
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(zhalf + 1);
  static_assert((2 * Cfg::WSLOTS + 12 + 2 * Cfg::ASLOTS) * 8 + 4 <= Cfg::BAR_BYTES, "barrier area");
  // Half-phase hand-overs (R = 128, where an epilogue warp owns two k-blocks of 64 channels): the MMA issuer starts the next
  // layer's centre taps on k-blocks 0 / 2 of y while the epilogue warps are still writing k-blocks 1 / 3, and GEMM2's k-block 2
  // while they are still gating k-block 3.  With 64-row tiles a warp owns ONE k-block, so nothing completes early.
  constexpr bool kHalf = (R == 128);
  // order of the centre-tap weight tiles of a layer (producers and issuer alike): (chunk, channel block)
  // (1,0) (1,2) (1,1) (1,3) (0,0) (0,1) (0,2) (0,3) -- for both tile heights (only the waits differ): the accumulation order
  // decides the rounding, and 64-row and 128-row tiles stay bit-identical
  auto ctr_h = [](int i) -> int { return i < 4 ? 1 : 0; };
  auto ctr_cb = [](int i) -> int { return i < 4 ? ((i & 1) * 2 + (i >> 1)) : (i & 3); };
  auto aslot = [&](int s) -> uint8_t* { return s < 4 ? zbuf + s * UNIT : yslots + (s - 4) * UNIT; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const uint32_t prank = crank & 1;
  const uint32_t lead = crank & ~1u;
  const uint16_t pair_mask = static_cast<uint16_t>(3u << lead);
  const int tile = p.tile0 + blockIdx.x;                     // R-frame tile
  const bool tile_valid = tile < p.tile_end;
  const int b = tile / p.tiles_per_utt, tr = tile % p.tiles_per_utt;
  const int bq = tile_valid ? b : p.B;            // b == B: every TMA row out of bounds (zeros)
  const int t0 = tile_valid ? tr * R : 0;
  // CP is laid out by 128-frame tiles: this CTA's rows start at cp_row0 of tile cp_tile (padding CTAs read tile 0)
  const int cp_tile = tile_valid ? (b * (p.Tp / 128) + t0 / 128) : 0;
  const int cp_row0 = t0 % 128;
  const bool nb_lo = tile_valid && tr > 0, nb_hi = tile_valid && tr + 1 < p.tiles_per_utt;
  const int zq = tile_valid ? b : p.L * p.B;      // Z coordinate base: (l * B + b); out of bounds for padding CTAs

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tm_w);
    tma_prefetch_desc(&p.tm_y0);
    tma_prefetch_desc(&p.tm_z);
    tma_prefetch_desc(&p.tm_s16[0]);
    tma_prefetch_desc(&p.tm_s16[1]);
    if (p.head_flags) {
      tma_prefetch_desc(&p.tm_wh);
      tma_prefetch_desc(&p.tm_xst);
      tma_prefetch_desc(&p.tm_y0st);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < WS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kEpiWarps * G);
    }
    mbar_init(y0full, 1);
    mbar_init(yhalo, kEpiWarps * G);
    mbar_init(zdone, kEpiWarps);
    mbar_init(zfree, 1);
    mbar_init(lfin, 1);
    mbar_init(sdone, kEpiWarps);
    mbar_init(yhalf, kEpiWarps * G);
    mbar_init(zhalf, kEpiWarps * G);
    for (int s = 0; s < AS; ++s) {
      mbar_init(&afull[s], 1);
      mbar_init(&aempty[s], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc<G>(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  cluster_arrive();
  cluster_wait();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  Watchdog wd{p.status, globaltimer_ns() + p.budget_ns};

  // weight tile row in tm_w: GEMM1 (chunk h, tap, channel block cb, plane) / GEMM2 (half q, k-block kb, plane)
  auto w1_row = [&](int l, int h, int tap, int cb, int plane) -> int {
    const int idx = p.w_sr ? (h * 12 + tap * 4 + cb) : ((plane * 2 + h) * 12 + tap * 4 + cb);
    return p.w_row0 + l * p.w_layer_rows + idx * 256 + static_cast<int>(prank) * 128;
  };
  auto w2_row = [&](int l, int q, int kb, int plane) -> int {
    const int idx = p.w_sr ? (24 + q * 4 + kb) : (48 + (plane * 2 + q) * 4 + kb);
    return p.w_row0 + l * p.w_layer_rows + idx * 256 + static_cast<int>(prank) * 128;
  };

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(Cfg::REGS_LOW));
    if (warp == 0 && lane == 0) {
      // ================================ activation producer ================================
      bool ok = true;
      const uint64_t z_policy = l2_policy_evict_last();   // z comes back for the skip GEMM: keep it in L2 ahead of the CP stream
      // ---- L2 prefetch (cp.async.bulk.prefetch.L2, 16 KB pieces) ----
      // CP of layer l + 1: 2 * NPF pieces per CTA (the two CTAs of a pair share a 128-frame tile when R = 64: half a chunk each),
      // PACED over layer l while this thread waits for z_l.  Issued in one burst at the layer boundary (rounds 1-2) the 128
      // CTAs' requests -- 33 MB -- queued at HBM in front of the next layer's first weight tiles: the centre-tap phase ran at
      // 170-250 cycles per MMA instead of the 134 of the halo phase (timeline, profiles/README.md).
      constexpr int NPF = (R == 128 ? 8 : 4);
      constexpr long long kCpLead = 8000, kCpStep = 16000 / (2 * NPF);   // cycles: first piece after the z store, piece spacing
      auto cp_piece = [&](int l, int i) {
        const char* src = reinterpret_cast<const char*>(p.CP + ((static_cast<size_t>(l) * p.cp_tiles + cp_tile) * 2 + i / NPF) * kCpChunk);
        prefetch_l2_bulk(src + (R == 64 && cp_row0 ? NPF * 16384 : 0) + (i % NPF) * 16384, 16384);
      };
      // weights of layer l: every CTA of the launch prefetches its share of the layer's tile block (all CTAs then load the
      // same tiles by TMA, in lockstep: without this the first requester of every tile pays the HBM latency and a ring of
      // WS tiles does not cover it)
      auto w_prefetch = [&](int l) {
        if (l >= p.nl || !p.wbase) return;
        const size_t bytes = static_cast<size_t>(p.w_layer_rows) * 128;
        size_t share = ((bytes + gridDim.x - 1) / gridDim.x + 15) & ~static_cast<size_t>(15);
        if (share > 8 * 16384) share = 8 * 16384;
        const size_t off = static_cast<size_t>(blockIdx.x) * share;
        if (off >= bytes) return;
        if (share > bytes - off) share = bytes - off;
        const char* src = reinterpret_cast<const char*>(p.wbase) + (static_cast<size_t>(p.w_row0) + static_cast<size_t>(l) * p.w_layer_rows) * 128 + off;
        while (share > 0) {
          const uint32_t n = share > 16384 ? 16384u : static_cast<uint32_t>(share);
          prefetch_l2_bulk(src, n);
          src += n;
          share -= n;
        }
      };
      // layer 0: the whole [8 | R | 8]-row slots come from Y buffer 0 (written by the input projection kernel)
      DSX_STRACE(0, 0);
      if (prank == 0) mbar_arrive_expect_tx(y0full, G * Cfg::Y_BYTES);
      for (int cb = 0; cb < 4; ++cb) tma_load_3d<G>(&p.tm_y0, y0full, yslots + cb * Cfg::YSLOT, cb * 64, t0 - 8, bq, lead);
      DSX_STRACE(0, 1);
      w_prefetch(0);
      w_prefetch(1);
      if (p.cp_prefetch)
        for (int i = 0; i < 2 * NPF; ++i) cp_piece(0, i);
      DSX_STRACE(0, 2);
      for (int l = 0; l < p.nl && ok; ++l) {
        // z_l (complete once this CTA's epilogue warps are through chunk 1) -> Z[l] in HBM for the deferred skip GEMM;
        // the z area may be overwritten (next layer's chunk 0) once the store has read it.  While waiting: CP of layer l + 1
        int pf_i = (p.cp_prefetch && l + 1 < p.nl) ? 0 : 2 * NPF;
        long long pf_next = clock64() + kCpLead;
        uint32_t spins = 0;
        while (!mbar_try_wait(zdone, l & 1)) {
          if (pf_i < 2 * NPF && clock64() >= pf_next) {
            cp_piece(l + 1, pf_i++);
            pf_next += kCpStep;
          }
          if (((++spins) & 0x3ff) == 0) {
            if (*(volatile int*)wd.status != 0) { ok = false; break; }
            if (globaltimer_ns() > wd.deadline_ns) {
              atomicCAS(wd.status, 0, 108);
              ok = false;
              break;
            }
          }
        }
        if (!ok) break;
        while (pf_i < 2 * NPF) cp_piece(l + 1, pf_i++);      // (a layer faster than the pacing: the rest at once)
        if (!Cfg::SKIP_IN_LAYER) {
          for (int kb = 0; kb < 4; ++kb) tma_store_3d_hint(&p.tm_z, zbuf + kb * UNIT, kb * 64, t0, l * p.B + zq, z_policy);
          bulk_commit_group();
          bulk_wait_group_read0();
          mbar_arrive(zfree);
        }                                                    // (SKIP_IN_LAYER: the issuer's commit after the skip MMAs frees z)
        DSX_STRACE(0, l * 4 + 3);
        w_prefetch(l + 2);
      }
      // ---- deferred skip GEMM: A tiles = z of every layer, back from L2 / HBM (this tile's own stores) ----
      if (ok && !Cfg::SKIP_IN_LAYER) {
        bulk_wait_group0();                               // the stores are complete (visible to the loads below)
        ok = mbar_wait(lfin, 0, wd, 109);                 // no MMA reads the y / z areas any more
        uint32_t ai = 0;
        for (int l = 0; l < p.nl && ok; ++l)                // (ascending: the summation order of the in-layer form)
          for (int kb = 0; kb < 4 && ok; ++kb, ++ai) {
            const uint32_t s = ai % AS;
            ok = mbar_wait(&aempty[s], ((ai / AS) & 1) ^ 1, wd, 110);
            if (!ok) break;
            if (prank == 0) mbar_arrive_expect_tx(&afull[s], G * UNIT);
            tma_load_3d<G>(&p.tm_z, &afull[s], aslot(s), kb * 64, t0, l * p.B + zq, lead);
          }
      }
    } else if ((warp == 2 || warp == 3) && lane == 0) {
      // ================================ weight producers ================================
      const uint32_t wid = warp - 2;
      uint32_t wi = 0;
      bool ok = true;
      auto load_w = [&](int row) {
        if ((wi & 1) == wid) {
          const uint32_t s = wi % WS;
          ok = mbar_wait(&empty[s], ((wi / WS) & 1) ^ 1, wd, 102);
          if (ok) {
            if (prank == 0) mbar_arrive_expect_tx(&full[s], G * kUnitBytes);
            tma_load_2d<G>(&p.tm_w, &full[s], wring + s * kUnitBytes, 0, row, lead);
          }
        }
        ++wi;
      };
      for (int l = 0; l < p.nl && ok; ++l) {
        for (int i = 0; i < 8 && ok; ++i)                           // centre taps of both chunks first: they need no halo rows
          for (int pl = 0; pl < WP && ok; ++pl) load_w(w1_row(l, ctr_h(i), 1, ctr_cb(i), pl));
        for (int h = 0; h < 2 && ok; ++h)
          for (int cb = 0; cb < 4 && ok; ++cb)
            for (int tap = 0; tap < 3 && ok; tap += 2)
              for (int pl = 0; pl < WP && ok; ++pl) load_w(w1_row(l, h, tap, cb, pl));
        for (int kb = 0; kb < 4 && ok; ++kb)
          for (int pl = 0; pl < WP && ok; ++pl) load_w(w2_row(l, 0, kb, pl));
        if (Cfg::SKIP_IN_LAYER)                                       // the skip half of this layer, right after its GEMM2
          for (int kb = 0; kb < 4 && ok; ++kb)
            for (int pl = 0; pl < WP && ok; ++pl) load_w(w2_row(l, 1, kb, pl));
      }
      if (!Cfg::SKIP_IN_LAYER)
        for (int l = 0; l < p.nl && ok; ++l)                          // deferred skip GEMM (same order as its A tiles)
          for (int kb = 0; kb < 4 && ok; ++kb)
            for (int pl = 0; pl < WP && ok; ++pl) load_w(w2_row(l, 1, kb, pl));
      if (p.head_flags) {
        // fused head: 128-row tiles of the whead pack (hi plane, lo plane per k-block).  The N = 256 operand of a pair is
        // [leader's tile | peer's tile]: the row halves of skip_projection / input_projection, twice the same tile for
        // output_projection (N = 80 padded to 128; the upper 128 columns of its accumulator are a copy)
        auto load_wh = [&](int tileidx) {
          if ((wi & 1) == wid) {
            const uint32_t s = wi % WS;
            ok = mbar_wait(&empty[s], ((wi / WS) & 1) ^ 1, wd, 111);
            if (ok) {
              if (prank == 0) mbar_arrive_expect_tx(&full[s], G * kUnitBytes);
              tma_load_2d<G>(&p.tm_wh, &full[s], wring + s * kUnitBytes, 0, tileidx * 128, lead);
            }
          }
          ++wi;
        };
        const int nh = static_cast<int>(prank);
        for (int kb = 0; kb < 4 && ok; ++kb)
          for (int pl = 0; pl < 2 && ok; ++pl) load_wh((pl * 2 + nh) * 4 + kb);
        for (int kb = 0; kb < 4 && ok; ++kb)
          for (int pl = 0; pl < 2 && ok; ++pl) load_wh(16 + pl * 4 + kb);
        if (p.head_flags & TC_INPROJ)
          for (int kb = 0; kb < 2 && ok; ++kb)
            for (int pl = 0; pl < 2 && ok; ++pl) load_wh(24 + (pl * 2 + nh) * 2 + kb);
      }
    } else if (warp == 1 && lane == 0 && prank == 0) {
      // ================================ MMA issuer (pair leader) ================================
      constexpr uint32_t idesc = umma_idesc_f16(R * G, 256);
      const uint32_t dF1 = tmem_base + Cfg::F1_COL;
      const uint32_t dSkip = tmem_base + Cfg::SKIP_COL;
      uint32_t wi = 0, accs = 0;
      bool ok = true;
      auto mma_tile = [&](uint32_t d, uint64_t a, uint32_t& acc, int code) {   // one weight tile of the global order
        const uint32_t s = wi % WS;
        ok = ok && mbar_wait(&full[s], (wi / WS) & 1, wd, code);
        if (!ok) return;
        tc_fence_after();
        const uint64_t w = umma_desc_sw128(smem_u32(wring + s * kUnitBytes));
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          umma_f16<G>(d, a + 2 * k4, w + 2 * k4, idesc, acc);
          acc = 1;
        }
        umma_commit<G>(&empty[s], pair_mask);
        ++wi;
      };
      // epilogue phases (drained accumulator, its z / y in shared memory).  tempty[0] completes twice per layer: chunk 0's
      // gate epilogue (parity 0), then the residual epilogue (parity 1); tempty[1] once per layer (parity l & 1)
      auto wait_epi = [&](uint64_t* bar, uint32_t parity, int code) {
        ok = ok && mbar_wait(bar, parity, wd, code);
        tc_fence_after();
      };
      for (int l = 0; l < p.nl && ok; ++l) {
        const int dil = 1 << (l % p.cycle);
        uint32_t acc0 = 0, acc1 = 0;
        if (l == 0) {                                   // layer 0: the whole slots (centre rows too) arrive by TMA
          ok = mbar_wait(y0full, 0, wd, 206);
          tc_fence_after();
        } else if (kHalf) {
          wait_epi(yhalf, (l - 1) & 1, 208);            // first half of epi2 of layer l-1: k-blocks 0, 2 of y_l written
        } else {
          wait_epi(&tempty[0], 1, 201);                 // epi2 of layer l-1: F0 drained, centre rows of y_l written
        }
        DSX_STRACE(1, l * 8);
        // centre taps.  F1 has been free since chunk 1's epilogue of layer l-1; with half-phase hand-over the first two tiles
        // (chunk 1, k-blocks 0 and 2) are issued under the second half of epi2, and F0 is touched only after all of it
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (kHalf && i == 2 && l > 0) wait_epi(&tempty[0], 1, 201);
          if (!ok) break;
          const int h = ctr_h(i), cb = ctr_cb(i);
          const uint64_t a = umma_desc_sw128(smem_u32(yslots + cb * Cfg::YSLOT)) + static_cast<uint64_t>((8 * 128) >> 4);
          for (int pl = 0; pl < WP && ok; ++pl) mma_tile(h == 0 ? tmem_base : dF1, a, h == 0 ? acc0 : acc1, 207);
        }
        DSX_STRACE(1, l * 8 + 1);
        if (l > 0 && ok) {                              // halo rows of this layer (from the neighbour tiles) are in the slots
          ok = mbar_wait(yhalo, (l - 1) & 1, wd, 206);
          tc_fence_after();
        }
        DSX_STRACE(1, l * 8 + 2);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          for (int cb = 0; cb < 4 && ok; ++cb) {
            const uint64_t y = umma_desc_sw128(smem_u32(yslots + cb * Cfg::YSLOT));
            for (int tap = 0; tap < 3 && ok; tap += 2) {
              const uint64_t a = y + static_cast<uint64_t>(((8 + (tap - 1) * dil) * 128) >> 4);   // row-shifted start
              for (int pl = 0; pl < WP && ok; ++pl) mma_tile(h == 0 ? tmem_base : dF1, a, h == 0 ? acc0 : acc1, 207);
            }
          }
          if (ok) umma_commit<G>(&tfull[h], pair_mask);
        }
        DSX_STRACE(1, l * 8 + 3);
        // GEMM2 (residual half) -> F0: k-blocks 0, 1 after chunk 0's epilogue (F0 drained, z k-blocks 0, 1 written),
        // k-blocks 2, 3 after chunk 1's
        uint32_t acc2 = 0;
        for (int kb = 0; kb < 4 && ok; ++kb) {
          if (kb == 0) wait_epi(&tempty[0], 0, 203);
          if (kb == 2) wait_epi(kHalf ? zhalf : &tempty[1], l & 1, 204);   // kHalf: z k-block 2 is complete half a phase early
          if (kb == 3 && kHalf) wait_epi(&tempty[1], l & 1, 204);
          if (!ok) break;
          if (kb == 0) DSX_STRACE(1, l * 8 + 4);
          if (kb == 2) DSX_STRACE(1, l * 8 + 5);
          const uint64_t z = umma_desc_sw128(smem_u32(zbuf + kb * UNIT));
          for (int pl = 0; pl < WP && ok; ++pl) mma_tile(tmem_base, z, acc2, 205);
        }
        if (ok) umma_commit<G>(&tfull[0], pair_mask);
        DSX_STRACE(1, l * 8 + 6);
        if (Cfg::SKIP_IN_LAYER) {
          // skip half of this layer -> its own accumulator, under the residual epilogue (z is complete: GEMM2's k-block 3 waited
          // for it); the z area is free for the next layer's gate epilogue once these MMAs have read it
          for (int kb = 0; kb < 4 && ok; ++kb) {
            const uint64_t z = umma_desc_sw128(smem_u32(zbuf + kb * UNIT));
            for (int pl = 0; pl < WP && ok; ++pl) mma_tile(dSkip, z, accs, 210);
          }
          if (ok) umma_commit<G>(zfree, pair_mask);
        }
      }
      if (!Cfg::SKIP_IN_LAYER) {
        // ---- deferred skip GEMM -> F1 (free since chunk 1's epilogue of the last layer), layers in ascending order: the
        //      same summation order as the in-layer form of the 64-row tiles ----
        if (ok) umma_commit<G>(lfin, pair_mask);
        uint32_t ai = 0;
        for (int l = 0; l < p.nl && ok; ++l)
          for (int kb = 0; kb < 4 && ok; ++kb, ++ai) {
            const uint32_t s = ai % AS;
            ok = mbar_wait(&afull[s], (ai / AS) & 1, wd, 209);
            if (!ok) break;
            tc_fence_after();
            const uint64_t a = umma_desc_sw128(smem_u32(aslot(s)));
            for (int pl = 0; pl < WP && ok; ++pl) mma_tile(dSkip, a, accs, 210);
            if (ok) umma_commit<G>(&aempty[s], pair_mask);
          }
      }
      if (ok) umma_commit<G>(&tfull[1], pair_mask);
      DSX_STRACE(1, 250);
      if (p.head_flags && ok) {
        // ---- fused head: three small GEMMs, hi/lo split of both operands (A_hi W_hi + A_lo W_hi + A_hi W_lo), each K block's A
        //      tiles (hi: A-ring units 0-3, lo: 4-7) written by the epilogue warps of both CTAs ----
        auto mma_pair = [&](uint32_t d, uint64_t a_hi, uint64_t a_lo, uint32_t& acc) {
          const uint32_t s = wi % WS;                                   // W_hi tile: with A_hi and A_lo
          ok = ok && mbar_wait(&full[s], (wi / WS) & 1, wd, 215);
          if (!ok) return;
          tc_fence_after();
          const uint64_t w = umma_desc_sw128(smem_u32(wring + s * kUnitBytes));
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) {
            umma_f16<G>(d, a_hi + 2 * k4, w + 2 * k4, idesc, acc);
            acc = 1;
          }
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) umma_f16<G>(d, a_lo + 2 * k4, w + 2 * k4, idesc, acc);
          umma_commit<G>(&empty[s], pair_mask);
          ++wi;
          mma_tile(d, a_hi, acc, 215);                                  // W_lo tile: with A_hi
        };
        wait_epi(&tempty[0], 1, 211);                                   // residual epilogue of the last layer: F0 drained
        wait_epi(&tempty[1], p.nl & 1, 212);                            // skip sum -> S16 tiles in shared memory, F1 drained
        uint32_t acch = 0;
        for (int kb = 0; kb < 4 && ok; ++kb)                            // H1 = S16 . W_skip^T -> F0
          mma_pair(tmem_base, umma_desc_sw128(smem_u32(aslot(kb))), umma_desc_sw128(smem_u32(aslot(4 + kb))), acch);
        if (ok) umma_commit<G>(&tfull[0], pair_mask);
        wait_epi(&tempty[0], 0, 213);                                   // h = relu(H1 + b) tiles written, F0 drained
        acch = 0;
        for (int kb = 0; kb < 4 && ok; ++kb)                            // H2 = h . W_out^T -> F1 (eps in columns [0, M))
          mma_pair(dF1, umma_desc_sw128(smem_u32(aslot(kb))), umma_desc_sw128(smem_u32(aslot(4 + kb))), acch);
        if (ok) umma_commit<G>(&tfull[1], pair_mask);
        if (p.head_flags & TC_INPROJ) {
          wait_epi(&tempty[1], (p.nl + 1) & 1, 214);                    // sampler update done: x_in tiles written, F1 drained
          acch = 0;
          for (int kb = 0; kb < 2 && ok; ++kb)                          // I = x_in . W_in^T -> F0
            mma_pair(tmem_base, umma_desc_sw128(smem_u32(aslot(kb))), umma_desc_sw128(smem_u32(aslot(4 + kb))), acch);
          if (ok) umma_commit<G>(&tfull[0], pair_mask);
        }
        DSX_STRACE(1, 251);
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(Cfg::REGS_HIGH));
    // ================================ epilogue (8 warps) ================================
    // thread <-> accumulator: TMEM lane quadrant `quad` (32 lanes) is fixed by the warp index; the two warps of a quadrant
    // (wh = 0, 1) split the columns.  R = 128: row = lane index, N indices [wh * 128, +128).  R = 64: rows (quad & 1) * 32 + lane,
    // N half quad >> 1, of which this warp has columns [wh * 64, +64).
    const int quad = warp & 3;
    const int wh = (warp - 4) >> 2;
    const int r = (R == 128 ? quad : (quad & 1)) * 32 + lane;             // frame row in the tile
    const int ng = (R == 128) ? wh : (quad >> 1);                          // 128-wide N group of this thread
    const uint32_t tlane = static_cast<uint32_t>(quad * 32) << 16;
    const int nbase = (R == 128) ? wh * 128 : (quad >> 1) * 128 + wh * 64;  // first N index (= channel in epi2 / exit)
    const int cbase = (R == 128) ? nbase : wh * 64;                        // its TMEM column
    constexpr int NCH = Cfg::NCH, NSP = Cfg::NSP, NQ = 2 * NSP;
    const bool tracer = (warp == 4 && lane == 0);
    const bool row_valid = tile_valid && (t0 + r < p.T);
    const bool edge = (r < 8 || r >= R - 8) && tile_valid;               // rows the neighbour tiles need as halo rows
    const int et = threadIdx.x - 128;               // 0..255: halo reception (side, row, 16-channel group)
    const size_t grow = (static_cast<size_t>(tile_valid ? b : 0) * p.Tp + t0 + r) * kC + nbase;   // this thread's row / channels
    bool ok = true;
    auto release = [&](uint64_t* bar) {             // this warp's part of the phase on F0 / F1 is done
      tc_fence_before();
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(bar, lead);
    };
    // tfull[0] completes twice per layer (GEMM1 chunk 0: parity 0, GEMM2: parity 1), tfull[1] once (parity l & 1; the skip GEMM
    // after the last layer: parity nl & 1).  One lane polls, the warp reconverges on the shuffle.
    auto wait_acc = [&](uint64_t* bar, uint32_t parity, int code) -> bool {
      int okv = 1;
      if (lane == 0) okv = mbar_wait(bar, parity, wd, code) ? 1 : 0;
      okv = __shfl_sync(0xffffffffu, okv, 0);
      tc_fence_after();
      return okv != 0;
    };
    const uint64_t cp_policy = l2_policy_evict_first();

    // residual stream of this thread's row: NCH channels, fp32, in registers for the whole stack.  First needed by epi2 of
    // layer 0, ~35 k cycles in.  Issued at the kernel's entry these loads (128 KB per CTA, 16 MB over the machine) queued in
    // front of the y0 and weight tiles the first MMAs wait for (entry -> first MMA 11-17 k cycles); issued after the first
    // accumulator they delayed the first gate epilogue instead.  So: a fixed head start for the TMA loads of the producers.
    float x[NCH];
    {
      const long long t_go = clock64() + 5000;
      while (clock64() < t_go) {}
    }
#pragma unroll
    for (int i = 0; i < NCH / 4; ++i) {
      const float4 v = *reinterpret_cast<const float4*>(p.X + grow + i * 4);
      x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
    }
    const float* dbase = p.dtab + static_cast<size_t>(tile_valid ? b : 0) * p.d_row_stride;
    float* const tb = tab + (warp - 4) * 256;       // this warp's table: [bias(NCH) | d_next(NCH)]

    for (int l = 0; l < p.nl && ok; ++l) {
      const bool has_next = (l + 1 < p.nl);
      // ---- per-layer vectors of this warp's channels -> its own shared-memory table (the polling loads of the halo
      //      exchange and the fences of the hand-over keep L1 cold, so reading them from global inside the epilogue would cost
      //      an L2 round trip each; one table per warp: no cross-warp barrier) ----
      __syncwarp();
      if (lane < NCH / 4) {
        // (the bias already scaled by 1 / sqrt 2: epi2 is x <- fma(x, c, fma(o, c, b c)), two packed FMAs per channel pair)
        float4 bl = __ldg(reinterpret_cast<const float4*>(p.b2 + static_cast<size_t>(l) * 512 + nbase) + lane);
        bl.x *= 0.70710678118654752440f; bl.y *= 0.70710678118654752440f; bl.z *= 0.70710678118654752440f; bl.w *= 0.70710678118654752440f;
        *reinterpret_cast<float4*>(tb + lane * 4) = bl;
        *reinterpret_cast<float4*>(tb + NCH + lane * 4) =
            has_next ? __ldg(reinterpret_cast<const float4*>(dbase + static_cast<size_t>(l + 1) * kC + nbase) + lane)
                     : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      __syncwarp();

      // ---- epi1: z = sigmoid(gate) * tanh(filter), gate / filter = accumulator + CP.  NQ sub-passes of 8 channels (NSP per
      //      chunk); the CP stream is the latency that matters (ncu: long-scoreboard stalls on the accumulator + CP adds), so its
      //      loads run TWO sub-passes ahead through three register buffers, across the chunk boundary too.
      //      Sub-pass sp of a chunk: chunk-channels c .. c + 8, gate in TMEM column tg, filter in tg + 64 (N order g * 128 + j) ----
      const float* cpl = p.CP + (static_cast<size_t>(l) * p.cp_tiles + cp_tile) * 2 * kCpChunk + (cp_row0 + r) * 4;
      constexpr int NB = 3;
      float4 cg[NB][2], cf[NB][2];
      // R = 128: a warp takes 32 channels of the chunk's first k-block (sub-passes 0-3), then 32 of its second (4-7), so the
      // first k-block of a chunk is complete -- over both warps of a quadrant -- half a phase early (zhalf)
      auto chan = [&](int sp) { return (R == 128) ? (sp >> 2) * 64 + wh * 32 + (sp & 3) * 8 : ng * 64 + wh * 32 + sp * 8; };      // chunk-channel
      auto tcol = [&](int sp) { return (R == 128) ? (sp >> 2) * 128 + wh * 32 + (sp & 3) * 8 : wh * 32 + sp * 8; };                // TMEM column of its gate
      auto cp_issue = [&](int q, float4* g4, float4* f4) {                               // q = chunk * NSP + sub-pass
        const float* cph = cpl + (q / NSP) * kCpChunk;
        const int c = chan(q % NSP);
#pragma unroll
        for (int v4 = 0; v4 < 2; ++v4) {
          g4[v4] = ld_stream_f4(cph + ((c >> 2) + v4) * (kTile * 4), cp_policy);
          f4[v4] = ld_stream_f4(cph + (((128 + c) >> 2) + v4) * (kTile * 4), cp_policy);
        }
      };
      cp_issue(0, cg[0], cf[0]);
      cp_issue(1, cg[1], cf[1]);
      if (l > 0) {                                  // the TMA store of z_{l-1} has finished reading the z area
        int okv = 1;
        if (lane == 0) okv = mbar_wait(zfree, (l - 1) & 1, wd, 305) ? 1 : 0;
        ok = __shfl_sync(0xffffffffu, okv, 0) != 0;
        if (!ok) break;
      }
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        const int h = q / NSP, sp = q % NSP;
        if (sp == 0) {
          if (tracer) DSX_STRACE(2, l * 12 + h * 3);
          ok = wait_acc(&tfull[h], h == 0 ? 0u : static_cast<uint32_t>(l & 1), 301 + h);
          if (!ok) break;
          if (tracer) DSX_STRACE(2, l * 12 + h * 3 + 1);
        }
        const uint32_t tF = tmem_base + tlane + h * Cfg::F1_COL + tcol(sp);
        uint32_t g[8], f[8];
        tmem_ld_32x8(tF, g);
        tmem_ld_32x8(tF + 64, f);
        if (q + 2 < NQ) cp_issue(q + 2, cg[(q + 2) % NB], cf[(q + 2) % NB]);
        tmem_ld_wait();
        uint32_t hz[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float4 bg = cg[q % NB][e >> 1], bf = cf[q % NB][e >> 1];
          const float2 gg = add2(make_float2(__uint_as_float(g[2 * e]), __uint_as_float(g[2 * e + 1])),
                                 (e & 1) ? make_float2(bg.z, bg.w) : make_float2(bg.x, bg.y));
          const float2 ff = add2(make_float2(__uint_as_float(f[2 * e]), __uint_as_float(f[2 * e + 1])),
                                 (e & 1) ? make_float2(bf.z, bf.w) : make_float2(bf.x, bf.y));
          float z0, z1;
          if (p.fast_act) {                         // sigmoid_fast(g) * tanh_approx(f), two channels per instruction
            const float2 hg = mul2(gg, make_float2(0.5f, 0.5f));
            const float2 sg = fma2(make_float2(0.5f, 0.5f), make_float2(tanh_approx(hg.x), tanh_approx(hg.y)), make_float2(0.5f, 0.5f));
            const float2 zz = mul2(sg, make_float2(tanh_approx(ff.x), tanh_approx(ff.y)));
            z0 = zz.x;
            z1 = zz.y;
          } else {
            z0 = gate_acc(gg.x, ff.x);
            z1 = gate_acc(gg.y, ff.y);
          }
          hz[e] = h2_bits(__floats2half2_rn(z0, z1));
        }
        // channel 128 h + c  ->  z k-block 2 h + (c >> 6), 16-byte chunk (c & 63) >> 3 of row r
        const int c = chan(sp);
        uint8_t* zrow = zbuf + (2 * h + (c >> 6)) * UNIT + r * 128;
        *reinterpret_cast<uint4*>(zrow + ((((c & 63) >> 3) ^ (r & 7)) << 4)) = make_uint4(hz[0], hz[1], hz[2], hz[3]);
        if (kHalf && h == 1 && sp == NSP / 2 - 1) {     // z k-block 2 complete: GEMM2 may consume it under sub-passes 4-7
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(zhalf, lead);
        }
        if (sp == NSP - 1) {
          release(&tempty[h]);
          if (h == 1 && lane == 0) mbar_arrive(zdone);    // (after the proxy fence + warp sync of release())
          if (tracer) DSX_STRACE(2, l * 12 + h * 3 + 2);
        }
      }
      if (!ok) break;

      // ---- epi2: x <- (x + D2res + b) / sqrt2 in registers (two packed FMAs per channel pair, the bias pre-scaled);
      //      y_{l+1} = fp16(x + d_{l+1}) -> next layer's A tiles ----
      if (tracer) DSX_STRACE(2, l * 12 + 6);
      ok = wait_acc(&tfull[0], 1, 303);
      if (!ok) break;
      if (tracer) DSX_STRACE(2, l * 12 + 7);
      {
        const float4* bt = reinterpret_cast<const float4*>(tb);
        const float4* dt = reinterpret_cast<const float4*>(tb + NCH);
        // halo packets of y_{l+1}: side 0 = this tile's first 8 rows, side 1 = its last 8 rows
        uint4* const ll_out = p.ll + ((static_cast<size_t>(tile_valid ? tile : 0) * 2 + ((l + 1) & 1)) * 2 + (r < 8 ? 0 : 1)) * 512 +
                              (r & 7) * 64 + nbase / 4;
        const unsigned int seq_next = p.seq_base + static_cast<unsigned int>(l + 1);
        uint32_t o[2][16];                          // accumulator pieces of 16 columns, the next one in flight
        tmem_ld_32x16(tmem_base + tlane + cbase, o[0]);
#pragma unroll
        for (int pc = 0; pc < NCH / 16; ++pc) {
          tmem_ld_wait();
          if (pc + 1 < NCH / 16) tmem_ld_32x16(tmem_base + tlane + cbase + (pc + 1) * 16, o[(pc + 1) & 1]);
#pragma unroll
          for (int c2 = 0; c2 < 2; ++c2) {
            uint32_t hy[4];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int i = c2 * 8 + e * 4, col = pc * 16 + i;
              const float4 bias = bt[col >> 2], dn = dt[col >> 2];
              const float2 c2v = make_float2(0.70710678118654752440f, 0.70710678118654752440f);
              const float2 xa = fma2(make_float2(x[col], x[col + 1]), c2v,
                                     fma2(make_float2(__uint_as_float(o[pc & 1][i]), __uint_as_float(o[pc & 1][i + 1])), c2v,
                                          make_float2(bias.x, bias.y)));
              const float2 xb = fma2(make_float2(x[col + 2], x[col + 3]), c2v,
                                     fma2(make_float2(__uint_as_float(o[pc & 1][i + 2]), __uint_as_float(o[pc & 1][i + 3])), c2v,
                                          make_float2(bias.z, bias.w)));
              x[col] = xa.x; x[col + 1] = xa.y; x[col + 2] = xb.x; x[col + 3] = xb.y;
              const float2 ya = add2(xa, make_float2(dn.x, dn.y)), yb = add2(xb, make_float2(dn.z, dn.w));
              hy[2 * e] = row_valid ? h2_bits(__floats2half2_rn(ya.x, ya.y)) : 0u;
              hy[2 * e + 1] = row_valid ? h2_bits(__floats2half2_rn(yb.x, yb.y)) : 0u;
            }
            if (has_next) {
              // channel ch .. ch + 8 of row r: y k-block ch >> 6, 16-byte chunk (ch & 63) >> 3 of slot row 8 + r
              const int ch = nbase + pc * 16 + c2 * 8;
              const uint4 v = make_uint4(hy[0], hy[1], hy[2], hy[3]);
              *reinterpret_cast<uint4*>(yslots + (ch >> 6) * Cfg::YSLOT + (8 + r) * 128 + ((((ch & 63) >> 3) ^ (r & 7)) << 4)) = v;
              if (edge) {                               // rows beyond T travel as zeros (the conv's zero padding)
                uint4* q = ll_out + pc * 4 + c2 * 2;
                asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(q), "r"(v.x), "r"(seq_next), "r"(v.y), "r"(seq_next) : "memory");
                asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(q + 1), "r"(v.z), "r"(seq_next), "r"(v.w), "r"(seq_next) : "memory");
              }
            }
          }
          if (kHalf && has_next && pc == NCH / 32 - 1) {   // this warp's first k-block of y_{l+1} (0 or 2) is written: the issuer
            fence_proxy_async_smem();                     // starts the next layer's centre taps on it (-> F1) under the second half
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(yhalf, lead);
          }
        }
      }
      release(&tempty[0]);
      if (tracer) DSX_STRACE(2, l * 12 + 8);
      if (has_next) {
        // ---- receive the halo rows of y_{l+1} from the neighbour tiles (GEMM2 of this layer has completed, so no MMA reads
        //      the slots): thread -> (side, row, 16 channels) = 4 packets; a packet is valid once both of its sequence words
        //      match.  Tiles at an utterance end (and padding CTAs) write zeros. ----
        const int side = et >> 7, row8 = (et >> 4) & 7, c16 = et & 15;
        const bool have = side == 0 ? nb_lo : nb_hi;
        uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0, q2 = q0, q3 = q0;
        if (have) {
          const unsigned int seq_next = p.seq_base + static_cast<unsigned int>(l + 1);
          const uint4* src = p.ll + ((static_cast<size_t>(side == 0 ? tile - 1 : tile + 1) * 2 + ((l + 1) & 1)) * 2 + (side == 0 ? 1 : 0)) * 512 +
                             row8 * 64 + c16 * 4;
          uint32_t spins = 0;
          while (true) {
            asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(q0.x), "=r"(q0.y), "=r"(q0.z), "=r"(q0.w) : "l"(src) : "memory");
            asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(q1.x), "=r"(q1.y), "=r"(q1.z), "=r"(q1.w) : "l"(src + 1) : "memory");
            asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(q2.x), "=r"(q2.y), "=r"(q2.z), "=r"(q2.w) : "l"(src + 2) : "memory");
            asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(q3.x), "=r"(q3.y), "=r"(q3.z), "=r"(q3.w) : "l"(src + 3) : "memory");
            if (q0.y == seq_next && q0.w == seq_next && q1.y == seq_next && q1.w == seq_next && q2.y == seq_next && q2.w == seq_next &&
                q3.y == seq_next && q3.w == seq_next)
              break;
            if (((++spins) & 0x3f) == 0) {
              if (*(volatile int*)wd.status != 0) { ok = false; break; }
              if (globaltimer_ns() > wd.deadline_ns) {
                atomicCAS(wd.status, 0, 307);
                ok = false;
                break;
              }
            }
          }
        }
        {
          const int hrow = (side == 0 ? 0 : R + 8) + row8;                 // row of the slot: [0, 8) left halo, [R + 8, R + 16) right halo
          uint8_t* dst = yslots + (c16 >> 2) * Cfg::YSLOT + hrow * 128;
          const int ch = (c16 & 3) * 2;                                    // first of the two 16-byte chunks
          *reinterpret_cast<uint4*>(dst + ((ch ^ row8) << 4)) = make_uint4(q0.x, q0.z, q1.x, q1.z);
          *reinterpret_cast<uint4*>(dst + (((ch + 1) ^ row8) << 4)) = make_uint4(q2.x, q2.z, q3.x, q3.z);
        }
        fence_proxy_async_smem();
        ok = __all_sync(0xffffffffu, ok);
        if (lane == 0) mbar_arrive_remote(yhalo, lead);
        if (tracer) DSX_STRACE(2, l * 12 + 9);
      }
    }

    // ---- exit: skip sum (deferred GEMM over all layers, in F1) -> fp16 hi / lo operand of the head GEMM, written as
    //      swizzled tiles into the (now idle) z / y areas and stored to S16 by TMA; debug taps (dsx_diffnet_forward only):
    //      fp32 skip sum -> SKIP, residual stream -> X ----
    if (tracer) DSX_STRACE(2, 248);
    if (ok) ok = wait_acc(&tfull[1], static_cast<uint32_t>(p.nl & 1), 304);
    if (tracer) DSX_STRACE(2, 249);
    if (ok) {
      // summed skip-half biases of this warp's channels -> its shared-memory table (as the per-layer vectors)
      __syncwarp();
      if (lane < NCH / 4)
        *reinterpret_cast<float4*>(tb + lane * 4) =
            __ldg(reinterpret_cast<const float4*>(p.bskip + static_cast<size_t>(p.nl - 1) * kC + nbase) + lane);
      __syncwarp();
      // (the exit / head epilogues run once per launch from a cold instruction cache -- ncu: no_instruction is their top
      //  stall, and fully unrolled they took 3 x as long as the same work inside the layer loop: rolled loops, compact bodies)
      const float4* bs4 = reinterpret_cast<const float4*>(tb);
#pragma unroll 1
      for (int pc = 0; pc < NCH / 16; ++pc) {
        uint32_t o[16];
        tmem_ld_32x16(tmem_base + tlane + Cfg::SKIP_COL + cbase + pc * 16, o);
        tmem_ld_wait();
#pragma unroll
        for (int c2 = 0; c2 < 2; ++c2) {
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int i = c2 * 8 + e * 4, col = pc * 16 + i;
            const float4 bb = bs4[col >> 2];
            float4 v;
            v.x = __uint_as_float(o[i]) + bb.x;
            v.y = __uint_as_float(o[i + 1]) + bb.y;
            v.z = __uint_as_float(o[i + 2]) + bb.z;
            v.w = __uint_as_float(o[i + 3]) + bb.w;
            if (p.taps && row_valid) *reinterpret_cast<float4*>(p.SKIP + grow + col) = v;
            const float sa = v.x * p.inv_sqrt_l, sb = v.y * p.inv_sqrt_l, sc = v.z * p.inv_sqrt_l, sd = v.w * p.inv_sqrt_l;
            const __half2 h0 = __floats2half2_rn(sa, sb), h1 = __floats2half2_rn(sc, sd);
            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
            hi[2 * e] = h2_bits(h0);
            hi[2 * e + 1] = h2_bits(h1);
            lo[2 * e] = h2_bits(__floats2half2_rn(sa - f0.x, sb - f0.y));
            lo[2 * e + 1] = h2_bits(__floats2half2_rn(sc - f1.x, sd - f1.y));
          }
          // channel ch .. ch + 8 of row r: k-block ch >> 6, 16-byte chunk (ch & 63) >> 3
          const int ch = nbase + pc * 16 + c2 * 8;
          const int off = r * 128 + ((((ch & 63) >> 3) ^ (r & 7)) << 4);
          *reinterpret_cast<uint4*>(aslot(ch >> 6) + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(aslot(4 + (ch >> 6)) + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      if (row_valid && p.taps) {
#pragma unroll
        for (int i = 0; i < NCH / 4; ++i)
          *reinterpret_cast<float4*>(p.X + grow + i * 4) = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
      }
      if (p.head_flags) {
        release(&tempty[1]);                          // S16 tiles -> the head GEMM of this launch
      } else {
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(sdone);
        if (p.nl == p.L && warp == 4 && lane == 0) {    // one thread stores the 2 x 4 tiles (rows beyond T are clipped)
          if (mbar_wait(sdone, 0, wd, 306)) {
            for (int pl = 0; pl < 2; ++pl)
              for (int kb = 0; kb < 4; ++kb) tma_store_3d(&p.tm_s16[pl], aslot(pl * 4 + kb), kb * 64, t0, bq);
            bulk_commit_group();
            bulk_wait_group0();
          }
        }
      }
    }
    if (tracer) DSX_STRACE(2, 250);

    if (p.head_flags && ok) {
      // ================================ fused head ================================
      // ---- epi-H: h = relu(H1 + b_skip_projection) -> fp16 hi / lo tiles (A operand of H2) ----
      __syncwarp();
      if (lane < NCH / 4) *reinterpret_cast<float4*>(tb + lane * 4) = __ldg(reinterpret_cast<const float4*>(p.bs + nbase) + lane);
      __syncwarp();
      ok = wait_acc(&tfull[0], 0, 311);
      if (ok) {
        const float4* b4 = reinterpret_cast<const float4*>(tb);
#pragma unroll 1
        for (int pc = 0; pc < NCH / 16; ++pc) {
          uint32_t o[16];
          tmem_ld_32x16(tmem_base + tlane + cbase + pc * 16, o);
          tmem_ld_wait();
#pragma unroll
          for (int c2 = 0; c2 < 2; ++c2) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int i = c2 * 8 + e * 4, col = pc * 16 + i;
              const float4 bb = b4[col >> 2];
              const float a0 = fmaxf(__uint_as_float(o[i]) + bb.x, 0.f), a1 = fmaxf(__uint_as_float(o[i + 1]) + bb.y, 0.f);
              const float a2 = fmaxf(__uint_as_float(o[i + 2]) + bb.z, 0.f), a3 = fmaxf(__uint_as_float(o[i + 3]) + bb.w, 0.f);
              const __half2 h0 = __floats2half2_rn(a0, a1), h1 = __floats2half2_rn(a2, a3);
              const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
              hi[2 * e] = h2_bits(h0);
              hi[2 * e + 1] = h2_bits(h1);
              lo[2 * e] = h2_bits(__floats2half2_rn(a0 - f0.x, a1 - f0.y));
              lo[2 * e + 1] = h2_bits(__floats2half2_rn(a2 - f1.x, a3 - f1.y));
            }
            const int ch = nbase + pc * 16 + c2 * 8;
            const int off = r * 128 + ((((ch & 63) >> 3) ^ (r & 7)) << 4);
            *reinterpret_cast<uint4*>(aslot(ch >> 6) + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(aslot(4 + (ch >> 6)) + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
        release(&tempty[0]);
      }
      if (tracer) DSX_STRACE(2, 251);

      // ---- mel phase: eps = H2 + b, sampler update of the mel state (thread = frame: coalesced in the reference's [B,1,M,T]
      //      layout), x_in operand of the input projection.  Bins are split over the warps that hold the row: R = 128: two
      //      (40 + 40); R = 64: four (the upper 128 accumulator columns are a copy): 24 + 16 + 24 + 16 ----
      if (ok) ok = wait_acc(&tfull[1], static_cast<uint32_t>((p.nl + 1) & 1), 312);
      if (ok) {
        const int part = (R == 128) ? wh : (quad >> 1) * 2 + wh;
        const int m_lo = (R == 128) ? part * 40 : (part >> 1) * 40 + (part & 1) * 24;
        const int m_hi = (R == 128) ? m_lo + 40 : m_lo + ((part & 1) ? 16 : 24);
        const int t = t0 + r;
        const bool do_in = (p.head_flags & TC_INPROJ) != 0;
        const bool need_z = (p.head_flags & TC_UPDATE) && p.c.sigma != 0.f;
        // Addressing by running pointers (ncu, round 2: 477 warp-instructions per 4 bins, a quarter of them 64-bit index
        // arithmetic of the strided accesses) and warp-uniform branches on the launch's flags only: rows beyond T compute on
        // zeros and are masked at the memory operations (predicated loads / stores instead of divergent blocks).
        const bool upd = (p.head_flags & TC_UPDATE) != 0, plms = (p.head_flags & TC_PLMS) != 0, weps = (p.head_flags & TC_WRITE_EPS) != 0;
        const size_t xc = static_cast<size_t>(p.xs.c), ec = static_cast<size_t>(p.T);       // bin strides: mel state, [B][M][T] arrays
        const size_t xrow = static_cast<size_t>(tile_valid ? b : 0) * p.xs.b + static_cast<size_t>(t) * p.xs.t;
        const size_t erow = static_cast<size_t>(tile_valid ? b : 0) * p.M * p.T + t;
        float* xp = p.xmel + xrow + static_cast<size_t>(m_lo) * xc;                         // bins m0 .. m0 + 3 of this row
        size_t eo = erow + static_cast<size_t>(m_lo) * ec;                                  // their index in the [B][M][T] arrays
        const float* bfp = p.bf + m_lo;
        size_t nblk = mel_noise_block(b + p.b_off, m_lo, t, p.M, p.T);                      // Philox block of the 4 bins (+T per step)
        float xn[4];                                          // the next iteration's mel state, loaded one iteration ahead
#pragma unroll
        for (int i = 0; i < 4; ++i) xn[i] = row_valid ? xp[i * xc] : 0.f;
        // PNDM: the eps history (up to three [B][M][T] arrays) likewise -- loaded inside the iteration, after the TMEM wait, the
        // three streams were a serial L2 / HBM round trip per 4 bins (ncu launch list: 447 us per PNDM launch against 375 us for
        // a DDPM one)
        const float* const hp[3] = {plms ? p.pl.h1 : nullptr, plms ? p.pl.h2 : nullptr, plms ? p.pl.h3 : nullptr};
        float hn[3][4];
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
          for (int i = 0; i < 4; ++i) hn[j][i] = (hp[j] && row_valid) ? hp[j][eo + i * ec] : 0.f;
#pragma unroll 1
        for (int m0 = m_lo; m0 < m_hi; m0 += 4, xp += 4 * xc, eo += 4 * ec, bfp += 4, nblk += ec) {
          uint32_t e4[4];
          tmem_ld_32x4(tmem_base + tlane + Cfg::F1_COL + m0, e4);
          float xv[4], zn[4], hv[3][4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            zn[i] = 0.f;
            xv[i] = xn[i];
#pragma unroll
            for (int j = 0; j < 3; ++j) hv[j][i] = hn[j][i];
          }
          if (m0 + 4 < m_hi) {
#pragma unroll
            for (int i = 0; i < 4; ++i) xn[i] = row_valid ? xp[(4 + i) * xc] : 0.f;
#pragma unroll
            for (int j = 0; j < 3; ++j)
#pragma unroll
              for (int i = 0; i < 4; ++i) hn[j][i] = (hp[j] && row_valid) ? hp[j][eo + (4 + i) * ec] : 0.f;
          }
          if (need_z) {
            if (p.noise) {
#pragma unroll
              for (int i = 0; i < 4; ++i) zn[i] = row_valid ? p.noise[eo + i * ec] : 0.f;
            } else {
              const float4 z4 = philox_normal4(p.seed, p.offset, nblk);
              zn[0] = z4.x; zn[1] = z4.y; zn[2] = z4.z; zn[3] = z4.w;
            }
          }
          const float4 bf4 = __ldg(reinterpret_cast<const float4*>(bfp));
          const float bfv[4] = {bf4.x, bf4.y, bf4.z, bf4.w};
          tmem_ld_wait();
          float ev[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) ev[i] = __uint_as_float(e4[i]) + bfv[i];
          if (weps) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (row_valid) p.eps_out[eo + i * ec] = ev[i];
          }
          if (upd) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              xv[i] = ddpm_step(p.c, xv[i], ev[i], zn[i]);
              if (row_valid) xp[i * xc] = xv[i];
            }
          }
          if (plms) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const size_t ei = eo + i * ec;
              xv[i] = plms_step(p.pl.c, xv[i], ev[i], hv[0][i], hv[1][i], hv[2][i], hp[0], hp[1], hp[2]);
              if (row_valid) {
                if (p.pl.eps_store) p.pl.eps_store[ei] = ev[i];
                if (p.pl.x_out) p.pl.x_out[ei] = xv[i];
                else xp[i * xc] = xv[i];
              }
            }
          }
          if (do_in) {                                        // 4 bins = half a 16-byte chunk of row r in k-block m0 >> 6
            uint32_t hi[2], lo[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const float a0 = row_valid ? xv[2 * e] : 0.f, a1 = row_valid ? xv[2 * e + 1] : 0.f;
              const __half2 hh = __floats2half2_rn(a0, a1);
              const float2 hf = __half22float2(hh);
              hi[e] = h2_bits(hh);
              lo[e] = h2_bits(__floats2half2_rn(a0 - hf.x, a1 - hf.y));
            }
            const int off = r * 128 + ((((m0 & 63) >> 3) ^ (r & 7)) << 4) + (m0 & 4) * 2;
            *reinterpret_cast<uint2*>(aslot(m0 >> 6) + off) = make_uint2(hi[0], hi[1]);
            *reinterpret_cast<uint2*>(aslot(4 + (m0 >> 6)) + off) = make_uint2(lo[0], lo[1]);
          }
        }
        if (do_in) {
          if (m_hi == p.M) {                                  // the K padding (bins M .. 127 = chunks 2 .. 7 of k-block 1)
#pragma unroll
            for (int c = 2; c < 8; ++c) {
              const int off = r * 128 + ((c ^ (r & 7)) << 4);
              *reinterpret_cast<uint4*>(aslot(1) + off) = make_uint4(0, 0, 0, 0);
              *reinterpret_cast<uint4*>(aslot(5) + off) = make_uint4(0, 0, 0, 0);
            }
          }
          release(&tempty[1]);
        }
      }
      if (tracer) DSX_STRACE(2, 252);

      // ---- epi-I: x0 = relu(I + b_in) (fp32) and y0 = fp16(x0 + d_0(next step)) as swizzled tiles over the idle W / y / z areas,
      //      stored by TMA to X and to Y buffer 0: the entry state of the next evaluation's launch ----
      if (ok && (p.head_flags & TC_INPROJ)) {
        __syncwarp();
        if (lane < NCH / 4) {
          *reinterpret_cast<float4*>(tb + lane * 4) = __ldg(reinterpret_cast<const float4*>(p.bin + nbase) + lane);
          *reinterpret_cast<float4*>(tb + NCH + lane * 4) =
              __ldg(reinterpret_cast<const float4*>(p.d0 + static_cast<size_t>(tile_valid ? b : 0) * p.d0_row_stride + nbase) + lane);
        }
        __syncwarp();
        ok = wait_acc(&tfull[0], 1, 313);
        if (ok) {
          const float4* b4 = reinterpret_cast<const float4*>(tb);
          const float4* d4 = reinterpret_cast<const float4*>(tb + NCH);
          uint8_t* const xt = wring;                          // 8 tiles of [R rows][32 fp32], then 4 tiles of [R rows][64 fp16]
          uint8_t* const yt = wring + 8 * UNIT;
#pragma unroll 1
          for (int pc = 0; pc < NCH / 16; ++pc) {
            uint32_t o[16];
            tmem_ld_32x16(tmem_base + tlane + cbase + pc * 16, o);
            tmem_ld_wait();
#pragma unroll
            for (int c2 = 0; c2 < 2; ++c2) {
              uint32_t hy[4];
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const int i = c2 * 8 + e * 4, col = pc * 16 + i;
                const float4 bb = b4[col >> 2], dn = d4[col >> 2];
                float4 v;
                v.x = fmaxf(__uint_as_float(o[i]) + bb.x, 0.f);
                v.y = fmaxf(__uint_as_float(o[i + 1]) + bb.y, 0.f);
                v.z = fmaxf(__uint_as_float(o[i + 2]) + bb.z, 0.f);
                v.w = fmaxf(__uint_as_float(o[i + 3]) + bb.w, 0.f);
                const int ch = nbase + col;                    // 4 channels = one 16-byte chunk of the fp32 tile ch >> 5
                *reinterpret_cast<float4*>(xt + (ch >> 5) * UNIT + r * 128 + ((((ch & 31) >> 2) ^ (r & 7)) << 4)) = v;
                hy[2 * e] = h2_bits(__floats2half2_rn(v.x + dn.x, v.y + dn.y));
                hy[2 * e + 1] = h2_bits(__floats2half2_rn(v.z + dn.z, v.w + dn.w));
              }
              const int ch = nbase + pc * 16 + c2 * 8;
              *reinterpret_cast<uint4*>(yt + (ch >> 6) * UNIT + r * 128 + ((((ch & 63) >> 3) ^ (r & 7)) << 4)) = make_uint4(hy[0], hy[1], hy[2], hy[3]);
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(sdone);
          if (warp == 4 && lane == 0) {
            if (mbar_wait(sdone, 0, wd, 314)) {
              for (int k = 0; k < 8; ++k) tma_store_3d(&p.tm_xst, xt + k * UNIT, k * 32, t0, bq);
              for (int k = 0; k < 4; ++k) tma_store_3d(&p.tm_y0st, yt + k * UNIT, k * 64, t0, bq);
              bulk_commit_group();
              bulk_wait_group_read0();          // the shared-memory source must outlive the copies; the writes complete with the grid
            }
          }
        }
      }
      if (tracer) DSX_STRACE(2, 253);
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  cluster_arrive();
  cluster_wait();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<G>(tmem_base, 512);
  }
  if (p.trace && threadIdx.x == 0 && blockIdx.x < 256) {
    p.trace[6 * 256 + blockIdx.x * 4 + 2] = static_cast<long long>(globaltimer_ns());
    p.trace[6 * 256 + blockIdx.x * 4 + 3] = clock64();
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// prefix sums over layers of the skip-half biases of output_projection: bskip[l][c] = sum_{j <= l} b2[j][256 + c]
__global__ void k_bskip_prefix(const float* __restrict__ b2, float* __restrict__ bskip, int L) {
  const int c = threadIdx.x;
  float acc = 0.f;
  for (int l = 0; l < L; ++l) {
    acc += b2[static_cast<size_t>(l) * 512 + 256 + c];
    bskip[static_cast<size_t>(l) * 256 + c] = acc;
  }
}

// Source row (in w1f / w2f, see dsx_simt.cu) of row n of a stack-kernel weight tile.  GEMM1 tile (chunk h): N index
// n = g * 128 + j; j < 64 -> gate of channel 128 h + 64 g + j (conv output row of that channel), j >= 64 -> its filter
// (row 256 + channel): a channel's gate and filter share a TMEM lane in both accumulator layouts (StackCfg).
__device__ __forceinline__ const float* stack_w_src(const float* w1f, const float* w2f, int l, bool is_w1, int hq, int kb, int n) {
  if (is_w1) {
    const int g = n >> 7, j = n & 127;
    const int ch = 128 * hq + 64 * g + (j & 63);
    const int row = (j < 64) ? ch : kC + ch;
    return w1f + (static_cast<size_t>(l) * 2 * kC + row) * (4 * kC) + kb * 64;
  }
  return w2f + (static_cast<size_t>(l) * 2 * kC + hq * 256 + n) * kC + kb * 64;
}

// hi / lo fp16 planes for the fp16x2 / fp16 modes: [L][64 tiles][256 rows][64]; W1 tile = (plane * 2 + h) * 12 + tap * 4 + cb
// (k-block kb = tap * 4 + cb of [tap0 | tap1 | tap2]), W2 tile = 48 + (plane * 2 + q) * 4 + kb
__global__ void k_pack_wstk(const float* __restrict__ w1f, const float* __restrict__ w2f, __half* __restrict__ wstk) {
  const int l = blockIdx.y, tileidx = blockIdx.x, n = threadIdx.x;
  const float* src;
  int plane;
  if (tileidx < 48) {
    plane = tileidx / 24;
    src = stack_w_src(w1f, w2f, l, true, (tileidx / 12) & 1, tileidx % 12, n);
  } else {
    const int u = tileidx - 48;
    plane = u / 8;
    src = stack_w_src(w1f, w2f, l, false, (u / 4) & 1, u & 3, n);
  }
  __half* dst = wstk + ((static_cast<size_t>(l) * 64 + tileidx) * 256 + n) * 64;
  for (int kk = 0; kk < 64; ++kk) {
    const float v = src[kk];
    const __half hi = __float2half_rn(v);
    dst[kk] = plane == 0 ? hi : __float2half_rn(v - __half2float(hi));
  }
}

// R stochastically rounded fp16 copies of the GEMM1 / GEMM2 weights (fp16s mode): element v lies between two fp16
// neighbours lo <= v <= hi and becomes hi with probability (v - lo) / (hi - lo), so E[w] = v; set r is used by diffusion
// step j with j % R == r.  Layout [R][L][32 tiles][256 rows][64]: W1 tile = h * 12 + tap * 4 + cb, W2 tile = 24 + q * 4 + kb.
// Philox4x32-10 keyed by (seed, set), counter = element index.
__global__ void k_pack_wsr(const float* __restrict__ w1f, const float* __restrict__ w2f, __half* __restrict__ wsr, int L,
                           unsigned long long seed) {
  const int l = blockIdx.y, tileidx = blockIdx.x, set = blockIdx.z, n = threadIdx.x;
  const float* src = (tileidx < 24) ? stack_w_src(w1f, w2f, l, true, tileidx / 12, tileidx % 12, n)
                                    : stack_w_src(w1f, w2f, l, false, (tileidx - 24) / 4, (tileidx - 24) & 3, n);
  const size_t row = ((static_cast<size_t>(set) * L + l) * 32 + tileidx) * 256 + n;
  __half* dst = wsr + row * 64;
  const uint2 key = make_uint2(static_cast<uint32_t>(seed) ^ (0x9E3779B9u * static_cast<uint32_t>(set + 1)),
                               static_cast<uint32_t>(seed >> 32) + static_cast<uint32_t>(set));
  for (int k4 = 0; k4 < 16; ++k4) {
    const size_t ctr = (static_cast<size_t>(l) * 32 + tileidx) * 256 * 16 + static_cast<size_t>(n) * 16 + k4;
    const uint4 rnd = philox4x32_10(make_uint4(static_cast<uint32_t>(ctr), static_cast<uint32_t>(ctr >> 32), 0x5352u, 0u), key);
    const uint32_t u4[4] = {rnd.x, rnd.y, rnd.z, rnd.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float v = src[k4 * 4 + e];
      const __half hn = __float2half_rn(v);
      const float fn = __half2float(hn);
      // the other neighbour: one fp16 ulp towards v
      __half ho = hn;
      if (fn != v) {
        unsigned short bits = __half_as_ushort(hn);
        const bool away = (fn < v) == (fn >= 0.f);     // move away from zero when v lies beyond |hn|
        if (fn == 0.f) bits = (v > 0.f) ? 0x0001 : 0x8001;
        else bits = static_cast<unsigned short>(away ? bits + 1 : bits - 1);
        ho = __ushort_as_half(bits);
      }
      const float fo = __half2float(ho);
      // P(take the other neighbour) = |v - fn| / |fo - fn|
      const float pr = (fo != fn) ? fabsf(v - fn) / fabsf(fo - fn) : 0.f;
      const float uu = static_cast<float>(u4[e] >> 8) * (1.0f / 16777216.0f);
      dst[k4 * 4 + e] = (uu < pr) ? ho : hn;
    }
  }
}

int tc_stack_pack(dsx_handle* h, cudaStream_t s) {
  float* bskip;
  DSX_TRY(dev_alloc(h, reinterpret_cast<void**>(&bskip), static_cast<size_t>(h->m.L) * 256 * sizeof(float), true));
  k_bskip_prefix<<<1, 256, 0, s>>>(h->m.b2f, bskip, h->m.L);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  h->m.bskip = bskip;
  h->m.wsr = nullptr;
  h->m.wsr_sets = 0;
  h->m.wstk = nullptr;
  if (h->precision == DSX_PREC_FP16S) {
    const int R = std::max(1, h->sr_sets);
    __half* wsr;
    const size_t rows = static_cast<size_t>(R) * h->m.L * kStackSetRowsPerLayer;
    DSX_TRY(dev_alloc(h, reinterpret_cast<void**>(&wsr), rows * 64 * sizeof(__half), true));
    dim3 grid(32, h->m.L, R);
    k_pack_wsr<<<grid, 256, 0, s>>>(h->m.w1f, h->m.w2f, wsr, h->m.L, h->sr_seed);
    h->launches++;
    DSX_CUDA(cudaGetLastError());
    h->m.wsr = wsr;
    h->m.wsr_sets = R;
    DSX_TRY(make_map_2d(&h->tm_wsr, wsr, rows, 128));
  } else if (h->precision == DSX_PREC_FP16 || h->precision == DSX_PREC_FP16X2) {
    __half* wstk;
    const size_t rows = static_cast<size_t>(h->m.L) * kStackRowsPerLayer;
    DSX_TRY(dev_alloc(h, reinterpret_cast<void**>(&wstk), rows * 64 * sizeof(__half), true));
    dim3 grid(64, h->m.L);
    k_pack_wstk<<<grid, 256, 0, s>>>(h->m.w1f, h->m.w2f, wstk);
    h->launches++;
    DSX_CUDA(cudaGetLastError());
    h->m.wstk = wstk;
    DSX_TRY(make_map_2d(&h->tm_wstk, wstk, rows, 128));
  }
  return DSX_OK;
}

template <int WP, int R>
static int stack_occupancy(dsx_handle* h) {
  int& cache = h->stack_occ[WP - 1][R == 128 ? 0 : 1];
  if (cache == 0) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(kG);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = StackCfg<R>::SMEM_BYTES;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    cudaFuncSetAttribute(k_tc_stack<WP, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, StackCfg<R>::SMEM_BYTES);
    cudaError_t e = cudaOccupancyMaxActiveClusters(&n, k_tc_stack<WP, R>, &cfg);
    if (e != cudaSuccess) cudaGetLastError();
    cache = (e == cudaSuccess && n >= 1) ? n : -1;
  }
  return cache;
}

static int stack_occ(dsx_handle* h, int rows) {
  const bool x2 = (h->precision == DSX_PREC_FP16X2);
  if (rows == 64) return x2 ? stack_occupancy<2, 64>(h) : stack_occupancy<1, 64>(h);
  return x2 ? stack_occupancy<2, 128>(h) : stack_occupancy<1, 128>(h);
}

// Rows per CTA for this call: 64-frame tiles (twice the CTAs, about half the time per layer) whenever the whole batch then
// still fits the machine at once, i.e. for small batches that would otherwise leave most SMs idle; 128-frame tiles otherwise.
static int stack_rows(dsx_handle* h, const Geom& g) {
  if (h->stack_rows == 64 || h->stack_rows == 128) return h->stack_rows;      // DSX_OPT_STACK_ROWS
  const int occ64 = stack_occ(h, 64);
  if (occ64 > 0 && g.B * (g.Tp / 64) <= occ64 * kG) return 64;
  return 128;
}

// Can the register-resident stack kernel take this call?  (every tile of an utterance must be co-resident)
bool tc_stack_usable(dsx_handle* h, const Geom& g) {
  if (h->stack_kernel == 0 || !h->stack_mode) return false;
  if (h->precision != DSX_PREC_FP16 && h->precision != DSX_PREC_FP16X2 && h->precision != DSX_PREC_FP16S) return false;
  const int rows = stack_rows(h, g);
  const int occ = stack_occ(h, rows);
  h->cluster_occ = occ;
  return occ > 0 && g.Tp / rows <= occ * kG;
}

template <int WP, int R>
static int launch_stack_t(dsx_handle* h, TcStackParams& prm, const Geom& g, cudaStream_t s) {
  const int occ = stack_occupancy<WP, R>(h);
  const int tiles_per_utt = g.Tp / R;
  const int utt_per_group = occ > 0 ? occ * kG / tiles_per_utt : 0;
  DSX_CHECK(utt_per_group >= 1, DSX_E_INVALID, "stack kernel: an utterance of %d tiles does not fit %d co-resident CTAs",
            tiles_per_utt, occ * kG);
  bool& attr_done = h->attr_stack[WP - 1][R == 128 ? 0 : 1];
  if (!attr_done) {
    DSX_CUDA(cudaFuncSetAttribute(k_tc_stack<WP, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, StackCfg<R>::SMEM_BYTES));
    attr_done = true;
  }
  prm.tiles_per_utt = tiles_per_utt;
  for (int b0 = 0; b0 < g.B; b0 += utt_per_group) {
    const int nb = std::min(utt_per_group, g.B - b0);
    prm.tile0 = b0 * tiles_per_utt;
    prm.tile_end = (b0 + nb) * tiles_per_utt;
    const int grid = (prm.tile_end - prm.tile0 + kG - 1) / kG * kG;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = StackCfg<R>::SMEM_BYTES;
    cfg.stream = s;
    // (Not a cooperative launch: Nsight Compute cannot replay a cooperative cluster launch -- `LaunchFailed` -- and a launch that
    //  cannot be profiled is worse than the documented requirement that the device is not shared while a step runs,
    //  INTEGRATION.md section 3; a lost peer ends in the in-kernel watchdog, and the handle stays usable.)
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    DSX_CUDA(cudaLaunchKernelEx(&cfg, k_tc_stack<WP, R>, prm));
    h->launches++;
    h->stack_launches++;
  }
  return DSX_OK;
}

// Layers [0, nl) of one evaluation (table row row0, weight set `wset`), one persistent launch per group of utterances.
int launch_tc_stack(dsx_handle* h, int nl, const Geom& g, int row0, int row_per_b, int wset, cudaStream_t s, const HeadArgs* head) {
  const ModelDev& m = h->m;
  const bool x2 = (h->precision == DSX_PREC_FP16X2);
  const bool sr = (h->precision == DSX_PREC_FP16S);
  if (nl <= 0) return DSX_OK;
  const int rows = stack_rows(h, g);
  const int ri = rows == 128 ? 0 : 1;
  h->stack_rows_used = rows;
  TcStackParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.tm_w = sr ? h->tm_wsr : h->tm_wstk;
  prm.wbase = sr ? static_cast<const void*>(m.wsr) : static_cast<const void*>(m.wstk);
  prm.tm_y0 = h->tm_y0s[ri];
  prm.tm_z = h->tm_zs[ri];
  prm.tm_s16[0] = h->tm_s16s[ri][0];
  prm.tm_s16[1] = h->tm_s16s[ri][1];
  prm.taps = h->want_taps;
  prm.X = h->ws.X;
  prm.SKIP = h->ws.SKIP;
  prm.CP = h->ws.CP;
  prm.cp_tiles = g.tiles;
  prm.cp_prefetch = h->cp_prefetch;
  prm.b2 = m.b2f;
  prm.bskip = m.bskip;
  prm.dtab = h->ws.DTAB + static_cast<size_t>(row0) * m.L * kC;
  prm.d_row_stride = row_per_b * m.L * kC;
  prm.T = g.T; prm.Tp = g.Tp; prm.B = g.B;
  prm.nl = nl; prm.L = m.L; prm.cycle = m.cycle;
  prm.w_sr = sr ? 1 : 0;
  prm.w_layer_rows = sr ? kStackSetRowsPerLayer : kStackRowsPerLayer;
  prm.w_row0 = sr ? (wset % std::max(1, m.wsr_sets)) * m.L * kStackSetRowsPerLayer : 0;
  prm.inv_sqrt_l = 1.0f / sqrtf(static_cast<float>(m.L));
  prm.fast_act = h->gate_approx >= 0 ? h->gate_approx : 1;
  prm.status = h->status_dev;
  prm.budget_ns = 4000000000ull;
  prm.trace = h->trace_dev;
  if (head && head->flags) {
    DSX_CHECK(nl == m.L, DSX_E_INVALID, "the fused head needs the whole stack");
    prm.head_flags = head->flags | TC_HEAD;
    prm.tm_wh = h->tm_whead;
    prm.tm_xst = h->tm_xst[ri];
    prm.tm_y0st = h->tm_y0st[ri];
    prm.xmel = head->x;
    prm.xs = head->xs;
    prm.eps_out = head->eps;
    prm.noise = head->noise;
    prm.seed = head->seed;
    prm.offset = head->offset;
    prm.b_off = h->batch_offset;
    prm.c = head->c;
    if (head->plms) prm.pl = *head->plms;
    prm.bs = m.skip_b;
    prm.bf = m.fin_b;
    prm.bin = m.in_b;
    prm.d0 = h->ws.DTAB + static_cast<size_t>(head->next_row0) * m.L * kC;
    prm.d0_row_stride = head->row_per_b * m.L * kC;
    prm.M = m.M;
  }
  // halo packets: 32 KB per tile, zeroed once (sequence numbers start at 1 and only grow, so packets left behind by earlier
  // evaluations, other geometries or an aborted launch can never be mistaken for the current layer's)
  const size_t ll_bytes = static_cast<size_t>(g.B * (g.Tp / 64) + 2) * 4 * 512 * sizeof(uint4);
  if (h->ll_cap < ll_bytes) {
    if (h->ll_dev) cudaFree(h->ll_dev);
    h->ll_dev = nullptr;
    h->ll_cap = 0;
    DSX_CUDA(cudaMalloc(&h->ll_dev, ll_bytes));
    DSX_CUDA(cudaMemsetAsync(h->ll_dev, 0, ll_bytes, s));
    h->ll_cap = ll_bytes;
  }
  if (h->ll_seq > 0xFFFF0000u) {                      // (practically unreachable) wrap: start over on a clean buffer
    DSX_CUDA(cudaMemsetAsync(h->ll_dev, 0, h->ll_cap, s));
    h->ll_seq = 1;
  }
  prm.ll = static_cast<uint4*>(h->ll_dev);
  prm.seq_base = h->ll_seq;
  int rc;
  if (rows == 128) rc = x2 ? launch_stack_t<2, 128>(h, prm, g, s) : launch_stack_t<1, 128>(h, prm, g, s);
  else rc = x2 ? launch_stack_t<2, 64>(h, prm, g, s) : launch_stack_t<1, 64>(h, prm, g, s);
  DSX_TRY(rc);
  h->ll_seq += static_cast<unsigned int>(nl);
  return DSX_OK;
}

}  // namespace dsx
