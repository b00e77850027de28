// tcgen05 / TMEM / TMA path of the dsx sampler (sm_100a).  Three kernels:
//   k_tc_layer<P>   all residual layers of one DiffNet evaluation (usr/diff/net.py:58-78), persistent, one launch
//   k_tc_head<P>    skip / output projections, the DDPM update and the next step's input projection (net.py:115-130,
//                   shallow_diffusion_tts.py:134-166)
//   k_tc_condproj   conditioner projection of every layer, once per call (it does not depend on the diffusion step)
//
// Per residual layer and 128-frame tile:
//   GEMM1  D1[128 frames x 512] = [y(t-d) | y(t) | y(t+d)] (K = 768) . W1^T                  y = x + d_l
//   epi1   z = sigmoid(D1[:, gate] + CP) * tanh(D1[:, filter] + CP)  -> fp16 (hi [, lo]) in shared memory
//   GEMM2  D2[128 x 512] = z (K = 256) . W2^T
//   epi2   x <- (x + D2[:, :256] + b) / sqrt2 ;  y_next = fp16 (split) of (x + d_{l+1}) ;  skip += D2[:, 256:] + b
// where CP = conditioner_projection_l(cond) + biases comes from HBM (fp32, accumulator layout, written by k_tc_condproj).
//
// Layout: activations are frames-major ([B][Tp][256], Tp = T rounded up to 128) so a 128-frame tile
// of 64 channels is one TMA box that lands in shared memory as the canonical K-major SWIZZLE_128B
// UMMA operand (rows of 128 B, 8-row atoms 1024 B apart).  The dilated taps read the same tensor at
// frame offsets -d, 0, +d; TMA zero-fills rows outside [0, T), which is exactly the conv's zero
// padding applied after the FiLM add.  Weights are pre-packed into 256x64 fp16 tiles (32 KB) in the
// order the K loop consumes them; the gate/filter rows of a 256-wide N chunk are interleaved as
// [128 gate | 128 filter] so TMEM columns j and j+128 belong to the same channel.
//
// Precision: P = 1 fp16 operands (fp32 accumulate); P = 2 adds a W_lo pass (weights as hi+lo fp16 pairs);
// P = 3 accumulates A_hi*W_hi + A_hi*W_lo + A_lo*W_hi into the same TMEM tile (~2^-22 relative).
//
// Roles (384 threads): lane 0 of warps 0, 2, 3 = TMA producers (a thread gets one load accepted per ~430 cycles),
// warp 1 = MMA issuer (one thread of the pair's leader CTA), warp 2 also allocates TMEM, warps 4-11 = epilogue
// (thread = frame row = TMEM lane; two warps per lane quadrant split the columns).
// cta_group::2: a cluster of two CTAs, each with its own 128 frames (UMMA M = 256); every CTA loads half of each
// weight tile, halving weight traffic from L2 and shared-memory operand reads.
#include <cuda.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <type_traits>
#include <vector>

#include "dsx_internal.h"
#include "dsx_ptx.cuh"
#include "dsx_rng.cuh"
#include "dsx_tc_common.cuh"
#include "dsx_update.cuh"

namespace dsx {

template <int P>
struct TcCfg {
  // P = number of MMA passes of the parity scheme: 1 = fp16 operands; 2 = weights hi+lo, running activations fp16;
  // 3 = hi+lo on both operands.  (The conditioner projection is hoisted out of the loop and always exact.)
  static constexpr bool WLO = (P >= 2);     // W_lo pass
  static constexpr bool ALO_T = (P == 3);   // A_lo pass on the conv taps (y) and on z
  static constexpr int Z_PLANES = ALO_T ? 2 : 1;
  // z (the A operand of GEMM2) is [planes][4 k-blocks] of 16 KB: k-blocks 0,1 (written while GEMM1 still runs) have
  // their own buffer z01; k-blocks 2,3 are written after GEMM1 has finished and alias operand buffers of GEMM1.
  // Epilogue 2 transposes the accumulator through a 32 KB staging area (8 warps x 32 rows x 128 B).
  //
  // SHIFT (P <= 2): the three dilated taps of a 64-channel block share ONE shared-memory copy of the activations: a y
  // slot holds [8 halo rows | 128 centre rows | 8 halo rows] (18 KB, one TMA box) and tap j's UMMA descriptor simply
  // starts (8 + (j-1)*d) rows in (SWIZZLE_128B is a function of the absolute address; verified by dsx_selftest(2)).
  // Shared memory: [W ring: WSLOTS x 16 KB | 2 y slots x 18 KB (z k-blocks 2,3 alias them) | staging 32 KB | z01].
  // All weight tiles of GEMM1 and GEMM2, layer after layer, flow through the ONE W ring in a fixed global order, so
  // the weight producers run ahead of every dependency (flags, epilogues, layer boundaries); the y slots double-buffer
  // the activation blocks.
  // (Splitting chunk 1 into two N = 128 sub-chunks to hide half of its gate epilogue was tried: a cta_group::2 MMA with
  // N = 128 takes as long as one with N = 256 here, so it lost.)
  // P == 3 has no shared memory for that and keeps one 16 KB tile per tap in a ring of UNITS units:
  // [ring2 (GEMM2 weights) | z23 | staging] alias the ring once GEMM1 is done.
  static constexpr bool SHIFT = (P <= 2);
  static constexpr int SLOT = SHIFT ? (kTile + 16) * 128 : kUnitBytes;   // y slot (SHIFT) / ring unit
  static constexpr int WSLOTS = 7;
  static constexpr int UNITS = 10;
  static constexpr int Z23_UNITS = 2 * Z_PLANES;
  static constexpr int STG_UNITS = 2;
  static constexpr int UNITS2 = UNITS - Z23_UNITS - STG_UNITS;
  static constexpr int Z01_BYTES = Z_PLANES * 2 * kUnitBytes;
  static constexpr int BAR_BYTES = 512;
  static constexpr int OPER_BYTES = SHIFT ? WSLOTS * kUnitBytes + 2 * SLOT + STG_UNITS * kUnitBytes : UNITS * kUnitBytes;
  static constexpr int SMEM_BYTES = 1024 + OPER_BYTES + Z01_BYTES + BAR_BYTES;
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
  // P == 3 ring units consumed per k-block: GEMM1 {A_hi, W_hi, W_lo, A_lo}, GEMM2 {W_hi, W_lo}
  static constexpr int UT = 2 + (WLO ? 1 : 0) + (ALO_T ? 1 : 0);
  static constexpr int U2 = 1 + (WLO ? 1 : 0);
  // P == 3 ring slot of unit `ul` of a layer: the first S0 units cycle through the non-staging slots only, so they can
  // be loaded and multiplied while the previous layer's skip epilogue still owns the staging slots.
  static constexpr int S0 = 4 * UT;
  __host__ __device__ static constexpr int slot(int ul) { return ul < S0 ? ul % (UNITS - STG_UNITS) : (ul - S0) % UNITS; }
};

struct TcLayerParams {
  CUtensorMap tm_w;          // packed weights, 2D [rows][64], box 64 x 128 rows
  CUtensorMap tm_y[2][2];    // conv input, [buffer = layer parity][plane hi/lo], 3D [B][T][256]
  CUtensorMap tm_yh[2];      // conv input hi plane of buffer 0 / 1 with a box of 8 + 128 + 8 frames (SHIFT layout)
  float* X;                  // [B][Tp][256] residual stream (in/out)
  float* SKIP;               // [B][Tp][256]
  __half* Y;                 // [2 buffers][2 planes][plane_elems]: layer l reads buffer l&1, writes buffer (l+1)&1
  size_t plane_elems;
  int cp_prefetch;           // SHIFT: the activation producer streams CP into L2 half a layer ahead (tuning knob)
  const float* CP;           // [L][tiles][2 chunks][64 column groups][128 rows][4]: cond projection + bias (fp32)
  const float* b2;           // [L][512]
  const float* dtab;         // FiLM table row of this evaluation: [L][256], utterance b at + b * d_row_stride
  int d_row_stride;
  int T, Tp, tiles_per_utt, tiles, B;
  int tile0, tile_end;       // this launch covers tiles [tile0, tile_end) (whole utterances); CTA i -> tile tile0 + i
  int l0, l1, L, cycle;      // layers [l0, l1); dilation of layer l = 1 << (l % cycle)
  unsigned int* flags;       // [tiles] monotonic publish counters (multi-layer launches), else nullptr
  unsigned int flag_base;    // counter value every valid tile had when this launch started
  __half* s16;               // fp16 split of skip_total * inv_sqrt_l (written by layer L-1), plane 1 at + plane_elems
  float inv_sqrt_l;
  int* status;
  unsigned long long budget_ns;
  long long* trace;          // debug: [2 CTAs][3 roles][256] clock64 stamps, or nullptr
  int seq;                   // debug: launch sequence number (slot of the entry / exit wall-clock stamps)
};

#define DSX_TRACE(role, slot)                                                              \
  do {                                                                                     \
    if (p.trace && blockIdx.x < 2 && (slot) < 256)                                          \
      p.trace[(blockIdx.x * 3 + (role)) * 256 + (slot)] = clock64();                       \
  } while (0)

// Residual layers [l0, l1) of one DiffNet evaluation.
//
// Multi-layer launches (l1 - l0 > 1, every CTA co-resident): the only cross-CTA dependency of the stack is that
// layer l+1 of tile i reads the conv input y_{l+1} of tiles i-1, i, i+1 of the same utterance.  After its residual
// epilogue every epilogue warp of a tile does a release-increment of that tile's publish counter in global memory;
// the TMA producer of a tile acquire-polls the counters of its (up to) three source tiles before the first
// activation load of the next layer.  No grid-wide barrier exists; weight loads run ahead of the dependency.
template <int P>
__global__ void __launch_bounds__(kThreads, 1) k_tc_layer(const __grid_constant__ TcLayerParams p) {
  using Cfg = TcCfg<P>;
  constexpr int G = kG;
  constexpr int NU = Cfg::UNITS;
  constexpr int NU2 = Cfg::UNITS2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // SHIFT: ring = W ring (WSLOTS x 16 KB), then the two y slots, then staging; otherwise the 10-unit ring whose last
  // units double as z23 / staging
  uint8_t* yslots = ring + Cfg::WSLOTS * kUnitBytes;                                     // SHIFT only
  uint8_t* staging = Cfg::SHIFT ? yslots + 2 * Cfg::SLOT : ring + (NU - Cfg::STG_UNITS) * kUnitBytes;
  uint8_t* z01 = ring + Cfg::OPER_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(z01 + Cfg::Z01_BYTES);
  uint64_t* full = bars;             // [NU]   P == 3: GEMM1 ring; SHIFT: W ring (first WSLOTS)
  uint64_t* empty = full + NU;       // [NU]
  uint64_t* full2 = empty + NU;      // [NU2]  P == 3: GEMM2 weight ring (aliases ring units 0..NU2-1)
  uint64_t* empty2 = full2 + NU2;    // [NU2]
  uint64_t* tfull = empty2 + NU2;    // [2]
  uint64_t* tempty = tfull + 2;      // [2]
  uint64_t* zf = tempty + 2;         // [2] z k-block 2 / 3 written (both CTAs of the pair); k-blocks 0,1 ride on tempty[0]
  uint64_t* g1done = zf + 2;         // P == 3: all GEMM1 MMAs of the layer complete
  uint64_t* g2done = g1done + 1;     // all GEMM2 MMAs of the layer complete (z units reusable)
  uint64_t* edone = g2done + 1;      // P == 3: this CTA's epilogue has left the staging units
  uint64_t* yfull = edone + 1;       // [2] SHIFT: y slots
  uint64_t* yempty = yfull + 2;      // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(yempty + 2);
  static_assert((2 * Cfg::UNITS + 2 * Cfg::UNITS2 + 13) * 8 + 4 <= Cfg::BAR_BYTES, "barrier area");
  // z k-block address: plane 0 = hi, 1 = lo.  k-blocks 2,3 alias the y slots (SHIFT) / ring units [NU2, NU2 + Z23_UNITS)
  auto zaddr = [&](int plane, int kb) -> uint8_t* {
    if (kb < 2) return z01 + (plane * 2 + kb) * kUnitBytes;
    return Cfg::SHIFT ? yslots + (kb - 2) * Cfg::SLOT : ring + (NU2 + plane * 2 + (kb - 2)) * kUnitBytes;
  };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const uint32_t prank = crank & 1;               // rank inside the cta_group::2 pair
  const uint32_t lead = crank & ~1u;              // cluster rank of the pair's leader
  const uint16_t pair_mask = static_cast<uint16_t>(3u << lead);
  if (threadIdx.x == 0) {
    DSX_TRACE(0, 250);                                           // kernel entry (clock64)
    if (p.trace && blockIdx.x < 2) p.trace[(blockIdx.x * 3 + 1) * 256 + 250] = static_cast<long long>(globaltimer_ns());
    if (p.trace && blockIdx.x == 0) p.trace[220 + (p.seq % 8) * 2] = static_cast<long long>(globaltimer_ns());
  }
  // tile -> (utterance, 128-frame tile in the utterance); the grid is padded to an even number of CTAs
  const int tile = p.tile0 + blockIdx.x;
  const bool tile_valid = tile < p.tile_end;
  const int b = tile / p.tiles_per_utt, tr = tile % p.tiles_per_utt;
  const int bq = tile_valid ? b : p.B;            // b == B -> every TMA row is out of bounds (zeros)
  const int cp_tile = tile_valid ? tile : 0;      // padding CTAs read (and discard) tile 0's slice of CP
  const int t0 = tile_valid ? tr * kTile : 0;
  const bool multi = (p.l1 - p.l0 > 1);
  const bool nb_lo = multi && tile_valid && tr > 0, nb_hi = multi && tile_valid && tr + 1 < p.tiles_per_utt;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tm_w);
    tma_prefetch_desc(&p.tm_y[0][0]);
    tma_prefetch_desc(&p.tm_y[1][0]);
    tma_prefetch_desc(&p.tm_yh[0]);
    tma_prefetch_desc(&p.tm_yh[1]);
    if (Cfg::ALO_T) {
      tma_prefetch_desc(&p.tm_y[0][1]);
      tma_prefetch_desc(&p.tm_y[1][1]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NU; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < NU2; ++s) {
      mbar_init(&full2[s], 1);
      mbar_init(&empty2[s], 1);
    }
    mbar_init(g1done, 1);
    mbar_init(g2done, 1);
    mbar_init(edone, kEpiWarps);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kEpiWarps * G);
    }
    mbar_init(&zf[0], kEpiWarps * G);
    mbar_init(&zf[1], kEpiWarps * G);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&yfull[i], 1);
      mbar_init(&yempty[i], 1);
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
  if (threadIdx.x == 0) DSX_TRACE(0, 254);

  // A thread gets one TMA load accepted per ~430 cycles whatever its size (dsx_selftest(3)), so three threads (lane 0
  // of warps 0, 2, 3) produce.  SHIFT: producer 0 owns the activation blocks (and their dependencies), producers 1, 2
  // alternate over the weight tiles.  P == 3: the three take the ring units round-robin.
  const int prod_id = (warp == 0) ? 0 : (warp == 2 ? 1 : (warp == 3 ? 2 : -1));
  if (prod_id >= 0 && lane == 0) {
    bool ok = true;
    if constexpr (Cfg::SHIFT) {
      if (prod_id == 0) {
        // ================================ activation producer ================================
        uint32_t yi = 0;                                            // running block index: slot yi & 1
        for (int l = p.l0; l < p.l1 && ok; ++l) {
          const int li = l - p.l0;
          if (li > 0) {
            ok = mbar_wait(g2done, (li - 1) & 1, wd, 105);          // z k-blocks 2,3 (in the y slots) consumed
            if (li < 10) DSX_TRACE(0, 200 + li);
            if (ok && multi && tile_valid) {                        // y_l of this tile and its neighbours published
              const unsigned int target = p.flag_base + static_cast<unsigned int>(kEpiWarps * li);
              ok = flag_wait3(p.flags + tile, nb_lo ? p.flags + tile - 1 : nullptr, nb_hi ? p.flags + tile + 1 : nullptr,
                              target, wd, 107);
              fence_proxy_async_all();
            }
            if (li < 10) DSX_TRACE(0, 210 + li);
          }
          for (int hc = 0; hc < 8 && ok; ++hc, ++yi) {              // (chunk h, channel block cb) = (hc >> 2, hc & 3)
            const int s = yi & 1;
            ok = mbar_wait(&yempty[s], ((yi >> 1) & 1) ^ 1, wd, 110);
            if (!ok) break;
            DSX_TRACE(0, hc);
            if (prank == 0) mbar_arrive_expect_tx(&yfull[s], G * Cfg::SLOT);
            tma_load_3d<G>(&p.tm_yh[l & 1], &yfull[s], yslots + s * Cfg::SLOT, (hc & 3) * 64, t0 - 8, bq, lead);
            if (p.cp_prefetch) {
              // stream the conditioner projection HBM -> L2 half a layer ahead of the gate epilogue that reads it:
              // during chunk 0's blocks chunk 1 of this layer, during chunk 1's blocks chunk 0 of the next layer
              const int pl = (hc < 4) ? l : l + 1, ph = (hc < 4) ? 1 : 0;
              if (pl < p.l1) {
                const char* src = reinterpret_cast<const char*>(p.CP + ((static_cast<size_t>(pl) * p.tiles + cp_tile) * 2 + ph) * kCpChunk);
                prefetch_l2_bulk(src + (hc & 3) * 32768, 16384);
                prefetch_l2_bulk(src + (hc & 3) * 32768 + 16384, 16384);
              }
            }
          }
        }
      } else {
        // ================================ weight producers ================================
        const uint32_t wid = prod_id - 1;
        uint32_t wi = 0;                                            // running W tile index: slot wi % WSLOTS
        for (int l = p.l0; l < p.l1 && ok; ++l) {
          const int w_row0 = l * kRowsPerLayer;
          auto load_w = [&](int tileidx) {
            if ((wi & 1) == wid) {
              const uint32_t s = wi % Cfg::WSLOTS;
              ok = mbar_wait(&empty[s], ((wi / Cfg::WSLOTS) & 1) ^ 1, wd, 102);
              if (ok) {
                if (prank == 0) mbar_arrive_expect_tx(&full[s], G * kUnitBytes);
                tma_load_2d<G>(&p.tm_w, &full[s], ring + s * kUnitBytes, 0,
                               w_row0 + tileidx * 256 + static_cast<int>(prank) * 128, lead);
              }
            }
            ++wi;
          };
          for (int h = 0; h < 2 && ok; ++h)
            for (int cb = 0; cb < 4 && ok; ++cb)
              for (int tj = 0; tj < 3 && ok; ++tj) {                // tap order: centre, left, right
                const int tap = tj == 0 ? 1 : (tj == 1 ? 0 : 2);
                load_w((0 * 2 + h) * 16 + tap * 4 + cb);
                if (Cfg::WLO && ok) load_w((1 * 2 + h) * 16 + tap * 4 + cb);
              }
          for (int q = 0; q < 2 && ok; ++q)
            for (int kb = 0; kb < 4 && ok; ++kb) {
              load_w(64 + (0 * 2 + q) * 4 + kb);
              if (Cfg::WLO && ok) load_w(64 + (1 * 2 + q) * 4 + kb);
            }
        }
      }
    } else {
      // ================================ ring producers (P == 3) ================================
      constexpr int NP = 3;
      uint32_t pbits = 0, pbits2 = 0;                 // per-slot use parity of ring 1 / ring 2
      for (int l = p.l0; l < p.l1 && ok; ++l) {
        const int li = l - p.l0;
        const uint32_t prev = (li - 1) & 1;
        const int dil = 1 << (l % p.cycle);
        const int w_row0 = l * kRowsPerLayer;
        const CUtensorMap* ymap = p.tm_y[l & 1];
        bool y_ok = (li == 0) || !multi || !tile_valid, e_ok = (li == 0);
        if (li > 0) ok = mbar_wait(g2done, prev, wd, 105);            // ring-2 / z units of the previous layer are free
        if (prod_id == 0 && li < 10) DSX_TRACE(0, 200 + li);
        int ul = 0;                                                   // unit index within the layer
        // Slot of unit `ul` if it is this producer's, waited empty and armed; nullptr otherwise (check `ok`).
        auto acquire = [&](int code) -> uint8_t* {
          const int s = Cfg::slot(ul);
          const uint32_t par = ((pbits >> s) & 1) ^ 1;
          pbits ^= 1u << s;
          if (ul % NP != prod_id) return nullptr;
          if (!e_ok && s >= NU - Cfg::STG_UNITS) {                    // staging units: previous epilogue must be done
            ok = mbar_wait(edone, prev, wd, 106);
            e_ok = true;
            if (!ok) return nullptr;
          }
          ok = mbar_wait(&empty[s], par, wd, code);
          if (!ok) return nullptr;
          DSX_TRACE(0, ul);
          if (prank == 0) mbar_arrive_expect_tx(&full[s], G * kUnitBytes);
          return ring + s * kUnitBytes;
        };
        const unsigned int target = p.flag_base + static_cast<unsigned int>(kEpiWarps * li);
        bool yn_ok = y_ok;                                            // neighbours' y (halo taps)
        auto load_a = [&](int plane, int kb) {
          if (ul % NP == prod_id) {
            if (!y_ok) {                                              // centre tap: y_l of this tile
              ok = flag_wait(p.flags + tile, target, wd, 107);
              fence_proxy_async_all();
              y_ok = true;
            }
            if (ok && (kb >> 2) != 1 && !yn_ok) {                     // halo taps: y_l of the neighbour tiles
              if (nb_lo) ok = flag_wait(p.flags + tile - 1, target, wd, 108);
              if (ok && nb_hi) ok = flag_wait(p.flags + tile + 1, target, wd, 109);
              fence_proxy_async_all();
              yn_ok = true;
            }
            if (!ok) return;
          }
          const int s = Cfg::slot(ul);
          uint8_t* dst = acquire(101);
          if (dst) tma_load_3d<G>(&ymap[plane], &full[s], dst, (kb & 3) * 64, t0 + ((kb >> 2) - 1) * dil, bq, lead);
          ++ul;
        };
        auto load_w = [&](int tileidx) {
          const int s = Cfg::slot(ul);
          uint8_t* dst = acquire(102);
          if (dst) tma_load_2d<G>(&p.tm_w, &full[s], dst, 0, w_row0 + tileidx * 256 + static_cast<int>(prank) * 128, lead);
          ++ul;
        };
        for (int h = 0; h < 2 && ok; ++h)
          for (int ko = 0; ko < 12 && ok; ++ko) {
            const int kb = kb_order(ko);
            load_a(0, kb);
            if (ok) load_w((0 * 2 + h) * 16 + kb);
            if (ok) load_w((1 * 2 + h) * 16 + kb);
            if (ok) load_a(1, kb);
          }
        // GEMM2 weights: second ring over units 0..NU2-1, usable once every GEMM1 MMA has completed
        if (ok) ok = mbar_wait(g1done, li & 1, wd, 103);
        int u2 = 0;
        auto load_w2 = [&](int tileidx) {
          const int s = u2 % NU2;
          const uint32_t par = ((pbits2 >> s) & 1) ^ 1;
          pbits2 ^= 1u << s;
          if (u2 % NP == prod_id) {
            ok = mbar_wait(&empty2[s], par, wd, 104);
            if (!ok) return;
            DSX_TRACE(0, 128 + u2);
            if (prank == 0) mbar_arrive_expect_tx(&full2[s], G * kUnitBytes);
            tma_load_2d<G>(&p.tm_w, &full2[s], ring + s * kUnitBytes, 0,
                           w_row0 + tileidx * 256 + static_cast<int>(prank) * 128, lead);
          }
          ++u2;
        };
        for (int q = 0; q < 2 && ok; ++q)
          for (int kb = 0; kb < 4 && ok; ++kb) {
            load_w2(64 + (0 * 2 + q) * 4 + kb);
            if (ok) load_w2(64 + (1 * 2 + q) * 4 + kb);
          }
      }
    }
  } else if (warp == 1 && lane == 0 && prank == 0) {
    // ================================ MMA issuer (pair leader) ================================
    constexpr uint32_t idesc = umma_idesc_f16(128 * G, 256);
    uint32_t tuse[2] = {0, 0};
    bool ok = true;
    auto mma4 = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t& acc) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        umma_f16<G>(d, ad + 2 * k4, bd + 2 * k4, idesc, acc);
        acc = 1;
      }
    };
    // GEMM2 of one layer given a functor that multiplies z k-block kb (accumulator d) by the next weight tile(s)
    auto gemm2 = [&](int li, auto&& kblock) {
      for (int q = 0; q < 2 && ok; ++q) {
        ok = mbar_wait(&tempty[q], (tuse[q] & 1) ^ 1, wd, 204);
        if (!ok) break;
        tuse[q]++;
        DSX_TRACE(1, 202 + q);
        tc_fence_after();
        const uint32_t d = tmem_base + q * 256;
        uint32_t acc = 0;
        for (int kb = 0; kb < 4 && ok; ++kb) {
          if (q == 0 && kb >= 2) {                     // z k-blocks 2, 3 arrive from the chunk-1 gate epilogue
            ok = mbar_wait(&zf[kb - 2], li & 1, wd, 203);
            if (kb == 3) DSX_TRACE(1, 201);
            if (!ok) break;
            tc_fence_after();
          }
          kblock(d, q, kb, acc);
        }
        if (ok) umma_commit<G>(&tfull[q], pair_mask);
      }
      if (ok) umma_commit<G>(g2done, pair_mask);
      if (li < 10) DSX_TRACE(1, 220 + li);
    };
    if constexpr (Cfg::SHIFT) {
      uint32_t wi = 0, yi = 0;
      auto wait_w = [&](int code) -> uint64_t {        // next weight tile of the global order
        const uint32_t s = wi % Cfg::WSLOTS;
        ok = ok && mbar_wait(&full[s], (wi / Cfg::WSLOTS) & 1, wd, code);
        return umma_desc_sw128(smem_u32(ring + s * kUnitBytes));
      };
      auto done_w = [&]() {
        umma_commit<G>(&empty[wi % Cfg::WSLOTS], pair_mask);
        ++wi;
      };
      for (int l = p.l0; l < p.l1 && ok; ++l) {
        const int li = l - p.l0;
        const int dil = 1 << (l % p.cycle);
        for (int h = 0; h < 2 && ok; ++h) {
          ok = mbar_wait(&tempty[h], (tuse[h] & 1) ^ 1, wd, 201);
          if (!ok) break;
          tuse[h]++;
          tc_fence_after();
          const uint32_t d = tmem_base + h * 256;
          uint32_t acc = 0;
          if (h == 0 && li < 10) DSX_TRACE(1, 210 + li);            // TMEM buffer 0 free: GEMM1 of this layer may start
          for (int cb = 0; cb < 4 && ok; ++cb, ++yi) {
            const int ys = yi & 1;
            ok = mbar_wait(&yfull[ys], (yi >> 1) & 1, wd, 206);     // [8 halo | 128 centre | 8 halo] rows of 64 channels
            if (!ok) break;
            const uint64_t y = umma_desc_sw128(smem_u32(yslots + ys * Cfg::SLOT));
            DSX_TRACE(1, 4 + cb + 16 * h);
            if (h == 0 && cb == 0 && li < 10) DSX_TRACE(1, 230 + li);
            for (int tj = 0; tj < 3 && ok; ++tj) {
              const int tap = tj == 0 ? 1 : (tj == 1 ? 0 : 2);
              const uint64_t a = y + static_cast<uint64_t>(((8 + (tap - 1) * dil) * 128) >> 4);   // row-shifted start
              for (int pl = 0; pl < (Cfg::WLO ? 2 : 1) && ok; ++pl) {
                const uint64_t w = wait_w(207);
                if (!ok) break;
                tc_fence_after();
                mma4(d, a, w, acc);
                done_w();
              }
            }
            umma_commit<G>(&yempty[ys], pair_mask);                 // the y slot, after its last tap
          }
          if (ok) umma_commit<G>(&tfull[h], pair_mask);
        }
        DSX_TRACE(1, 200);
        gemm2(li, [&](uint32_t d, int, int kb, uint32_t& acc) {
          const uint64_t z_hi = umma_desc_sw128(smem_u32(zaddr(0, kb)));
          for (int pl = 0; pl < (Cfg::WLO ? 2 : 1) && ok; ++pl) {
            const uint64_t w = wait_w(205);
            if (!ok) break;
            tc_fence_after();
            mma4(d, z_hi, w, acc);
            done_w();
          }
        });
      }
    } else {
      uint32_t mbits = 0, mbits2 = 0;
      for (int l = p.l0; l < p.l1 && ok; ++l) {
        const int li = l - p.l0;
        int ul = 0, u2 = 0;
        auto wait_unit = [&](int uu, int code) -> uint64_t {
          const int s = Cfg::slot(uu);
          ok = ok && mbar_wait(&full[s], (mbits >> s) & 1, wd, code);
          mbits ^= 1u << s;
          return umma_desc_sw128(smem_u32(ring + s * kUnitBytes));
        };
        auto wait_unit2 = [&](int uu, int code) -> uint64_t {
          const int s = uu % NU2;
          ok = ok && mbar_wait(&full2[s], (mbits2 >> s) & 1, wd, code);
          mbits2 ^= 1u << s;
          return umma_desc_sw128(smem_u32(ring + s * kUnitBytes));
        };
        for (int h = 0; h < 2 && ok; ++h) {
          ok = mbar_wait(&tempty[h], (tuse[h] & 1) ^ 1, wd, 201);
          if (!ok) break;
          tuse[h]++;
          tc_fence_after();
          const uint32_t d = tmem_base + h * 256;
          uint32_t acc = 0;
          if (h == 0 && li < 10) DSX_TRACE(1, 210 + li);
          for (int ko = 0; ko < 12 && ok; ++ko) {
            const uint64_t a_hi = wait_unit(ul, 202);
            const uint64_t w_hi = wait_unit(ul + 1, 202);
            if (!ok) break;
            DSX_TRACE(1, ko + 16 * h);
            if (h == 0 && ko == 0 && li < 10) DSX_TRACE(1, 230 + li);
            tc_fence_after();
            mma4(d, a_hi, w_hi, acc);
            const uint64_t w_lo = wait_unit(ul + 2, 202);
            if (!ok) break;
            tc_fence_after();
            mma4(d, a_hi, w_lo, acc);
            const uint64_t a_lo = wait_unit(ul + 3, 202);
            if (!ok) break;
            tc_fence_after();
            mma4(d, a_lo, w_hi, acc);
            for (int i = 0; i < Cfg::UT; ++i) umma_commit<G>(&empty[Cfg::slot(ul + i)], pair_mask);
            ul += Cfg::UT;
          }
          if (ok) umma_commit<G>(&tfull[h], pair_mask);
        }
        if (ok) umma_commit<G>(g1done, pair_mask);
        DSX_TRACE(1, 200);
        gemm2(li, [&](uint32_t d, int, int kb, uint32_t& acc) {
          const uint64_t z_hi = umma_desc_sw128(smem_u32(zaddr(0, kb)));
          const uint64_t w_hi = wait_unit2(u2, 205);
          if (!ok) return;
          DSX_TRACE(1, 128 + u2);
          tc_fence_after();
          mma4(d, z_hi, w_hi, acc);
          const uint64_t w_lo = wait_unit2(u2 + 1, 205);
          if (!ok) return;
          tc_fence_after();
          mma4(d, z_hi, w_lo, acc);
          mma4(d, umma_desc_sw128(smem_u32(zaddr(1, kb))), w_hi, acc);
          for (int i = 0; i < Cfg::U2; ++i) umma_commit<G>(&empty2[(u2 + i) % NU2], pair_mask);
          u2 += Cfg::U2;
        });
      }
    }
  } else if (warp >= 4) {
    // ================================ epilogue (8 warps) ================================
    const int quad = warp & 3;                      // TMEM lane quadrant this warp may access
    const int half = (warp - 4) >> 2;               // which half of the columns
    const int r = quad * 32 + lane;                 // frame row in the tile == TMEM lane
    const uint32_t tlane = static_cast<uint32_t>(quad * 32) << 16;
    const bool tracer = (warp == 4 && lane == 0);
    uint32_t tf[2] = {0, 0};
    bool ok = true;
    auto release = [&](uint64_t* bar) {             // hand a TMEM buffer / z back to the pair leader's MMA thread
      if (lane == 0) mbar_arrive_remote(bar, lead);
    };
    // one lane polls the barrier; the warp reconverges on the shuffle
    auto wait_warp = [&](uint64_t* bar, uint32_t parity, int code) -> bool {
      int okv = 1;
      if (lane == 0) okv = mbar_wait(bar, parity, wd, code) ? 1 : 0;
      return __shfl_sync(0xffffffffu, okv, 0) != 0;
    };
    const uint64_t cp_policy = l2_policy_evict_first();
    uint8_t* stg = staging + (warp - 4) * 4096;
    const int lrow = lane >> 3;                               // epi2 reader: 8 lanes = one row of 32 columns (4 rows per access)
    const int lc4 = lane & 7;                                 // 4-column chunk within the 32-column group
    const int urow0 = tile_valid ? t0 + quad * 32 : p.T;      // first frame of this warp's 32 rows
    const int nrows = min(max(p.T - urow0, 0), 32);           // valid rows of this warp (warp-uniform)
    const size_t rbase = (static_cast<size_t>(tile_valid ? b : 0) * p.Tp + (tile_valid ? t0 + quad * 32 : 0) + lrow) * kC +
                         half * 128 + lc4 * 4;
    const uint8_t* stg_rd = stg + lrow * 128;

    for (int l = p.l0; l < p.l1 && ok; ++l) {
      const float* b2 = p.b2 + static_cast<size_t>(l) * 512;
      const bool skip_init = (l == 0);
      __half* const s16 = (l == p.L - 1) ? p.s16 : nullptr;
      __half* const yout = p.Y + static_cast<size_t>(((l + 1) & 1) * 2) * p.plane_elems;
      const float* dnext = (l + 1 < p.L) ? p.dtab + static_cast<size_t>(l + 1) * kC : nullptr;
      // ---- epi1: z = sigmoid(gate) * tanh(filter), gate/filter = accumulator + CP (conditioner projection + bias,
      //      streamed in the accumulator's own layout: one float4 = 4 columns of this thread's row).  A phase drains one
      //      accumulator in sub-passes of 16 gate/filter column pairs per warp; CP loads run one sub-pass ahead (the
      //      first is issued before the accumulator wait).
      //      Sub-passes 2*it, 2*it+1 of all 8 warps complete z k-block 2h + it, so GEMM2 can start on k-block 2 while
      //      k-block 3 is still being gated. ----
      const float* cpl = p.CP + (static_cast<size_t>(l) * p.tiles + cp_tile) * 2 * kCpChunk + r * 4;
      struct SubPass { int tg, tf, cpg, zkb, zchunk, zsig; };   // TMEM gate / filter column, CP gate column (filter + 128),
                                                                 // z k-block, first 16-byte chunk, zf barrier to signal or -1
      // CP double buffer in registers: sub-pass sp reads buffer sp & 1 while the loads of sub-pass sp + 1 fly -- also across
      // the chunk boundary (the first loads of chunk 1 are issued during the last sub-pass of chunk 0)
      float4 cg[2][4], cf[2][4];
      auto cp_issue = [&](const float* cph, int cpg, float4* g4, float4* f4) {
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4) {
          g4[v4] = ld_stream_f4(cph + ((cpg >> 2) + v4) * (kTile * 4), cp_policy);
          f4[v4] = ld_stream_f4(cph + (((128 + cpg) >> 2) + v4) * (kTile * 4), cp_policy);
        }
      };
      auto epi1_phase = [&](int bar, const float* cph, auto geom, int trace0, bool preloaded, const float* next_cph,
                            auto next_geom) -> bool {
        constexpr int NSP = 4;
        if (!preloaded) cp_issue(cph, geom(0).cpg, cg[0], cf[0]);
        if (tracer) DSX_TRACE(2, trace0);
        if (!wait_warp(&tfull[bar], tf[bar] & 1, 301)) return false;
        if (tracer) DSX_TRACE(2, trace0 + 1);
        tf[bar]++;
        tc_fence_after();
#pragma unroll
        for (int sp = 0; sp < NSP; ++sp) {
          const SubPass sg = geom(sp);
          if (sp + 1 < NSP) cp_issue(cph, geom(sp + 1).cpg, cg[(sp + 1) & 1], cf[(sp + 1) & 1]);
          else if (next_cph) cp_issue(next_cph, next_geom(0).cpg, cg[0], cf[0]);
          uint8_t* zrow = zaddr(0, sg.zkb) + r * 128;
          uint8_t* zrow_lo = zaddr(1, sg.zkb) + r * 128;
          uint32_t g[16], f[16];
          tmem_ld_32x16(tmem_base + tlane + sg.tg, g);
          tmem_ld_32x16(tmem_base + tlane + sg.tf, f);
          tmem_ld_wait();
#pragma unroll
          for (int c8 = 0; c8 < 2; ++c8) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; e += 2) {
              const int i = c8 * 8 + e * 2;
              const float4 bgv = cg[sp & 1][i >> 2];
              const float4 bfv = cf[sp & 1][i >> 2];
              float z4[4];
              const float vg[4] = {__uint_as_float(g[i]) + bgv.x, __uint_as_float(g[i + 1]) + bgv.y,
                                   __uint_as_float(g[i + 2]) + bgv.z, __uint_as_float(g[i + 3]) + bgv.w};
              const float vf[4] = {__uint_as_float(f[i]) + bfv.x, __uint_as_float(f[i + 1]) + bfv.y,
                                   __uint_as_float(f[i + 2]) + bfv.z, __uint_as_float(f[i + 3]) + bfv.w};
#pragma unroll
              for (int q4 = 0; q4 < 4; ++q4)
                z4[q4] = (P == 1) ? sigmoid_fast(vg[q4]) * tanh_approx(vf[q4]) : gate_acc(vg[q4], vf[q4]);
              const __half2 h01 = __floats2half2_rn(z4[0], z4[1]), h23 = __floats2half2_rn(z4[2], z4[3]);
              hi[e] = h2_bits(h01);
              hi[e + 1] = h2_bits(h23);
              if (Cfg::ALO_T) {
                const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                lo[e] = h2_bits(__floats2half2_rn(z4[0] - f01.x, z4[1] - f01.y));
                lo[e + 1] = h2_bits(__floats2half2_rn(z4[2] - f23.x, z4[3] - f23.y));
              }
            }
            const int off = ((sg.zchunk + c8) ^ (r & 7)) << 4;
            *reinterpret_cast<uint4*>(zrow + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            if (Cfg::ALO_T) *reinterpret_cast<uint4*>(zrow_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
          if (sg.zsig >= 0) {
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            release(&zf[sg.zsig]);
          }
        }
        tc_fence_before();
        fence_proxy_async_smem();
        __syncwarp();
        if (tracer) DSX_TRACE(2, trace0 + 2);
        release(&tempty[bar]);
        return true;
      };
      auto wide = [&](int h) {
        return [=](int sp) {
          const int it = sp >> 1, sub = sp & 1, c = it * 64 + half * 32 + sub * 16;
          return SubPass{h * 256 + c, h * 256 + 128 + c, c, 2 * h + it, half * 4 + sub * 2, (h == 1 && sub == 1) ? it : -1};
        };
      };
      ok = epi1_phase(0, cpl, wide(0), 0, false, cpl + kCpChunk, wide(1));
      if (ok) ok = epi1_phase(1, cpl + kCpChunk, wide(1), 4, true, nullptr, wide(1));
      if (!ok) break;
      // ---- epi2: each warp moves its 32 rows x 32 columns through a swizzled shared-memory tile so that every
      //      global access instruction covers whole 128-byte row segments (4 rows x 32 columns of fp32, 16 bytes per
      //      lane: the LSU instruction queue is what throttles this phase).  All addresses are one base pointer per
      //      thread plus compile-time offsets; the row-validity test is hoisted (only the last tile of an utterance
      //      takes the predicated path). ----
      auto epi2_half = [&](auto full_tag, int q) {
        constexpr bool FULL = decltype(full_tag)::value;
        float* const gp = ((q == 0) ? p.X : p.SKIP) + rbase;
        __half* const yp = yout + rbase;
        __half* const sp = s16 ? s16 + rbase : nullptr;
        const int mode = (q == 0) ? 0 : (skip_init ? 1 : (s16 ? 2 : 3));   // 0 residual, 1 store, 2 load+add (+s16), 3 red.add
        const bool do_load = (mode == 0 || mode == 2);
        const float* dn = (q == 0 && dnext) ? dnext + static_cast<size_t>(tile_valid ? b : 0) * p.d_row_stride + half * 128 + lc4 * 4 : nullptr;
        const float* bp = b2 + q * 256 + half * 128 + lc4 * 4;
        // per-column vectors of the four 32-column groups: requested before the accumulator wait (these come
        // from L2: the proxy / gpu fences of the hand-over invalidate L1)
        float4 biasv[4], dnvv[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          biasv[jj] = __ldg(reinterpret_cast<const float4*>(bp + jj * 32));
          dnvv[jj] = dn ? __ldg(reinterpret_cast<const float4*>(dn + jj * 32)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float4 pre[8];
        auto prefetch = [&](int j) {
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            pre[it] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (do_load && (FULL || it * 4 + lrow < nrows)) pre[it] = *reinterpret_cast<const float4*>(gp + it * 4 * kC + j);
          }
        };
        prefetch(0);
        if (tracer) DSX_TRACE(2, 8 + 2 * q);
        if (!wait_warp(&tfull[q], tf[q] & 1, 302 + q)) return false;
        if (tracer) DSX_TRACE(2, 9 + 2 * q);
        tf[q]++;
        tc_fence_after();
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int j = jj * 32;
          uint32_t o[32];
          tmem_ld_32x32(tmem_base + tlane + q * 256 + half * 128 + j, o);
          tmem_ld_wait();
          __syncwarp();
#pragma unroll
          for (int c = 0; c < 8; ++c)
            *reinterpret_cast<uint4*>(stg + lane * 128 + ((c ^ (lane & 7)) << 4)) =
                make_uint4(o[c * 4], o[c * 4 + 1], o[c * 4 + 2], o[c * 4 + 3]);
          __syncwarp();
          const float4 bias = biasv[jj], dnv = dnvv[jj];
          float4 res[8];
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            // row rr = 4*it + lrow; its 16-byte chunk lc4 sits at position lc4 ^ (rr & 7)
            const float4 d = *reinterpret_cast<const float4*>(stg_rd + it * 512 + ((lc4 ^ ((it * 4 + lrow) & 7)) << 4));
            float4 v = pre[it];
            if (mode == 0) {
              v.x = (v.x + (d.x + bias.x)) * 0.70710678118654752440f;
              v.y = (v.y + (d.y + bias.y)) * 0.70710678118654752440f;
              v.z = (v.z + (d.z + bias.z)) * 0.70710678118654752440f;
              v.w = (v.w + (d.w + bias.w)) * 0.70710678118654752440f;
            } else {
              v.x += d.x + bias.x;
              v.y += d.y + bias.y;
              v.z += d.z + bias.z;
              v.w += d.w + bias.w;
            }
            res[it] = v;
          }
          if (j + 32 < 128) prefetch(j + 32);                   // next group's loads fly while this one is stored
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            if (FULL || it * 4 + lrow < nrows) {
              const float4 v = res[it];
              float* g = gp + it * 4 * kC + j;
              if (mode != 3) {
                *reinterpret_cast<float4*>(g) = v;
              } else {
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(g), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                             : "memory");
              }
              if (mode == 2) {
                const float sa = v.x * p.inv_sqrt_l, sb = v.y * p.inv_sqrt_l, sc = v.z * p.inv_sqrt_l, sd = v.w * p.inv_sqrt_l;
                const __half2 h0 = __floats2half2_rn(sa, sb), h1 = __floats2half2_rn(sc, sd);
                *reinterpret_cast<uint2*>(sp + it * 4 * kC + j) = make_uint2(h2_bits(h0), h2_bits(h1));
                if (P >= 2) {
                  const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
                  *reinterpret_cast<uint2*>(sp + p.plane_elems + it * 4 * kC + j) =
                      make_uint2(h2_bits(__floats2half2_rn(sa - f0.x, sb - f0.y)), h2_bits(__floats2half2_rn(sc - f1.x, sd - f1.y)));
                }
              }
              if (dn) {
                const float ya = v.x + dnv.x, yb = v.y + dnv.y, yc = v.z + dnv.z, yd = v.w + dnv.w;
                const __half2 h0 = __floats2half2_rn(ya, yb), h1 = __floats2half2_rn(yc, yd);
                *reinterpret_cast<uint2*>(yp + it * 4 * kC + j) = make_uint2(h2_bits(h0), h2_bits(h1));
                if (Cfg::ALO_T) {
                  const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
                  *reinterpret_cast<uint2*>(yp + p.plane_elems + it * 4 * kC + j) =
                      make_uint2(h2_bits(__floats2half2_rn(ya - f0.x, yb - f0.y)), h2_bits(__floats2half2_rn(yc - f1.x, yd - f1.y)));
                }
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        release(&tempty[q]);
        return true;
      };
      for (int q = 0; q < 2 && ok; ++q) {
        ok = (nrows == 32) ? epi2_half(std::true_type{}, q) : epi2_half(std::false_type{}, q);
        if (q == 0 && ok && multi && l + 1 < p.l1 && tile_valid) {   // (nobody waits on a padding tile)
          // publish y_{l+1}: generic-proxy global stores of every lane -> async-proxy (TMA) readers in this CTA and
          // its neighbours.  Proxy fence + gpu fence per lane, warp sync, then one release-increment per warp.
          fence_proxy_async_all();
          __threadfence();
          __syncwarp();
          if (lane == 0) flag_publish(p.flags + tile);
        }
        if (tracer && l - p.l0 < 10) DSX_TRACE(2, 100 + q * 10 + (l - p.l0));
      }
      if (!Cfg::SHIFT && ok && multi && l + 1 < p.l1) {           // P == 3: the staging units go back to the ring
        __syncwarp();
        if (lane == 0) mbar_arrive(edone);
      }
    }
    if (tracer) DSX_TRACE(2, 12);
  }
  if (threadIdx.x == 0) DSX_TRACE(0, 255);

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  cluster_arrive();
  cluster_wait();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<G>(tmem_base, 512);
  }
  if (threadIdx.x == 64) {
    DSX_TRACE(0, 251);                                           // after TMEM free (clock64)
    if (p.trace && blockIdx.x < 2) p.trace[(blockIdx.x * 3 + 1) * 256 + 251] = static_cast<long long>(globaltimer_ns());
    if (p.trace && blockIdx.x == 0) p.trace[221 + (p.seq % 8) * 2] = static_cast<long long>(globaltimer_ns());
  }
}

// ==========================================================================================
// Conditioner projection of every residual layer (usr/diff/net.py:56,70: conditioner_projection(cond), plus the
// summed dilated_conv / conditioner_projection biases), hoisted out of the sampling loop: it does not depend on the
// diffusion step.  CP[l][tile][chunk h][column group][row][4] (fp32) is laid out exactly as the layer kernel's epi1
// reads its accumulator: thread = row, one float4 = 4 consecutive accumulator columns.
//   D[128 x 256] = cond_tile (K = 256, hi+lo) . Wc(l, h)^T (hi+lo), 3 passes, fp32 accumulate; + b1p
// cta_group::1, one CTA per (tile, slice of the 2L (layer, chunk) jobs): the conditioner tile stays resident in shared
// memory (8 x 16 KB), the weight tiles (256 rows x 64, 32 KB) stream through a 3-deep ring, two TMEM accumulators.
// ==========================================================================================
struct TcCondParams {
  CUtensorMap tm_w;        // packed weights, box 64 x 128 rows
  CUtensorMap tm_cond[2];  // conditioner planes hi / lo
  float* CP;
  const float* b1p;        // [L][2][256] biases in accumulator column order
  int T, Tp, tiles_per_utt, tiles, B, L;
  int* status;
  unsigned long long budget_ns;
};
constexpr int kCondStages = 3;
constexpr int kCondSmem = 1024 + 8 * kUnitBytes + kCondStages * 2 * kUnitBytes + 256;

__global__ void __launch_bounds__(kThreads, 1) k_tc_condproj(const __grid_constant__ TcCondParams p) {
  constexpr int NS = kCondStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* abuf = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = abuf + 8 * kUnitBytes;                      // NS stages of one 256-row weight tile
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring + NS * 2 * kUnitBytes);
  uint64_t* full = bars;            // [NS]
  uint64_t* empty = full + NS;      // [NS]
  uint64_t* tfull = empty + NS;     // [2]
  uint64_t* tempty = tfull + 2;     // [2]
  uint64_t* afull = tempty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(afull + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x;
  const int b = tile / p.tiles_per_utt;
  const int t0 = (tile % p.tiles_per_utt) * kTile;
  const int njobs = 2 * p.L;
  const int j0 = static_cast<int>(static_cast<long long>(njobs) * blockIdx.y / gridDim.y);
  const int j1 = static_cast<int>(static_cast<long long>(njobs) * (blockIdx.y + 1) / gridDim.y);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tm_w);
    tma_prefetch_desc(&p.tm_cond[0]);
    tma_prefetch_desc(&p.tm_cond[1]);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kEpiWarps);
    }
    mbar_init(afull, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc<1>(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  Watchdog wd{p.status, globaltimer_ns() + p.budget_ns};

  const int prod_id = (warp == 0) ? 0 : (warp == 2 ? 1 : (warp == 3 ? 2 : -1));
  if (prod_id >= 0 && lane == 0) {
    // ---- TMA producers: thread 0 brings the conditioner tile, all three take the weight tiles round-robin ----
    if (prod_id == 0) {
      mbar_arrive_expect_tx(afull, 8 * kUnitBytes);
      for (int pl = 0; pl < 2; ++pl)
        for (int kb = 0; kb < 4; ++kb) tma_load_3d<1>(&p.tm_cond[pl], afull, abuf + (pl * 4 + kb) * kUnitBytes, kb * 64, t0, b);
    }
    uint32_t u = 0;
    bool ok = true;
    for (int j = j0; j < j1 && ok; ++j) {
      const int l = j >> 1, h = j & 1;
      for (int kb = 0; kb < 4 && ok; ++kb)
        for (int pl = 0; pl < 2 && ok; ++pl, ++u) {
          if (u % 3 != static_cast<uint32_t>(prod_id)) continue;
          const int s = u % NS;
          ok = mbar_wait(&empty[s], ((u / NS) & 1) ^ 1, wd, 121);
          if (!ok) break;
          mbar_arrive_expect_tx(&full[s], 2 * kUnitBytes);
          const int row = l * kRowsPerLayer + ((pl * 2 + h) * 16 + 12 + kb) * 256;
          tma_load_2d<1>(&p.tm_w, &full[s], ring + s * 2 * kUnitBytes, 0, row);
          tma_load_2d<1>(&p.tm_w, &full[s], ring + s * 2 * kUnitBytes + kUnitBytes, 0, row + 128);
        }
    }
  } else if (warp == 1 && lane == 0) {
    // ---- MMA issuer ----
    constexpr uint32_t idesc = umma_idesc_f16(128, 256);
    auto mma4 = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t& acc) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        umma_f16<1>(d, ad + 2 * k4, bd + 2 * k4, idesc, acc);
        acc = 1;
      }
    };
    bool ok = mbar_wait(afull, 0, wd, 221);
    tc_fence_after();
    uint32_t u = 0;
    for (int j = j0; j < j1 && ok; ++j) {
      const int jj = j - j0, buf = jj & 1;
      ok = mbar_wait(&tempty[buf], ((jj >> 1) & 1) ^ 1, wd, 222);
      if (!ok) break;
      tc_fence_after();
      const uint32_t d = tmem_base + buf * 256;
      uint32_t acc = 0;
      for (int kb = 0; kb < 4 && ok; ++kb) {
        const uint64_t a_hi = umma_desc_sw128(smem_u32(abuf + kb * kUnitBytes));
        const uint64_t a_lo = umma_desc_sw128(smem_u32(abuf + (4 + kb) * kUnitBytes));
        for (int pl = 0; pl < 2 && ok; ++pl, ++u) {
          const int s = u % NS;
          ok = mbar_wait(&full[s], (u / NS) & 1, wd, 223);
          if (!ok) break;
          tc_fence_after();
          const uint64_t w = umma_desc_sw128(smem_u32(ring + s * 2 * kUnitBytes));
          mma4(d, a_hi, w, acc);                      // A_hi.W_hi, A_hi.W_lo
          if (pl == 0) mma4(d, a_lo, w, acc);         // A_lo.W_hi
          umma_commit<1>(&empty[s]);
        }
      }
      if (ok) umma_commit<1>(&tfull[buf]);
    }
  } else if (warp >= 4) {
    // ---- epilogue: accumulator + bias -> CP ----
    const int quad = warp & 3, half = (warp - 4) >> 2;
    const int r = quad * 32 + lane;
    const uint32_t tlane = static_cast<uint32_t>(quad * 32) << 16;
    bool ok = true;
    for (int j = j0; j < j1 && ok; ++j) {
      const int l = j >> 1, h = j & 1, jj = j - j0, buf = jj & 1;
      int okv = 1;
      if (lane == 0) okv = mbar_wait(&tfull[buf], (jj >> 1) & 1, wd, 321) ? 1 : 0;
      ok = __shfl_sync(0xffffffffu, okv, 0) != 0;
      if (!ok) break;
      tc_fence_after();
      float* dst = p.CP + ((static_cast<size_t>(l) * p.tiles + tile) * 2 + h) * kCpChunk + r * 4;
      const float* bias = p.b1p + (static_cast<size_t>(l) * 2 + h) * 256;
#pragma unroll 1
      for (int c0 = half * 128; c0 < half * 128 + 128; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + tlane + buf * 256 + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 bb = __ldg(reinterpret_cast<const float4*>(bias + c0) + c4);
          float4 o;
          o.x = __uint_as_float(v[c4 * 4]) + bb.x;
          o.y = __uint_as_float(v[c4 * 4 + 1]) + bb.y;
          o.z = __uint_as_float(v[c4 * 4 + 2]) + bb.z;
          o.w = __uint_as_float(v[c4 * 4 + 3]) + bb.w;
          *reinterpret_cast<float4*>(dst + ((c0 >> 2) + c4) * (kTile * 4)) = o;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512);
  }
}

// ==========================================================================================
// Head / tail of DiffNet on tensor cores (usr/diff/net.py:115-118 and 126-130), one CTA per 128-frame tile:
//   H1   h   = relu(W_s . (skip_sum / sqrt L) + b_s)            A = S16 planes written by the last layer
//   H2   eps = W_out . h + b_out                                 N = 80 padded to 128
//   mel  DDPM update of the mel state x with eps (shallow_diffusion_tts.py:134-166), thread = frame
//   I    x0  = relu(W_in . x + b_in), y0 = fp16 split of (x0 + d_0)  -> residual stream of the NEXT evaluation
// Any subset runs (flags); the in-projection alone starts a sampling loop or a forward call.
// cta_group::1, UMMA M = 128, N = 128 per instruction (two column halves for the 256-wide outputs).
// ==========================================================================================
struct TcHeadParams {
  CUtensorMap tm_s16[2];   // 3D [B][T][256] hi/lo
  CUtensorMap tm_wh;       // 2D [32 tiles x 128 rows][64], box 64 x 128
  float* x;                // mel state (in/out), addressed through xs
  dsx_strides xs;
  float* eps;              // [B][M][T] contiguous (TC_WRITE_EPS)
  const float* noise;      // [B][M][T] for this step, or nullptr -> Philox
  unsigned long long seed, offset;
  int b_off;               // global index of utterance 0 (Philox counters of a sharded batch)
  DdpmCoef c;
  PlmsFuse pl;             // TC_PLMS
  float* X;                // [B][Tp][256]
  __half* Y;               // conv input of layer 0, plane 0; plane 1 at + plane_elems
  size_t plane_elems;
  const float* bs;         // skip_projection.bias   [256]
  const float* bf;         // output_projection.bias [M]
  const float* bin;        // input_projection.bias  [256]
  const float* d0;         // FiLM vector of layer 0 (row base of the evaluation being prepared)
  int d_row_stride;
  int T, Tp, tiles_per_utt, tiles, B, M;
  int flags;
  int* status;
  unsigned long long budget_ns;
  long long* trace;        // debug: CTA 0 writes clock64 stamps at [2*256 + 100 ...]
  int seq;                 // debug: launch sequence number
};

#define DSX_HTRACE(slot)                                                        \
  do {                                                                          \
    if (p.trace && blockIdx.x == 0 && warp == 4 && lane == 0) p.trace[2 * 256 + 100 + (slot)] = clock64(); \
  } while (0)

template <int P>
struct HeadCfg {
  static constexpr int UNITS = (P == 1) ? 9 : 5;              // ring of the H2 / I phases
  static constexpr int Z_PLANES = (P == 1) ? 1 : 2;
  static constexpr int H_BYTES = Z_PLANES * 4 * kUnitBytes;
  static constexpr int UNITS_H1 = UNITS + H_BYTES / kUnitBytes;   // H1 also streams through the not-yet-written h buffer
  static constexpr int SMEM_BYTES = 1024 + UNITS * kUnitBytes + H_BYTES + kStagingBytes + 512;
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
};

template <int P>
__global__ void __launch_bounds__(kThreads, 1) k_tc_head(const __grid_constant__ TcHeadParams p) {
  using Cfg = HeadCfg<P>;
  constexpr int NU = Cfg::UNITS;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* hbuf = ring + NU * kUnitBytes;                       // h [planes][4 k-blocks]; x_in aliases k-blocks 0,1
  uint8_t* staging = hbuf + Cfg::H_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + kStagingBytes);
  uint64_t* full = bars;           // [NU]
  uint64_t* empty = full + NU;     // [NU]
  constexpr int NA = Cfg::UNITS_H1;
  uint64_t* fullA = empty + NU;    // [NA]  H1 ring (ring + h buffer)
  uint64_t* emptyA = fullA + NA;   // [NA]
  uint64_t* tf = emptyA + NA;      // [3]  accumulator ready: H1, H2, I
  uint64_t* hfull = tf + 3;        // h written
  uint64_t* xfull = hfull + 1;     // x_in written
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xfull + 1);
  auto hk = [&](int plane, int kb) -> uint8_t* { return hbuf + (plane * 4 + kb) * kUnitBytes; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x;
  const int b = tile / p.tiles_per_utt;
  const int t0 = (tile % p.tiles_per_utt) * kTile;
  const bool do_head = p.flags & TC_HEAD, do_in = p.flags & TC_INPROJ;
  if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) {        // wall-clock entry stamp (tools/trace_gaps.py)
    p.trace[5 * 256 + 220 + (p.seq % 8) * 2] = static_cast<long long>(globaltimer_ns());
    p.trace[2 * 256 + 98] = clock64();
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tm_wh);
    tma_prefetch_desc(&p.tm_s16[0]);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NU; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < NA; ++s) {
      mbar_init(&fullA[s], 1);
      mbar_init(&emptyA[s], 1);
    }
    for (int i = 0; i < 3; ++i) mbar_init(&tf[i], 1);
    mbar_init(hfull, kEpiWarps);
    mbar_init(xfull, kEpiWarps);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc<1>(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  Watchdog wd{p.status, globaltimer_ns() + p.budget_ns};

  const int prod_id = (warp == 0) ? 0 : (warp == 2 ? 1 : (warp == 3 ? 2 : -1));
  if (prod_id >= 0 && lane == 0) {
    // ================================ TMA producers ================================
    // three threads take the units round-robin (one thread gets one load accepted per ~430 cycles: dsx_selftest(3))
    constexpr uint32_t NP = 3;
    uint32_t u = 0;
    bool ok = true;
    // slot of unit `u` if it is this producer's (waited empty and armed), else nullptr; always advances u
    auto acquire = [&](int code, uint64_t*& bar) -> uint8_t* {
      const uint32_t uu = u++;
      if (uu % NP != static_cast<uint32_t>(prod_id) || !ok) return nullptr;
      const int s = uu % NU;
      ok = mbar_wait(&empty[s], ((uu / NU) & 1) ^ 1, wd, code);
      if (!ok) return nullptr;
      mbar_arrive_expect_tx(&full[s], kUnitBytes);
      bar = &full[s];
      return ring + s * kUnitBytes;
    };
    auto load_w = [&](int tileidx) {
      uint64_t* bar = nullptr;
      uint8_t* dst = acquire(112, bar);
      if (dst) tma_load_2d<1>(&p.tm_wh, bar, dst, 0, tileidx * 128);
    };
    if (do_head) {
      // H1 streams through ring A = ring + h buffer (h is only written after H1's accumulator is complete)
      uint32_t ua = 0;
      auto acquireA = [&](uint64_t*& bar) -> uint8_t* {
        const uint32_t uu = ua++;
        if (uu % NP != static_cast<uint32_t>(prod_id) || !ok) return nullptr;
        const int s = uu % NA;
        ok = mbar_wait(&emptyA[s], ((uu / NA) & 1) ^ 1, wd, 113);
        if (!ok) return nullptr;
        mbar_arrive_expect_tx(&fullA[s], kUnitBytes);
        bar = &fullA[s];
        return ring + s * kUnitBytes;
      };
      auto loadA_a = [&](int plane, int kb) {
        uint64_t* bar = nullptr;
        uint8_t* dst = acquireA(bar);
        if (dst) tma_load_3d<1>(&p.tm_s16[plane], bar, dst, kb * 64, t0, b);
      };
      auto loadA_w = [&](int tileidx) {
        uint64_t* bar = nullptr;
        uint8_t* dst = acquireA(bar);
        if (dst) tma_load_2d<1>(&p.tm_wh, bar, dst, 0, tileidx * 128);
      };
      for (int kb = 0; kb < 4 && ok; ++kb) {
        loadA_a(0, kb);
        loadA_w((0 * 2 + 0) * 4 + kb);
        loadA_w((0 * 2 + 1) * 4 + kb);
        if (P == 3) {
          loadA_w((1 * 2 + 0) * 4 + kb);
          loadA_w((1 * 2 + 1) * 4 + kb);
          loadA_a(1, kb);
        }
      }
      // the H2 / I weights use the small ring, whose units alias ring A: wait for H1's MMAs
      if (ok) ok = mbar_wait(&tf[0], 0, wd, 114);
      for (int kb = 0; kb < 4 && ok; ++kb) {
        load_w(16 + 0 * 4 + kb);
        if (P == 3) load_w(16 + 1 * 4 + kb);
      }
    }
    if (do_in) {
      for (int kb = 0; kb < 2 && ok; ++kb) {
        load_w(24 + (0 * 2 + 0) * 2 + kb);
        load_w(24 + (0 * 2 + 1) * 2 + kb);
        if (P == 3) {
          load_w(24 + (1 * 2 + 0) * 2 + kb);
          load_w(24 + (1 * 2 + 1) * 2 + kb);
        }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ================================ MMA issuer ================================
    constexpr uint32_t idesc = umma_idesc_f16(128, 128);
    uint32_t u = 0;
    bool ok = true;
    auto wait_unit = [&](uint32_t uu, int code) -> uint64_t {
      const int s = uu % NU;
      ok = ok && mbar_wait(&full[s], (uu / NU) & 1, wd, code);
      return umma_desc_sw128(smem_u32(ring + s * kUnitBytes));
    };
    auto mma4 = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t& acc) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        umma_f16<1>(d, ad + 2 * k4, bd + 2 * k4, idesc, acc);
        acc = 1;
      }
    };
    auto release = [&](int n) {
      for (int i = 0; i < n; ++i) umma_commit<1>(&empty[(u + i) % NU]);
      u += n;
    };
    if (do_head) {
      uint32_t acc0 = 0, acc1 = 0, ua = 0;
      auto waitA = [&](uint32_t uu) -> uint64_t {
        const int s = uu % NA;
        ok = ok && mbar_wait(&fullA[s], (uu / NA) & 1, wd, 211);
        return umma_desc_sw128(smem_u32(ring + s * kUnitBytes));
      };
      for (int kb = 0; kb < 4 && ok; ++kb) {
        const uint64_t a_hi = waitA(ua), w0 = waitA(ua + 1), w1 = waitA(ua + 2);
        if (!ok) break;
        tc_fence_after();
        mma4(tmem_base, a_hi, w0, acc0);
        mma4(tmem_base + 128, a_hi, w1, acc1);
        if (P == 3) {
          const uint64_t l0 = waitA(ua + 3), l1 = waitA(ua + 4), a_lo = waitA(ua + 5);
          if (!ok) break;
          tc_fence_after();
          mma4(tmem_base, a_hi, l0, acc0);
          mma4(tmem_base + 128, a_hi, l1, acc1);
          mma4(tmem_base, a_lo, w0, acc0);
          mma4(tmem_base + 128, a_lo, w1, acc1);
        }
        const int nrel = (P == 1) ? 3 : 6;
        for (int i = 0; i < nrel; ++i) umma_commit<1>(&emptyA[(ua + i) % NA]);
        ua += nrel;
      }
      if (ok) umma_commit<1>(&tf[0]);
      if (ok) ok = mbar_wait(hfull, 0, wd, 212);
      tc_fence_after();
      uint32_t acc = 0;
      for (int kb = 0; kb < 4 && ok; ++kb) {
        const uint64_t h_hi = umma_desc_sw128(smem_u32(hk(0, kb)));
        const uint64_t w = wait_unit(u, 213);
        if (!ok) break;
        tc_fence_after();
        mma4(tmem_base + 256, h_hi, w, acc);
        if (P == 3) {
          const uint64_t wl = wait_unit(u + 1, 213);
          if (!ok) break;
          tc_fence_after();
          mma4(tmem_base + 256, h_hi, wl, acc);
          mma4(tmem_base + 256, umma_desc_sw128(smem_u32(hk(1, kb))), w, acc);
        }
        release(P == 1 ? 1 : 2);
      }
      if (ok) umma_commit<1>(&tf[1]);
    }
    if (do_in) {
      if (ok) ok = mbar_wait(xfull, 0, wd, 214);
      tc_fence_after();
      uint32_t acc0 = 0, acc1 = 0;
      for (int kb = 0; kb < 2 && ok; ++kb) {
        const uint64_t x_hi = umma_desc_sw128(smem_u32(hk(0, kb)));
        const uint64_t w0 = wait_unit(u, 215), w1 = wait_unit(u + 1, 215);
        if (!ok) break;
        tc_fence_after();
        mma4(tmem_base, x_hi, w0, acc0);
        mma4(tmem_base + 128, x_hi, w1, acc1);
        if (P == 3) {
          const uint64_t l0 = wait_unit(u + 2, 215), l1 = wait_unit(u + 3, 215);
          if (!ok) break;
          tc_fence_after();
          const uint64_t x_lo = umma_desc_sw128(smem_u32(hk(1, kb)));
          mma4(tmem_base, x_hi, l0, acc0);
          mma4(tmem_base + 128, x_hi, l1, acc1);
          mma4(tmem_base, x_lo, w0, acc0);
          mma4(tmem_base + 128, x_lo, w1, acc1);
        }
        release(P == 1 ? 2 : 4);
      }
      if (ok) umma_commit<1>(&tf[2]);
    }
  } else if (warp >= 4) {
    // ================================ epilogue (8 warps) ================================
    const int quad = warp & 3, half = (warp - 4) >> 2;
    const int r = quad * 32 + lane;
    const uint32_t tlane = static_cast<uint32_t>(quad * 32) << 16;
    const int t = t0 + r;
    const bool row_valid = t < p.T;
    bool ok = true;
    auto wait_warp = [&](uint64_t* bar, uint32_t parity, int code) -> bool {
      int okv = 1;
      if (lane == 0) okv = mbar_wait(bar, parity, wd, code) ? 1 : 0;
      return __shfl_sync(0xffffffffu, okv, 0) != 0;
    };
    DSX_HTRACE(0);
    if (do_head) {
      // ---- epi-H1: h = relu(D1 + b_s) -> fp16 planes, K-major swizzled rows ----
      ok = wait_warp(&tf[0], 0, 311);
      DSX_HTRACE(1);
      if (ok) {
        tc_fence_after();
#pragma unroll 1
        for (int j = 0; j < 128; j += 32) {
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + tlane + half * 128 + j, v);
          tmem_ld_wait();
          const int ch0 = half * 128 + j, kb = ch0 >> 6, chunk0 = (ch0 & 63) >> 3;
#pragma unroll
          for (int c8 = 0; c8 < 4; ++c8) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int i = c8 * 8 + e * 2;
              const float2 bb = __ldg(reinterpret_cast<const float2*>(p.bs + ch0 + i));
              const float a0 = fmaxf(__uint_as_float(v[i]) + bb.x, 0.f), a1 = fmaxf(__uint_as_float(v[i + 1]) + bb.y, 0.f);
              const __half2 hh = __floats2half2_rn(a0, a1);
              hi[e] = h2_bits(hh);
              if (P == 3) {
                const float2 hf = __half22float2(hh);
                lo[e] = h2_bits(__floats2half2_rn(a0 - hf.x, a1 - hf.y));
              }
            }
            const int off = r * 128 + (((chunk0 + c8) ^ (r & 7)) << 4);
            *reinterpret_cast<uint4*>(hk(0, kb) + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            if (P == 3) *reinterpret_cast<uint4*>(hk(1, kb) + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
        tc_fence_before();
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(hfull);
      }
      DSX_HTRACE(2);
    }
    // ---- mel phase: eps, DDPM update, x_in operand.  half 0: bins [0,40), half 1: bins [40,80), 8 bins a time ----
    if (ok && do_head) ok = wait_warp(&tf[1], 0, 312);
    DSX_HTRACE(3);
    if (ok) {
      tc_fence_after();
      const int m_lo = half * 40;
      const bool need_x = (p.flags & (TC_UPDATE | TC_INPROJ | TC_PLMS)) != 0;
      const bool need_z = (p.flags & TC_UPDATE) && p.c.sigma != 0.f;
      const size_t xrow = static_cast<size_t>(b) * p.xs.b + static_cast<size_t>(t) * p.xs.t;
#pragma unroll 1
      for (int m0 = m_lo; m0 < m_lo + 40; m0 += 8) {
        uint32_t e8[8];
        if (do_head) tmem_ld_32x8(tmem_base + tlane + 256 + m0, e8);
        float xv[8], zn[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          xv[i] = 0.f;
          zn[i] = 0.f;
          if (row_valid && need_x) xv[i] = p.x[xrow + static_cast<size_t>(m0 + i) * p.xs.c];
        }
        if (need_z && row_valid) {
          if (p.noise) {
#pragma unroll
            for (int i = 0; i < 8; ++i) zn[i] = p.noise[(static_cast<size_t>(b) * p.M + m0 + i) * p.T + t];
          } else {
#pragma unroll
            for (int i4 = 0; i4 < 2; ++i4) {
              const float4 z4 = philox_normal4(p.seed, p.offset, mel_noise_block(b + p.b_off, m0 + i4 * 4, t, p.M, p.T));
              zn[i4 * 4] = z4.x; zn[i4 * 4 + 1] = z4.y; zn[i4 * 4 + 2] = z4.z; zn[i4 * 4 + 3] = z4.w;
            }
          }
        }
        if (do_head) tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int m = m0 + i;
          float ev = 0.f;
          if (do_head) ev = __uint_as_float(e8[i]) + __ldg(p.bf + m);
          if ((p.flags & TC_WRITE_EPS) && row_valid) p.eps[(static_cast<size_t>(b) * p.M + m) * p.T + t] = ev;
          if (p.flags & TC_UPDATE) {
            xv[i] = ddpm_step(p.c, xv[i], ev, zn[i]);
            if (row_valid) p.x[xrow + static_cast<size_t>(m) * p.xs.c] = xv[i];
          }
          if ((p.flags & TC_PLMS) && row_valid) {
            const size_t ei = (static_cast<size_t>(b) * p.M + m) * p.T + t;
            xv[i] = plms_step(p.pl.c, xv[i], ev, p.pl.h1 ? p.pl.h1[ei] : 0.f, p.pl.h2 ? p.pl.h2[ei] : 0.f,
                              p.pl.h3 ? p.pl.h3[ei] : 0.f, p.pl.h1, p.pl.h2, p.pl.h3);
            if (p.pl.eps_store) p.pl.eps_store[ei] = ev;
            if (p.pl.x_out) p.pl.x_out[ei] = xv[i];
            else p.x[xrow + static_cast<size_t>(m) * p.xs.c] = xv[i];
          }
        }
        if (do_in) {
          // 8 bins = one 16-byte chunk of row r in k-block m0 >> 6
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float a0 = row_valid ? xv[2 * e] : 0.f, a1 = row_valid ? xv[2 * e + 1] : 0.f;
            const __half2 hh = __floats2half2_rn(a0, a1);
            hi[e] = h2_bits(hh);
            const float2 hf = __half22float2(hh);
            lo[e] = h2_bits(__floats2half2_rn(a0 - hf.x, a1 - hf.y));
          }
          const int kb = m0 >> 6, chunk = (m0 & 63) >> 3;
          const int off = r * 128 + ((chunk ^ (r & 7)) << 4);
          *reinterpret_cast<uint4*>(hk(0, kb) + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          if (P == 3) *reinterpret_cast<uint4*>(hk(1, kb) + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      if (do_in) {
        if (half == 1) {
          // zero the K padding (bins 80..127 = chunks 2..7 of k-block 1)
#pragma unroll
          for (int c = 2; c < 8; ++c) {
            const int off = r * 128 + ((c ^ (r & 7)) << 4);
            *reinterpret_cast<uint4*>(hk(0, 1) + off) = make_uint4(0, 0, 0, 0);
            if (P == 3) *reinterpret_cast<uint4*>(hk(1, 1) + off) = make_uint4(0, 0, 0, 0);
          }
        }
        tc_fence_before();
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(xfull);
      }
    }
    // ---- epi-I: x0 = relu(D3 + b_in) -> X ; y0 = split(x0 + d_0) -> Y (row-contiguous stores via the transpose staging) ----
    DSX_HTRACE(4);
    if (ok && do_in) ok = wait_warp(&tf[2], 0, 313);
    DSX_HTRACE(5);
    if (ok && do_in) {
      tc_fence_after();
      uint8_t* stg = staging + (warp - 4) * 32 * kStageRowBytes;
      const int lrow = lane >> 2, lcol = (lane & 3) * 2;
      const int urow0 = t0 + quad * 32;
      const float* d0 = p.d0 + static_cast<size_t>(b) * p.d_row_stride;
#pragma unroll 1
      for (int j = 0; j < 128; j += 32) {
        uint32_t o[32];
        tmem_ld_32x32(tmem_base + tlane + half * 128 + j, o);
        tmem_ld_wait();
#pragma unroll
        for (int sl = 0; sl < 4; ++sl) {
          const int col = half * 128 + j + sl * 8 + lcol;
          __syncwarp();
          *reinterpret_cast<uint4*>(stg + lane * kStageRowBytes) = make_uint4(o[sl * 8], o[sl * 8 + 1], o[sl * 8 + 2], o[sl * 8 + 3]);
          *reinterpret_cast<uint4*>(stg + lane * kStageRowBytes + 16) =
              make_uint4(o[sl * 8 + 4], o[sl * 8 + 5], o[sl * 8 + 6], o[sl * 8 + 7]);
          __syncwarp();
          const float2 bias = __ldg(reinterpret_cast<const float2*>(p.bin + col));
          const float2 dv = __ldg(reinterpret_cast<const float2*>(d0 + col));
#pragma unroll
          for (int itr = 0; itr < 4; ++itr) {
            const float2 d = *reinterpret_cast<const float2*>(stg + (itr * 8 + lrow) * kStageRowBytes + lcol * 4);
            const int tt = urow0 + itr * 8 + lrow;
            if (tt < p.T) {
              const size_t off = (static_cast<size_t>(b) * p.Tp + tt) * kC + col;
              const float x0 = fmaxf(d.x + bias.x, 0.f), x1 = fmaxf(d.y + bias.y, 0.f);
              *reinterpret_cast<float2*>(p.X + off) = make_float2(x0, x1);
              const float ya = x0 + dv.x, yb = x1 + dv.y;
              const __half2 hh = __floats2half2_rn(ya, yb);
              *reinterpret_cast<__half2*>(p.Y + off) = hh;
              if (P == 3) {
                const float2 hf = __half22float2(hh);
                *reinterpret_cast<__half2*>(p.Y + p.plane_elems + off) = __floats2half2_rn(ya - hf.x, yb - hf.y);
              }
            }
          }
        }
      }
    }
  }
  DSX_HTRACE(6);
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512);
  }
  if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) {
    p.trace[5 * 256 + 221 + (p.seq % 8) * 2] = static_cast<long long>(globaltimer_ns());
    p.trace[2 * 256 + 99] = clock64();
  }
}

// whead tile order (128 rows x 64 k each): skip_projection [plane][row half][kb 0..3] (16 tiles),
// output_projection [plane][kb 0..3] with rows >= M zero (8 tiles), input_projection [plane][row half][kb 0..1]
// with k >= M zero (8 tiles).
__global__ void k_pack_whead(const float* __restrict__ skip_w, const float* __restrict__ fin_w,
                             const float* __restrict__ in_w, __half* __restrict__ whead, int M) {
  const int tileidx = blockIdx.x, n = threadIdx.x;   // 128 threads = rows
  int plane;
  __half* dst = whead + (static_cast<size_t>(tileidx) * 128 + n) * 64;
  for (int kk = 0; kk < 64; ++kk) {
    float v = 0.f;
    if (tileidx < 16) {
      plane = tileidx / 8;
      const int nh = (tileidx / 4) & 1, kb = tileidx & 3;
      v = skip_w[static_cast<size_t>(nh * 128 + n) * kC + kb * 64 + kk];
    } else if (tileidx < 24) {
      const int u = tileidx - 16;
      plane = u / 4;
      const int kb = u & 3;
      v = (n < M) ? fin_w[static_cast<size_t>(n) * kC + kb * 64 + kk] : 0.f;
    } else {
      const int u = tileidx - 24;
      plane = u / 4;
      const int nh = (u / 2) & 1, kb = u & 1;
      const int k = kb * 64 + kk;
      v = (k < M) ? in_w[static_cast<size_t>(nh * 128 + n) * M + k] : 0.f;
    }
    const __half hi = __float2half_rn(v);
    dst[kk] = plane == 0 ? hi : __float2half_rn(v - __half2float(hi));
  }
}

// ------------------------------------------------------------------------------------------
// weight packing for the tcgen05 path
// tile order per layer (tiles of 256 rows x 64 k, fp16):
//   W1: idx = (plane*2 + chunk)*16 + kb      plane 0 = hi, 1 = lo; chunk h: rows n<128 -> gate channel
//       128h+n, n>=128 -> filter channel 128h+n-128 (= conv output row C + 128h + n - 128); k = kb*64+kk
//       over [tap0 | tap1 | tap2 | cond]
//   W2: idx = 64 + (plane*2 + half)*4 + kb   rows n -> output row half*256 + n
// ------------------------------------------------------------------------------------------
__global__ void k_pack_wtc(const float* __restrict__ w1f, const float* __restrict__ w2f,
                           const float* __restrict__ b1f, __half* __restrict__ wpack, float* __restrict__ b1p) {
  const int l = blockIdx.y, tileidx = blockIdx.x, n = threadIdx.x;
  const float* src;
  int plane;
  if (tileidx < 64) {
    plane = tileidx / 32;
    const int h = (tileidx / 16) & 1, kb = tileidx & 15;
    const int j = (n < 128) ? (128 * h + n) : (kC + 128 * h + (n - 128));
    src = w1f + (static_cast<size_t>(l) * 2 * kC + j) * (4 * kC) + kb * 64;
    if (plane == 0 && kb == 0) b1p[(static_cast<size_t>(l) * 2 + h) * 256 + n] = b1f[static_cast<size_t>(l) * 2 * kC + j];
  } else {
    const int u = tileidx - 64;
    plane = u / 8;
    const int q = (u / 4) & 1, kb = u & 3;
    src = w2f + (static_cast<size_t>(l) * 2 * kC + q * 256 + n) * kC + kb * 64;
  }
  __half* dst = wpack + (static_cast<size_t>(l) * kRowsPerLayer + static_cast<size_t>(tileidx) * 256 + n) * 64;
  for (int kk = 0; kk < 64; ++kk) {
    const float v = src[kk];
    const __half hi = __float2half_rn(v);
    dst[kk] = plane == 0 ? hi : __float2half_rn(v - __half2float(hi));
  }
}

bool tc_supported(const dsx_handle* h) { return h->m.C == kC && h->m.H == kC && h->m.M == 80; }

int tc_pack_model(dsx_handle* h, cudaStream_t s) {
  DSX_CHECK(tc_supported(h), DSX_E_INVALID, "tcgen05 path needs residual_channels == hidden_size == 256 (got %d, %d)",
            h->m.C, h->m.H);
  __half* wpack;
  float* b1p;
  const size_t rows = static_cast<size_t>(h->m.L) * kRowsPerLayer;
  DSX_TRY(dev_alloc(h, reinterpret_cast<void**>(&wpack), rows * 64 * sizeof(__half), true));
  DSX_TRY(dev_alloc(h, reinterpret_cast<void**>(&b1p), static_cast<size_t>(h->m.L) * 512 * sizeof(float), true));
  dim3 grid(kRowsPerLayer / 256, h->m.L);
  k_pack_wtc<<<grid, 256, 0, s>>>(h->m.w1f, h->m.w2f, h->m.b1f, wpack, b1p);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  h->m.wpack = wpack;
  h->m.b1p = b1p;
  __half* whead;
  DSX_TRY(dev_alloc(h, reinterpret_cast<void**>(&whead), static_cast<size_t>(32) * 128 * 64 * sizeof(__half), true));
  k_pack_whead<<<32, 128, 0, s>>>(h->m.skip_w, h->m.fin_w, h->m.in_w, whead, h->m.M);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  h->m.whead = whead;
  DSX_TRY(tc_stack_pack(h, s));
  return DSX_OK;
}

// ------------------------------------------------------------------------------------------
// tensor maps
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                        CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                        CUtensorMapFloatOOBfill);
static PFN_tmapEncodeTiled get_encode() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  return fn;
}

int make_map_2d(CUtensorMap* m, const void* base, uint64_t rows, uint32_t box_rows) {
  PFN_tmapEncodeTiled enc = get_encode();
  DSX_CHECK(enc, DSX_E_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[2] = {64, rows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DSX_CHECK(r == CUDA_SUCCESS, DSX_E_CUDA, "cuTensorMapEncodeTiled(2D) failed: %d", static_cast<int>(r));
  return DSX_OK;
}
// [B][T (stride Tp)][ch] fp16 (or fp32), box = 128 bytes of channels x box_frames frames x 1
static int make_map_act(CUtensorMap* m, const void* base, int ch, int T, int Tp, int B, int box_frames = kTile, bool f32 = false) {
  PFN_tmapEncodeTiled enc = get_encode();
  DSX_CHECK(enc, DSX_E_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  const cuuint64_t es_bytes = f32 ? 4 : 2;
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(ch), static_cast<cuuint64_t>(T), static_cast<cuuint64_t>(B)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(ch) * es_bytes, static_cast<cuuint64_t>(Tp) * ch * es_bytes};
  cuuint32_t box[3] = {static_cast<cuuint32_t>(128 / es_bytes), static_cast<cuuint32_t>(box_frames), 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = enc(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides,
                   box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DSX_CHECK(r == CUDA_SUCCESS, DSX_E_CUDA, "cuTensorMapEncodeTiled(3D) failed: %d", static_cast<int>(r));
  return DSX_OK;
}

int tc_prepare_maps(dsx_handle* h, const Geom& g) {
  const size_t plane = g.frames_padded() * kC;
  if (h->tm_geom.B == g.B && h->tm_geom.T == g.T && h->tm_epoch == h->ws_epoch) return DSX_OK;
  DSX_TRY(make_map_2d(&h->tm_w, h->m.wpack, static_cast<uint64_t>(h->m.L) * kRowsPerLayer, 128));
  for (int buf = 0; buf < 2; ++buf) {
    for (int pl = 0; pl < 2; ++pl)
      DSX_TRY(make_map_act(&h->tm_y[buf][pl], h->ws.Y + (static_cast<size_t>(buf) * 2 + pl) * plane, kC, g.T, g.Tp, g.B));
    DSX_TRY(make_map_act(&h->tm_yh[buf], h->ws.Y + static_cast<size_t>(buf) * 2 * plane, kC, g.T, g.Tp, g.B, kTile + 16));
    DSX_TRY(make_map_act(&h->tm_ye[buf], h->ws.Y + static_cast<size_t>(buf) * 2 * plane, kC, g.T, g.Tp, g.B, 8));
  }
  for (int pl = 0; pl < 2; ++pl) {
    DSX_TRY(make_map_act(&h->tm_cond[pl], h->ws.CONDH + static_cast<size_t>(pl) * plane, kC, g.T, g.Tp, g.B));
    DSX_TRY(make_map_act(&h->tm_s16[pl], h->ws.S16 + static_cast<size_t>(pl) * plane, kC, g.T, g.Tp, g.B));
  }
  DSX_TRY(make_map_2d(&h->tm_whead, h->m.whead, 32 * 128, 128));
  DSX_TRY(make_map_act(&h->tm_z, h->ws.Z, kC, g.T, g.Tp, h->m.L * g.B));
  for (int ri = 0; ri < 2; ++ri) {        // stack kernel: boxes of 128 / 64 frames per CTA
    const int rows = ri == 0 ? 128 : 64;
    DSX_TRY(make_map_act(&h->tm_y0s[ri], h->ws.Y, kC, g.T, g.Tp, g.B, rows + 16));
    DSX_TRY(make_map_act(&h->tm_zs[ri], h->ws.Z, kC, g.T, g.Tp, h->m.L * g.B, rows));
    DSX_TRY(make_map_act(&h->tm_y0st[ri], h->ws.Y, kC, g.T, g.Tp, g.B, rows));
    DSX_TRY(make_map_act(&h->tm_xst[ri], h->ws.X, kC, g.T, g.Tp, g.B, rows, true));
    for (int pl = 0; pl < 2; ++pl)
      DSX_TRY(make_map_act(&h->tm_s16s[ri][pl], h->ws.S16 + static_cast<size_t>(pl) * plane, kC, g.T, g.Tp, g.B, rows));
  }
  h->tm_geom = g;
  h->tm_epoch = h->ws_epoch;
  return DSX_OK;
}

template <int P>
static int launch_tc_layer_t(dsx_handle* h, const TcLayerParams& prm, int grid, int csize, cudaStream_t s) {
  using Cfg = TcCfg<P>;
  bool& attr_done = h->attr_layer[P - 1];      // function attributes are per device -> per handle
  if (!attr_done) {
    DSX_CUDA(cudaFuncSetAttribute(k_tc_layer<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_done = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = csize;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DSX_CUDA(cudaLaunchKernelEx(&cfg, k_tc_layer<P>, prm));
  h->launches++;
  return DSX_OK;
}

// Can a cluster of `csize` CTAs of the layer kernel be scheduled on this device?  (cached per size)
template <int P>
static int cluster_occupancy(dsx_handle* h, int csize) {
  int* cache = h->occ_cache[P - 1];   // per handle (= per device): 0 unknown, >0 max co-resident clusters, -1 none
  if (csize > 16) return -1;
  if (cache[csize] == 0) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(csize));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = TcCfg<P>::SMEM_BYTES;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = csize;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    cudaFuncSetAttribute(k_tc_layer<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<P>::SMEM_BYTES);
    cudaError_t e = cudaOccupancyMaxActiveClusters(&n, k_tc_layer<P>, &cfg);
    if (e != cudaSuccess) cudaGetLastError();
    cache[csize] = (e == cudaSuccess && n >= 1) ? n : -1;
  }
  return cache[csize];
}

int ensure_flags(dsx_handle* h, int n) {
  if (h->flags_cap >= n) return DSX_OK;
  if (h->flags_dev) cudaFree(h->flags_dev);
  h->flags_dev = nullptr;
  DSX_CUDA(cudaMalloc(&h->flags_dev, static_cast<size_t>(n) * sizeof(unsigned int)));
  DSX_CUDA(cudaMemset(h->flags_dev, 0, static_cast<size_t>(n) * sizeof(unsigned int)));
  h->flags_cap = n;
  h->flag_count = 0;
  return DSX_OK;
}

// Layers [l0, l1) of one evaluation: a single launch when every CTA can be co-resident (stack mode), otherwise one
// launch per layer.  Always clusters of two CTAs (cta_group::2 pairs).
int launch_tc_layers(dsx_handle* h, int l0, int l1, const Geom& g, int row0, int row_per_b, cudaStream_t s) {
  const ModelDev& m = h->m;
  TcLayerParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.tm_w = h->tm_w;
  for (int bf = 0; bf < 2; ++bf)
    for (int pl = 0; pl < 2; ++pl) prm.tm_y[bf][pl] = h->tm_y[bf][pl];
  prm.tm_yh[0] = h->tm_yh[0];
  prm.tm_yh[1] = h->tm_yh[1];
  prm.X = h->ws.X;
  prm.SKIP = h->ws.SKIP;
  prm.Y = h->ws.Y;
  prm.plane_elems = g.frames_padded() * kC;
  prm.CP = h->ws.CP;
  prm.cp_prefetch = h->cp_prefetch;
  prm.b2 = m.b2f;
  prm.dtab = h->ws.DTAB + static_cast<size_t>(row0) * m.L * kC;
  prm.d_row_stride = row_per_b * m.L * kC;
  prm.T = g.T; prm.Tp = g.Tp; prm.tiles_per_utt = g.tiles_per_utt; prm.tiles = g.tiles; prm.B = g.B;
  prm.L = m.L; prm.cycle = m.cycle;
  prm.s16 = h->ws.S16;
  prm.inv_sqrt_l = 1.0f / sqrtf(static_cast<float>(m.L));
  prm.status = h->status_dev;
  prm.budget_ns = 4000000000ull;
  prm.trace = h->trace_dev;
  prm.seq = h->trace_seq++;
  const int P = (h->precision == DSX_PREC_FP16S) ? 2 : h->precision;   // DSX_PREC_FP16 = 1, FP16X2 = 2, FP16X3 = 3 == MMA passes
                                                                        // (FP16S without the stack kernel: the fp16x2 scheme)
  auto launch = [&](int grid) -> int {
    return P == 1 ? launch_tc_layer_t<1>(h, prm, grid, kG, s)
                  : (P == 2 ? launch_tc_layer_t<2>(h, prm, grid, kG, s) : launch_tc_layer_t<3>(h, prm, grid, kG, s));
  };
  const int occ = P == 1 ? cluster_occupancy<1>(h, kG) : (P == 2 ? cluster_occupancy<2>(h, kG) : cluster_occupancy<3>(h, kG));
  h->cluster_occ = occ;
  // Stack mode needs every CTA of a launch co-resident (tiles wait on their neighbours' publish counters): the batch is
  // cut into groups of whole utterances that fit the machine, one persistent launch per group and evaluation.
  const int cap_tiles = occ > 0 ? occ * kG : 0;
  const int utt_per_group = (g.tiles_per_utt > 0) ? cap_tiles / g.tiles_per_utt : 0;
  const bool stack = h->stack_mode && (l1 - l0 > 1) && utt_per_group >= 1;
  if (stack) {
    DSX_TRY(ensure_flags(h, g.tiles + 2));
    if (h->flags_geom_b != g.B || h->flags_geom_t != g.T || h->flags_kind != 1) {   // counters are in lockstep only within one geometry
      DSX_CUDA(cudaMemsetAsync(h->flags_dev, 0, static_cast<size_t>(h->flags_cap) * sizeof(unsigned int), s));
      h->flag_count = 0;
      h->flags_geom_b = g.B;
      h->flags_geom_t = g.T;
      h->flags_kind = 1;
    }
    prm.l0 = l0; prm.l1 = l1;
    prm.flags = h->flags_dev;
    prm.flag_base = h->flag_count;
    for (int b0 = 0; b0 < g.B; b0 += utt_per_group) {
      const int nb = std::min(utt_per_group, g.B - b0);
      prm.tile0 = b0 * g.tiles_per_utt;
      prm.tile_end = (b0 + nb) * g.tiles_per_utt;
      const int grid = (prm.tile_end - prm.tile0 + kG - 1) / kG * kG;
      DSX_TRY(launch(grid));
    }
    h->flag_count += static_cast<unsigned int>(kEpiWarps * (l1 - l0 - 1));
    return DSX_OK;
  }
  const int grid = (g.tiles + kG - 1) / kG * kG;
  prm.tile0 = 0;
  prm.tile_end = g.tiles;
  for (int l = l0; l < l1; ++l) {
    prm.l0 = l; prm.l1 = l + 1;
    DSX_TRY(launch(grid));
  }
  return DSX_OK;
}

// CP for the conditioner currently packed in ws.CONDH (called once per API call, after launch_pack_cond).
int launch_tc_condproj(dsx_handle* h, const Geom& g, cudaStream_t s) {
  if (!h->attr_cond) {
    DSX_CUDA(cudaFuncSetAttribute(k_tc_condproj, cudaFuncAttributeMaxDynamicSharedMemorySize, kCondSmem));
    h->attr_cond = true;
  }
  TcCondParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.tm_w = h->tm_w;
  prm.tm_cond[0] = h->tm_cond[0];
  prm.tm_cond[1] = h->tm_cond[1];
  prm.CP = h->ws.CP;
  prm.b1p = h->m.b1p;
  prm.T = g.T; prm.Tp = g.Tp; prm.tiles_per_utt = g.tiles_per_utt; prm.tiles = g.tiles; prm.B = g.B;
  prm.L = h->m.L;
  prm.status = h->status_dev;
  prm.budget_ns = 2000000000ull;
  // few tiles: split the 2L (layer, chunk) jobs of a tile over several CTAs so the whole machine works
  const int split = std::max(1, std::min(2 * h->m.L, h->sm_count / std::max(g.tiles, 1)));
  dim3 grid(static_cast<unsigned>(g.tiles), static_cast<unsigned>(split));
  k_tc_condproj<<<grid, kThreads, kCondSmem, s>>>(prm);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

template <int P>
static int launch_tc_head_t(dsx_handle* h, const TcHeadParams& prm, int tiles, cudaStream_t s) {
  using Cfg = HeadCfg<P>;
  bool& attr_done = h->attr_head[P == 1 ? 0 : 1];
  if (!attr_done) {
    DSX_CUDA(cudaFuncSetAttribute(k_tc_head<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_done = true;
  }
  k_tc_head<P><<<tiles, kThreads, Cfg::SMEM_BYTES, s>>>(prm);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

int launch_tc_head(dsx_handle* h, const Geom& g, const HeadArgs& ha, cudaStream_t s) {
  const ModelDev& m = h->m;
  TcHeadParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.tm_s16[0] = h->tm_s16[0];
  prm.tm_s16[1] = h->tm_s16[1];
  prm.tm_wh = h->tm_whead;
  prm.x = ha.x;
  prm.xs = ha.xs;
  prm.eps = ha.eps;
  prm.noise = ha.noise;
  prm.seed = ha.seed;
  prm.b_off = h->batch_offset;
  prm.offset = ha.offset;
  prm.c = ha.c;
  if (ha.plms) prm.pl = *ha.plms;
  prm.X = h->ws.X;
  prm.Y = h->ws.Y;                       // layer 0 reads buffer 0
  prm.plane_elems = g.frames_padded() * kC;
  prm.bs = m.skip_b;
  prm.bf = m.fin_b;
  prm.bin = m.in_b;
  prm.d0 = h->ws.DTAB + static_cast<size_t>(ha.next_row0) * m.L * kC;
  prm.d_row_stride = ha.row_per_b * m.L * kC;
  prm.T = g.T; prm.Tp = g.Tp; prm.tiles_per_utt = g.tiles_per_utt; prm.tiles = g.tiles; prm.B = g.B; prm.M = m.M;
  prm.flags = ha.flags;
  prm.status = h->status_dev;
  prm.budget_ns = 2000000000ull;
  prm.trace = h->trace_dev;
  prm.seq = h->trace_seq++;
  return (h->precision == DSX_PREC_FP16) ? launch_tc_head_t<1>(h, prm, g.tiles, s) : launch_tc_head_t<3>(h, prm, g.tiles, s);
}

}  // namespace dsx
