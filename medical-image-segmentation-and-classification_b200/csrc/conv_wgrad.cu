// b200seg — convolution weight gradient on tcgen05 (the dW half of aten::convolution_backward).
//
//   dW[co][tap][ci] = sum over pixels p   dY[p][co] * X[p (+) tap][ci]
//
// GEMM view: M = 128 output channels, N = up to 4 column blocks of 64 (3x3: the three taps of one filter row for one
// 64-channel block of X; 1x1: up to four 64-channel blocks), K = pixels.  Both operands are pixel-major in NHWC
// memory, i.e. MN-major for the MMA: a TMA box of (64 ch, Wb, Hb, Nb) lands as 64 rows (pixels) of 128 B (channels)
// with the 128B swizzle, which is exactly the canonical MN-major SW128 atom stack (8 K-rows per 1024 B, 64-element
// MN blocks LBO apart).  X boxes are shifted by the tap offset; TMA zero fill supplies the padding halo.
// The dY tile is loaded once per K chunk and reused by every column block (3x3: 2 X blocks x 3 taps = N 384, issued as
// two N=192 MMAs into adjacent TMEM columns); the kernel is L2->SM bandwidth bound, so bytes per FLOP is what counts.
// Cout == 64 ("row pair" mode): instead of leaving half of the 128 MMA rows idle, rows 64..127 hold dY of the NEXT
// image row, so against the same X row they produce the gradient of the filter row above.  3x3: with X rows h and
// h+1 as two column groups one CTA yields all three filter rows from two MMAs per K step (one quarter is redundant);
// 2x2 (folded UpConv phases): one X row gives both filter rows, nothing is redundant.
// X-halo mode (3x3, unit stride — the default): one (Wb+2)-pixel-wide box per X block replaces the three tap-shifted
// boxes; tap s is an MMA whose B descriptor starts s pixels (s * 128 B) into the box — the 128B swizzle is a function
// of the absolute shared-memory address, so the shifted view reads the right bytes.  The kernel is bound by the bytes
// it pulls through the L2 -> SM fabric; this halves them (64 -> 33 KB per chunk): 128->128 @128^2 0.378 -> 0.226 ms
// (1367 TFLOP/s), 64->64 @256^2 0.720 -> 0.308 ms.
// CTA pairs (3x3 halo mode, Cout a multiple of 256, an even number of X blocks): the kernel is bound by shared-memory
// bandwidth — an M = 128 x N = 128 MMA reads 4 KB of dY and 4 KB of X per 64 issue clocks, the whole operand port, while
// TMA writes the next stage into the same memory.  tcgen05.mma.cta_group::2 runs M = 256 over two SMs: each CTA holds its
// own Cout tile of dY and HALF of the X operand (one of the two halo boxes), so a CTA reads 4 + 2 KB per MMA and
// receives 24 instead of 32.5 KB per stage.
// Split-K over pixel chunks across CTAs; partial tiles go to a workspace and a second kernel reduces them in a fixed
// order (deterministic), optionally accumulating into dW (shared weights of Recurrent_block, R2U_Net.py:15-20).
#include <stdlib.h>
#include <mutex>

#include "common.cuh"

namespace b2 {

int conv_tile_geometry(int n, int h, int w, int tile_pix, int* Wb, int* Hb, int* Nb, int* tw, int* th, int* tn);
int encode_act_tmap(CUtensorMap* tm, const void* base, int c, int ld, int n, int h, int w, int Wb, int Hb, int Nb);
int encode_act_tmap_ex(CUtensorMap* tm, const void* base, int c, int n, int h, int w, long long s_w, long long s_h,
                       long long s_n, int Wb, int Hb, int Nb, int es);

static constexpr int kChunkPix = 64;            // K per pipeline stage
static constexpr int kBoxBytes = kChunkPix * 128;  // 8 KB: 64 pixels x 64 channels bf16
static constexpr int kWgThreads = 192;
static constexpr int kXhBox = 9 * 1024;         // X-halo box slot: 66 pixels x 128 B = 8448 B, padded to 1 KB

struct WgradParams {
  int Wb, Hb, Nb, tw, th;
  int num_chunks, chunks_per_split;
  int taps;          // ksize^2
  int ksize, pad_h, pad_w, xstride;   // X-operand tap geometry: offsets (r - pad_h, s - pad_w), sampling stride
  int cpb;           // 64-channel X blocks per CTA
  int ncolb;         // column blocks per CTA = ksize (taps of one filter row) x cpb
  int cb0, cb1;      // 64-channel blocks per X source
  int cout, ctot;    // ctot = c0 + c1 (row length of dW)
  int a_boxes;       // 1 if cout <= 64 else 2
  int stages;
  int b_stage_bytes; // smem bytes reserved per stage for the X boxes
  int gy;            // CTAs per (split, channel group): filter rows handled by separate CTAs (1 in row-pair mode)
  int rowpair;       // Cout == 64: M rows 0..63 = dY of image row h, rows 64..127 = dY of row h+1 (see kernel);
                     // value = number of X-row column groups (3x3: 2, 2x2: 1), 0 = off
  int rp_dir;        // row-pair mode: rows 64..127 hold dY of image row h + rp_dir.  +1 when the filter has a row above
                     // the centre (pad_h >= 1); -1 for 2x2 taps with pad_h == 0, so that the one product the pairing
                     // cannot form always involves an out-of-image (zero) X row
  int xh;            // X-halo mode (3x3, chunk = 64 pixels of one image row): ONE (64+2)-pixel box per X block / row
                     // instead of three tap-shifted ones; tap s is an MMA whose B descriptor starts s*128 B into
                     // the box (the 128B swizzle is a function of the absolute smem address).  Halves the bytes a
                     // CTA pulls through the L2 -> SM fabric.  nbox = boxes per stage (2), kXhBox bytes apart.
  int nbox;
  int pair;          // CTA pair (cta_group::2): blockIdx.x = rank + 2 * (rg + gy * (co pair + co pairs * channel group))
  int fold;          // merged folded-UpConv weight gradient (b2_wgrad_args::fold): dY is the FINE tensor, phase (a, b) its
                     // (2h+a, 2w+b) sub-lattice; a CTA owns (a, filter row ty) = blockIdx % 4, loads the b = 0 and b = 1
                     // sub-lattice tiles and ONE halo row of X (coarse row h + a + ty - 1), and tap (b, tx) is the MMA
                     // whose B descriptor starts (b + tx) pixels into the halo box.  1: cout >= 128 — A = 128 channels
                     // per b, accumulators [b][tx][block][64] (512 TMEM columns).  2: cout == 64 — the two b tiles are
                     // the two halves of ONE M = 128 operand, three shift MMAs (rows 0..63 keep shifts 0, 1 = tx 0, 1;
                     // rows 64..127 keep shifts 1, 2), accumulators [shift][block][64]
  int a_bytes;       // smem bytes reserved per stage for the dY tiles (16 KB; 32 KB when fold == 1)
  int debug_skip;    // timing experiments only (B200SEG_DEBUG_SKIP): 1 = no TMA loads, 2 = no MMAs
  float* ws;         // [splits][cout][taps][ctot]
};

// kPair is a separate instantiation: a kernel that contains cta_group::2 instructions can only be launched as 2-CTA
// clusters, so the single-CTA kernel must not contain them.
template <bool kPair>
__global__ void __launch_bounds__(kWgThreads, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap tmDY, const __grid_constant__ CUtensorMap tmX0,
                  const __grid_constant__ CUtensorMap tmX1, const WgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int stage_bytes = p.a_bytes + p.b_stage_bytes;
  uint8_t* tail = smem + p.stages * stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + 8;
  uint64_t* tmem_full_bar = empty_bar + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // CTAs that read the same pixels (same split; different filter row / channel group) have adjacent block indices,
  // so they run in the same wave and the dY / X chunks they share are fetched from DRAM once
  const int split = blockIdx.y;
  const uint32_t crank = kPair ? cluster_ctarank() : 0u;     // pair: rank 0 issues the MMAs
  const int bx = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int rg = bx % p.gy;                           // filter row (3x3) or 0
  const int zz = bx / p.gy;
  const int co_tiles = (p.cout + 127) / 128;
  const int co_groups = kPair ? co_tiles / 2 : co_tiles;
  const int co_tile = kPair ? 2 * (zz % co_groups) + (int)crank : zz % co_groups;
  const int cgrp = zz / co_groups;                    // channel-block group
  const int cib_base = cgrp * p.cpb;
  const int cbt = p.cb0 + p.cb1;

  const int chunk_begin = split * p.chunks_per_split;
  int chunk_end = chunk_begin + p.chunks_per_split;
  if (chunk_end > p.num_chunks) chunk_end = p.num_chunks;
  const int nchunks = chunk_end - chunk_begin;        // may be <= 0 for trailing splits

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
    tma_prefetch_desc(&tmDY);
    tma_prefetch_desc(&tmX0);
  }
  const uint32_t tmem_cols = (p.fold == 1 ? 4 * p.cpb : p.fold == 2 ? 3 * p.cpb : p.ncolb) * 64 > 256 ? 512u : 256u;
  if (warp == 1) {
    if constexpr (kPair) {
      tmem_alloc_pair(tmem_slot, tmem_cols);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_slot, tmem_cols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) cluster_sync_all();       // the peer's barriers are initialised before anything can signal them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // number of live column blocks for this CTA (1x1 groups may run past the last channel block)
  int live_cb = p.cpb;
  if (cib_base + live_cb > cbt) live_cb = cbt - cib_base;
  const int rowpair = kPair ? 0 : p.rowpair;                    // pair mode never runs row pairs
  const int grp_cols = live_cb * p.ksize;                       // columns per X-row group (row-pair mode)
  const int ncol_live = rowpair ? rowpair * grp_cols : grp_cols;
  const int xh_live = rowpair ? rowpair : live_cb;              // X-halo mode: boxes this CTA fills per stage

  if (warp == 0) {
    // TMA producer: warp-uniform loop, one elected lane issues; chunk coordinates advance incrementally
    if (nchunks > 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t tx = p.fold ? (uint32_t)(2 * p.a_boxes * kBoxBytes + xh_live * (p.Wb + 2) * p.Hb * 128)
                          : p.xh ? (uint32_t)(p.a_boxes * kBoxBytes + xh_live * (p.Wb + 2) * p.Hb * 128)
                               : (uint32_t)((p.a_boxes + ncol_live) * kBoxBytes);
      int tw_i = chunk_begin % p.tw;
      int th_i = (chunk_begin / p.tw) % p.th;
      int tn_i = chunk_begin / (p.tw * p.th);
      for (int ck = chunk_begin; ck < chunk_end; ++ck) {
        const int w0 = tw_i * p.Wb, h0 = th_i * p.Hb, n0 = tn_i * p.Nb;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elect_one()) {
          uint8_t* sa = smem + stage * stage_bytes;
          uint8_t* sb = sa + p.a_bytes;
          if constexpr (kPair) {
            // both CTAs load into their own shared memory — their Cout tile of dY and ONE of the two X halo boxes —
            // and the bytes are counted on the LEADER's barrier, which only the leader arms
            const uint32_t lbar = mapa_shared(smem_u32(&full_bar[stage]), 0);
            if (crank == 0)
              mbar_arrive_expect_tx(&full_bar[stage], 2u * (uint32_t)(p.a_bytes + (p.Wb + 2) * p.Hb * 128));
            const int cib = cib_base + (int)crank;
            int xrow = h0 + rg - p.pad_h, xcol = w0 - p.pad_w;
            if (p.fold) {          // merged folded UpConv (fold == 1): both column-phase tiles of dY, X row h + a + ty - 1
              const int fa = rg >> 1, fty = rg & 1;
              for (int b = 0; b < 2; ++b)
                tma_load_5d_pair(sa + b * 2 * kBoxBytes, &tmDY, lbar, 0, 2 * w0 + b, 2 * h0 + fa, n0, co_tile * 2);
              xrow = h0 + fa + fty - 1;
              xcol = w0 - 1;
            } else {
              tma_load_5d_pair(sa, &tmDY, lbar, 0, w0, h0, n0, co_tile * 2);
            }
            if (cib < p.cb0)
              tma_load_4d_pair(sb, &tmX0, lbar, cib * 64, xcol, xrow, n0);
            else
              tma_load_4d_pair(sb, &tmX1, lbar, (cib - p.cb0) * 64, xcol, xrow, n0);
          } else
          if (p.debug_skip & 1) {
            mbar_arrive(&full_bar[stage]);
          } else if (p.fold) {
            mbar_arrive_expect_tx(&full_bar[stage], tx);
            const int fa = rg >> 1, fty = rg & 1;
            // dY: the (a, b = 0) and (a, b = 1) sub-lattices of the fine tensor (traversal stride 2 in w and h)
            for (int b = 0; b < 2; ++b)
              tma_load_5d(sa + b * p.a_boxes * kBoxBytes, &tmDY, &full_bar[stage], 0, 2 * w0 + b, 2 * h0 + fa, n0,
                          co_tile * 2);
            // X: one halo row per 64-channel block, coarse row h + a + ty - 1, pixels w0 - 1 .. w0 + Wb
            for (int b = 0; b < xh_live; ++b) {
              const int cib = cib_base + b;
              if (cib < p.cb0)
                tma_load_4d(sb + b * kXhBox, &tmX0, &full_bar[stage], cib * 64, w0 - 1, h0 + fa + fty - 1, n0);
              else
                tma_load_4d(sb + b * kXhBox, &tmX1, &full_bar[stage], (cib - p.cb0) * 64, w0 - 1, h0 + fa + fty - 1,
                            n0);
            }
          } else {
          mbar_arrive_expect_tx(&full_bar[stage], tx);
          // dY: both 64-channel blocks of the 128-row M tile in one 5-D box (.., channel block)
          if (rowpair) {       // dY rows h0 and h0 + 1 (zero fill below the image)
            tma_load_4d(sa, &tmDY, &full_bar[stage], 0, w0, h0, n0);
            tma_load_4d(sa + kBoxBytes, &tmDY, &full_bar[stage], 0, w0, h0 + p.rp_dir, n0);
          } else {
            tma_load_5d(sa, &tmDY, &full_bar[stage], 0, w0, h0, n0, co_tile * 2);
          }
          if (p.xh) {
            // one box per (X block | X row): pixels w0-1 .. w0+Wb of the chunk's Hb rows, shifted by the filter row
            for (int b = 0; b < xh_live; ++b) {
              const int cib = rowpair ? cib_base : cib_base + b;
              const int xh_row = rowpair ? h0 + (p.rp_dir > 0 ? b + 1 : 0) - p.pad_h : h0 + rg - p.pad_h;
              if (cib < p.cb0)
                tma_load_4d(sb + b * kXhBox, &tmX0, &full_bar[stage], cib * 64, w0 - p.pad_w, xh_row, n0);
              else
                tma_load_4d(sb + b * kXhBox, &tmX1, &full_bar[stage], (cib - p.cb0) * 64, w0 - p.pad_w, xh_row, n0);
            }
          } else
          for (int j = 0; j < ncol_live; ++j) {
            // row-pair mode: group jg reads X row h0 + (jg + 1) - pad_h (filter row jg + 1 for the top half)
            const int jg = rowpair ? j / grp_cols : 0;
            const int cib = cib_base + (j - jg * grp_cols) / p.ksize;
            const int xw = p.xstride * w0 + (j % p.ksize) - p.pad_w;
            const int xh = rowpair ? h0 + (p.rp_dir > 0 ? jg + 1 : 0) - p.pad_h : p.xstride * h0 + rg - p.pad_h;
            if (cib < p.cb0)
              tma_load_4d(sb + j * kBoxBytes, &tmX0, &full_bar[stage], cib * 64, xw, xh, n0);
            else
              tma_load_4d(sb + j * kBoxBytes, &tmX1, &full_bar[stage], (cib - p.cb0) * 64, xw, xh, n0);
          }
          }
        }
        __syncwarp();
        if (++tw_i == p.tw) {
          tw_i = 0;
          if (++th_i == p.th) {
            th_i = 0;
            ++tn_i;
          }
        }
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1 && !(kPair && crank != 0)) {
    if (nchunks > 0) {
      // up to 6 column blocks (3x3: two 64-channel X blocks x three taps): N <= 256 per instruction, so the columns
      // are issued as two MMAs that share the dY tile (A) and write adjacent TMEM column ranges
      const int ncol0 = ncol_live > 4 ? 3 : ncol_live;
      const int ncol1 = ncol_live - ncol0;
      const uint32_t idesc = umma_idesc_bf16(128, ncol0 * 64, 1, 1);
      const uint32_t idesc1 = ncol1 > 0 ? umma_idesc_bf16(128, ncol1 * 64, 1, 1) : 0u;
      const uint64_t desc0 = umma_desc_sw128(0, kBoxBytes, 1024);   // MN-major SW128 descriptor, start address 0
      const uint64_t desc_hi = desc0 & 0xFFFFFFFF00000000ull;
      const uint32_t desc_lo0 = (uint32_t)desc0;
      const uint64_t descx0 = umma_desc_sw128(0, kXhBox, 1024);     // X-halo boxes: MN blocks kXhBox apart
      const uint64_t descx_hi = descx0 & 0xFFFFFFFF00000000ull;
      const uint32_t descx_lo0 = (uint32_t)descx0;
      const uint32_t idescx = umma_idesc_bf16(128, xh_live * 64, 1, 1);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < nchunks; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_addr = smem_u32(smem + stage * stage_bytes);
          const uint32_t b_addr = a_addr + (uint32_t)p.a_bytes;
          // 16 pixels (K) = two 8-row groups, 1024 B apart (SBO); 64-channel MN blocks 8 KB apart (LBO).  A K step
          // of 16 pixels moves the start address by 2048 B = +128 in the (bytes >> 4) address field of the low word.
          uint32_t a_lo = desc_lo0 + (a_addr >> 4);
          uint32_t b_lo = desc_lo0 + (b_addr >> 4);
          const uint32_t b1_off = (uint32_t)(ncol0 * kBoxBytes) >> 4;
          const int nk = (p.debug_skip & 2) ? 0 : kChunkPix / 16;
          if constexpr (kPair) {
            // M = 256 over the pair: three taps x four K steps, B = one halo box per CTA (N = 128 in all)
            const uint32_t bx_lo = descx_lo0 + (b_addr >> 4);
            const uint32_t idescp = umma_idesc_bf16(256, 128, 1, 1);
#pragma unroll
            for (int k = 0; k < kChunkPix / 16; ++k) {
              const uint32_t koff = (uint32_t)(((16 * k) / p.Wb) * (p.Wb + 2) + (16 * k) % p.Wb) * 8u;
              if (p.fold) {        // taps (b, tx): A = the b sub-lattice tile, B shifted by b + tx pixels
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                  const uint64_t da = desc_hi | (uint64_t)(a_lo + (uint32_t)b * ((2u * kBoxBytes) >> 4) + 128u * k);
#pragma unroll
                  for (int tx = 0; tx < 2; ++tx)
                    umma_bf16_pair(tmem_base + (uint32_t)(b * 2 + tx) * 128u, da,
                                   descx_hi | (uint64_t)(bx_lo + 8u * (uint32_t)(b + tx) + koff), idescp,
                                   (it | k) != 0 ? 1u : 0u);
                }
              } else {
                const uint64_t da = desc_hi | (uint64_t)(a_lo + 128u * k);
#pragma unroll
                for (int tp = 0; tp < 3; ++tp)
                  umma_bf16_pair(tmem_base + tp * 128u, da, descx_hi | (uint64_t)(bx_lo + 8u * tp + koff), idescp,
                                 (it | k) != 0 ? 1u : 0u);
              }
            }
          } else
          if (p.fold == 1) {
            // taps (b, tx): A = the b sub-lattice tile, B = the halo boxes shifted by b + tx pixels
            const uint32_t bx_lo = descx_lo0 + (b_addr >> 4);
            const uint32_t ncx = (uint32_t)(xh_live * 64);
#pragma unroll
            for (int k = 0; k < kChunkPix / 16; ++k) {
              if (k < nk) {
                const uint32_t koff = (uint32_t)(((16 * k) / p.Wb) * (p.Wb + 2) + (16 * k) % p.Wb) * 8u;
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                  const uint64_t da = desc_hi | (uint64_t)(a_lo + (uint32_t)b * ((2u * kBoxBytes) >> 4) + 128u * k);
#pragma unroll
                  for (int tx = 0; tx < 2; ++tx)
                    umma_bf16(tmem_base + (uint32_t)(b * 2 + tx) * ncx, da,
                              descx_hi | (uint64_t)(bx_lo + 8u * (uint32_t)(b + tx) + koff), idescx,
                              (it | k) != 0 ? 1u : 0u);
                }
              }
            }
          } else if (p.xh) {
            // three taps = three MMAs on the same halo boxes, B start shifted by one pixel (128 B = +8) per tap;
            // N = all boxes of the stage (kXhBox apart), accumulator columns [tap][box][64]
            const uint32_t bx_lo = descx_lo0 + (b_addr >> 4);
            const uint32_t ncx = (uint32_t)(xh_live * 64);
#pragma unroll
            for (int k = 0; k < kChunkPix / 16; ++k) {
              if (k < nk) {
                const uint64_t da = desc_hi | (uint64_t)(a_lo + 128u * k);
#pragma unroll
                // the 16 pixels of this K step sit in box row (16k / Wb), (Wb + 2)-pixel rows, 8 x 16 B per pixel
                const uint32_t koff = (uint32_t)(((16 * k) / p.Wb) * (p.Wb + 2) + (16 * k) % p.Wb) * 8u;
#pragma unroll
                for (int tp = 0; tp < 3; ++tp)
                  umma_bf16(tmem_base + tp * ncx, da, descx_hi | (uint64_t)(bx_lo + 8u * tp + koff), idescx,
                            (it | k) != 0 ? 1u : 0u);
              }
            }
          } else
#pragma unroll
          for (int k = 0; k < kChunkPix / 16; ++k) {
            if (k < nk) {
              const uint64_t da = desc_hi | (uint64_t)(a_lo + 128u * k);
              umma_bf16(tmem_base, da, desc_hi | (uint64_t)(b_lo + 128u * k), idesc, (it | k) != 0 ? 1u : 0u);
              if (ncol1 > 0)
                umma_bf16(tmem_base + (uint32_t)(ncol0 * 64), da, desc_hi | (uint64_t)(b_lo + b1_off + 128u * k),
                          idesc1, (it | k) != 0 ? 1u : 0u);
            }
          }
          if constexpr (kPair) umma_commit_pair(&empty_bar[stage], 3);     // frees the stage in both CTAs
          else umma_commit(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one()) {
        if constexpr (kPair) umma_commit_pair(tmem_full_bar, 3);           // both CTAs drain their half of M = 256
        else umma_commit(tmem_full_bar);
      }
      __syncwarp();
    }
  } else if (warp >= 2) {
    // epilogue: row = output channel within the tile; columns = (column block, channel)
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const int co = (rowpair || p.fold == 2) ? (row & 63) : co_tile * 128 + row;
    const bool valid = co < p.cout;
    float* out = p.ws + ((size_t)split * p.cout + (valid ? co : 0)) * ((size_t)p.taps * p.ctot);
    if (p.fold) out = p.ws + (size_t)split * 16 * p.cout * p.ctot;      // [phase][cout][2x2][ctot]
    if (nchunks > 0) {
      mbar_wait(tmem_full_bar, 0);
      tc_fence_after();
    }
    const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
    const int ncol_epi = p.fold == 1 ? 4 * xh_live : p.xh ? 3 * xh_live : ncol_live;
    for (int j = 0; j < ncol_epi; ++j) {
      int tap = rg * p.ksize + (j % p.ksize);
      int cib = cib_base + j / p.ksize;
      bool live = valid;
      if (p.fold) {
        // accumulator columns are [q][box][64]; q = (b, tx) (fold 1) or the shift b + tx (fold 2: b = M half)
        const int q = j / xh_live;
        const int fb = p.fold == 1 ? q >> 1 : row >> 6;
        const int ftx = p.fold == 1 ? q & 1 : q - fb;
        live = valid && ftx >= 0 && ftx < 2;
        cib = cib_base + j % xh_live;
        const int ph = (rg >> 1) * 2 + fb;
        tap = (ph * p.cout + (valid ? co : 0)) * 4 + (rg & 1) * 2 + (live ? ftx : 0);     // row index into [ph][co][tap]
      } else if (p.xh) {
        // accumulator columns are [tap s][box b][64]: b = X block (plain) or X row group (row-pair mode)
        const int sx = j / xh_live, b = j % xh_live;
        if (rowpair) {
          const int fr = row < 64 ? b + 1 : (b == 0 ? 0 : -1);
          live = fr >= 0;
          tap = (fr < 0 ? 0 : fr) * 3 + sx;
          cib = cib_base;
        } else {
          tap = rg * 3 + sx;
          cib = cib_base + b;
        }
      } else if (rowpair) {
        // group jg (X row h + jg + 1 - pad): dY row h -> filter row jg + 1, dY row h+1 -> filter row jg; the bottom
        // half of every group but the first repeats a filter row that the previous group already produced
        const int jg = j / grp_cols;
        const int fr = p.rp_dir > 0 ? (row < 64 ? jg + 1 : (jg == 0 ? 0 : -1)) : (row < 64 ? 0 : 1);
        live = fr >= 0;
        tap = (fr < 0 ? 0 : fr) * p.ksize + j % p.ksize;
        cib = cib_base + (j - jg * grp_cols) / p.ksize;
      }
      float* dst = out + (size_t)tap * p.ctot + cib * 64;
      const int cvalid = p.ctot - cib * 64;   // channels left in this block (>= 64 except for a ragged tail)
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float v[32];
        if (nchunks > 0) {
          tmem_ld32(taddr + j * 64 + half * 32, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0.f;
        }
        if (live) {
          if (cvalid >= 64) {
            float4* d4 = reinterpret_cast<float4*>(dst + half * 32);
#pragma unroll
            for (int q = 0; q < 8; ++q) d4[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (half * 32 + i < cvalid) dst[half * 32 + i] = v[i];
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) cluster_sync_all();       // no CTA leaves while its peer may still signal its barriers
  if (warp == 1) {
    if constexpr (kPair) tmem_dealloc_pair(tmem_base, tmem_cols);
    else tmem_dealloc(tmem_base, tmem_cols);
  }
}

// dw[i] = (accumulate ? dw[i] : 0) + sum_s ws[s][i]   (fixed summation order)
__global__ void wgrad_reduce_kernel(const float* __restrict__ ws, float* __restrict__ dw, long long count,
                                    int splits, int accumulate) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= count) return;
  float4 acc = accumulate ? *reinterpret_cast<const float4*>(dw + i) : make_float4(0.f, 0.f, 0.f, 0.f);
  // eight partial tiles in flight per thread (the splits are `count` floats apart); summation order stays 0, 1, 2, ...
  int s = 0;
  for (; s + 8 <= splits; s += 8) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = __ldg(reinterpret_cast<const float4*>(ws + (size_t)(s + u) * count + i));
#pragma unroll
    for (int u = 0; u < 8; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
  }
  for (; s < splits; ++s) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(ws + (size_t)s * count + i));
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4*>(dw + i) = acc;
}

// Small gradients (1x1 gate convolutions, Cout = 64 layers) with many splits: 32 float4 columns x 8 split lanes per block —
// lane l adds splits l, l + 8, ..., the lanes are combined in lane order through shared memory (fixed order).  With one
// thread per column these launches were a chain of ~150 dependent-latency loads on 2-36 blocks (30 us for 1 MB).
__global__ void __launch_bounds__(256) wgrad_reduce_wide_kernel(const float* __restrict__ ws, float* __restrict__ dw,
                                                                long long count, int splits, int accumulate) {
  __shared__ float4 sh[8][32];
  const int col = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const long long i = ((long long)blockIdx.x * 32 + col) * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < count) {
    int s = sl;
    for (; s + 24 < splits; s += 32) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const float4*>(ws + (size_t)(s + 8 * u) * count + i));
#pragma unroll
      for (int u = 0; u < 4; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
    }
    for (; s < splits; s += 8) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(ws + (size_t)s * count + i));
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  sh[sl][col] = acc;
  __syncthreads();
  if (sl == 0 && i < count) {
    float4 t = accumulate ? *reinterpret_cast<const float4*>(dw + i) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 8; ++k) { t.x += sh[k][col].x; t.y += sh[k][col].y; t.z += sh[k][col].z; t.w += sh[k][col].w; }
    *reinterpret_cast<float4*>(dw + i) = t;
  }
}

struct WgradPlan {
  WgradParams p;
  int splits, gy, gz, tn;
  long long count;
  int smem_bytes;
};

static int wgrad_plan(const b2_wgrad_args* a, WgradPlan* pl) {
  B2_REQUIRE(a != nullptr, B2_ERR_SHAPE, "null args");
  const int xstride = a->x_stride == 0 ? 1 : a->x_stride;
  B2_REQUIRE(a->ksize >= 1 && a->ksize <= 3, B2_ERR_SHAPE, "ksize %d unsupported", a->ksize);
  B2_REQUIRE(xstride == 1 || (xstride == 2 && a->ksize == 2), B2_ERR_SHAPE,
             "x_stride %d unsupported (2 only with ksize 2)", xstride);
  B2_REQUIRE(a->ksize != 2 || xstride == 2 || a->custom_pad != 0 || a->fold != 0, B2_ERR_SHAPE,
             "ksize 2 needs x_stride 2 or explicit tap offsets");
  B2_REQUIRE(a->cout % 8 == 0 && a->c0 % 8 == 0 && a->c1 % 8 == 0, B2_ERR_SHAPE, "channels must be multiples of 8");
  B2_REQUIRE(a->c1 == 0 || a->c0 % 64 == 0, B2_ERR_SHAPE, "c0=%d must be a multiple of 64 when c1>0", a->c0);
  B2_REQUIRE((a->c0 + a->c1) % 4 == 0, B2_ERR_SHAPE, "cin must be a multiple of 4");
  if (a->fold) {
    B2_REQUIRE(a->ksize == 2 && xstride == 1 && a->dy_mul == 2 && !a->custom_pad && a->dy_off_h == 0 &&
                   a->dy_off_w == 0, B2_ERR_SHAPE, "fold: ksize 2, dy_mul 2, no offsets / custom taps");
    B2_REQUIRE((a->cout == 64 || a->cout % 128 == 0) && a->c0 % 64 == 0 && a->c1 % 64 == 0, B2_ERR_SHAPE,
               "fold: cout %d must be 64 or a multiple of 128, cin a multiple of 64", a->cout);
  }
  WgradParams& p = pl->p;
  memset(&p, 0, sizeof(p));
  int rc = conv_tile_geometry(a->n, a->h, a->w, kChunkPix, &p.Wb, &p.Hb, &p.Nb, &p.tw, &p.th, &pl->tn);
  if (rc) return rc;
  p.num_chunks = p.tw * p.th * pl->tn;
  p.taps = a->ksize * a->ksize;
  p.cb0 = (a->c0 + 63) / 64;
  p.cb1 = (a->c1 + 63) / 64;
  p.cout = a->cout;
  p.ctot = a->c0 + a->c1;
  p.a_boxes = a->cout <= 64 ? 1 : 2;
  const int cbt = p.cb0 + p.cb1;
  p.ksize = a->ksize;
  p.pad_h = a->custom_pad ? a->pad_h : (a->ksize == 3 ? 1 : 0);
  p.pad_w = a->custom_pad ? a->pad_w : (a->ksize == 3 ? 1 : 0);
  p.xstride = xstride;
  // 3x3: two 64-channel X blocks x 3 taps per CTA (N 384 as two MMAs that share the dY tile, 3 pipeline stages):
  // the kernel is bound by the L2 -> SM load rate, and this moves 64 KB per 6.3 MFLOP instead of 40 KB per 3.1
  p.debug_skip = env_switch("B200SEG_DEBUG_SKIP", 0);
  p.cpb = a->ksize == 1 ? 4 : 2;
  if (p.cpb > cbt) p.cpb = cbt;
  p.ncolb = p.ksize * p.cpb;
  pl->gy = p.ksize;
  {
    const int dm = a->dy_mul == 0 ? 1 : a->dy_mul;
    const bool rp_ok = a->cout == 64 && xstride == 1 && p.Hb == 1 && p.Nb == 1 &&
                       env_switch("B200SEG_WG_ROWPAIR", 1) != 0;
    (void)dm;
    p.rowpair = 0;
    p.rp_dir = p.pad_h >= 1 ? 1 : -1;
    if (rp_ok && a->ksize == 3 && p.pad_h == 1) {              // two X rows x 3 taps x one channel block: N 384
      p.rowpair = 2;
      p.cpb = 1;
    } else if (rp_ok && a->ksize == 2) {       // one X row x 2 taps x two channel blocks: N 256
      p.rowpair = 1;
      p.cpb = cbt < 2 ? cbt : 2;
    }
    if (p.rowpair) {
      p.ncolb = p.rowpair * p.ksize * p.cpb;
      p.a_boxes = 2;
      pl->gy = 1;
    }
  }
  if (a->fold) {
    p.fold = a->cout == 64 ? 2 : 1;
    p.taps = 16;
    p.rowpair = 0;
    p.cpb = cbt < 2 ? cbt : 2;
    p.ncolb = (p.fold == 1 ? 4 : 3) * p.cpb;
    p.a_boxes = p.fold == 1 ? 2 : 1;
    pl->gy = 4;
  }
  p.a_bytes = p.fold == 1 ? 4 * kBoxBytes : 2 * kBoxBytes;
  p.gy = pl->gy;
  pl->gz = ((a->cout + 127) / 128) * ((cbt + p.cpb - 1) / p.cpb);
  const int base = pl->gy * pl->gz;
  // split-K factor: one CTA per SM is resident, so pick the split count (up to ~3 waves) whose grid fills whole
  // waves best; ties go to fewer splits (less workspace traffic)
  const int max_splits = (p.num_chunks + 7) / 8;   // at least 8 chunks (512 pixels) per split
  const int sms = num_sms();
  int splits = 1;
  double best = 0.0;
  for (int s = 1; s <= max_splits && (long long)s * base <= 3ll * sms + base; ++s) {
    const long long ctas = (long long)s * base;
    const long long waves = (ctas + sms - 1) / sms;
    const double eff = (double)ctas / (double)(waves * sms);
    if (eff > best + 0.02) {
      best = eff;
      splits = s;
    }
  }
  p.chunks_per_split = (p.num_chunks + splits - 1) / splits;
  splits = (p.num_chunks + p.chunks_per_split - 1) / p.chunks_per_split;
  pl->splits = splits;
  pl->count = (long long)a->cout * p.taps * p.ctot;
  {
    // X-halo mode: 3x3, unit stride, chunk = 64 consecutive pixels of one image row
    // chunk = Hb rows of Wb pixels (64 x 1, 32 x 2, 16 x 4): the halo box has Hb rows of Wb + 2 pixels <= 72 rows
    p.xh = (a->ksize == 3 && xstride == 1 && !a->custom_pad && p.Nb == 1 && p.Wb >= 16 &&
            (p.Wb + 2) * p.Hb * 128 <= kXhBox) ? 1 : 0;
    p.nbox = p.rowpair ? p.rowpair : p.cpb;
    if (p.fold) {
      p.xh = (p.Nb == 1 && p.Wb >= 16 && (p.Wb + 2) * p.Hb * 128 <= kXhBox) ? 1 : 0;
      B2_REQUIRE(p.xh, B2_ERR_SHAPE, "fold: image %dx%d too small for the halo-row chunks (Wb %d Hb %d Nb %d)", a->h,
                 a->w, p.Wb, p.Hb, p.Nb);
    }
  }
  // CTA pairs: 3x3 halo mode, two Cout tiles per pair, each CTA holds one of the two X boxes
  p.pair = (env_switch("B200SEG_WG_PAIR", 1) != 0 && p.xh && (a->ksize == 3 || p.fold == 1) && !p.rowpair && p.fold != 2 &&
            p.cpb == 2 && a->cout % 256 == 0 && cbt % 2 == 0 && p.debug_skip == 0) ? 1 : 0;
  p.b_stage_bytes = p.pair ? kXhBox : (p.xh ? p.nbox * kXhBox : p.ncolb * kBoxBytes);
  const int stage_bytes = p.a_bytes + p.b_stage_bytes;
  int stages = (200 * 1024) / stage_bytes;
  if (stages > 8) stages = 8;
  p.stages = stages;
  pl->smem_bytes = stages * stage_bytes + 256 + 1024;
  return B2_OK;
}

}  // namespace b2

extern "C" int64_t b2_conv_wgrad_workspace(const b2_wgrad_args* a) {
  b2::WgradPlan pl;
  int rc = b2::wgrad_plan(a, &pl);
  if (rc) return rc;
  return (int64_t)pl.splits * pl.count * 4;
}

extern "C" int b2_conv_wgrad(const b2_wgrad_args* a, b2_stream_t stream_) {
  using namespace b2;
  int rc = b2_arch_check();
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  WgradPlan pl;
  rc = wgrad_plan(a, &pl);
  if (rc) return rc;
  const int64_t need = (int64_t)pl.splits * pl.count * 4;
  B2_REQUIRE(a->workspace != nullptr && a->workspace_bytes >= need, B2_ERR_WORKSPACE,
             "wgrad workspace too small: need %lld B, have %lld B", (long long)need, (long long)a->workspace_bytes);
  B2_REQUIRE((reinterpret_cast<uintptr_t>(a->workspace) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->dw) & 15) == 0,
             B2_ERR_ALIGN, "workspace / dw must be 16B aligned");
  pl.p.ws = static_cast<float*>(a->workspace);

  CUtensorMap tmDY, tmX0, tmX1;
  {
    // dY as a 5-D tensor (64 ch, W, H, N, channel block): one box brings both 64-channel halves of the M tile,
    // laid out [block][pixel][64 ch] in smem
    B2_REQUIRE(a->lddy % 8 == 0 && a->cout % 8 == 0, B2_ERR_ALIGN, "dy channel count / stride must be multiples of 8");
    const uint64_t c_in_block = a->cout < 64 ? (uint64_t)a->cout : 64ull;
    const int dm = a->dy_mul == 0 ? 1 : a->dy_mul;
    B2_REQUIRE(a->dy_off_h >= 0 && a->dy_off_h < dm && a->dy_off_w >= 0 && a->dy_off_w < dm, B2_ERR_SHAPE,
               "bad dY placement mul=%d off=(%d,%d)", dm, a->dy_off_h, a->dy_off_w);
    const uint64_t fw = (uint64_t)a->w * dm, fh = (uint64_t)a->h * dm;     // underlying dY image extent
    const __nv_bfloat16* dyb = static_cast<const __nv_bfloat16*>(a->dy) +
                               ((long long)a->dy_off_h * fw + a->dy_off_w) * a->lddy;
    uint64_t dims[5] = {c_in_block, (uint64_t)a->w, (uint64_t)a->h, (uint64_t)a->n, (uint64_t)((a->cout + 63) / 64)};
    uint64_t str[5] = {2, (uint64_t)dm * a->lddy * 2, (uint64_t)dm * fw * a->lddy * 2, fh * fw * a->lddy * 2, 128};
    uint32_t box[5] = {64, (uint32_t)pl.p.Wb, (uint32_t)pl.p.Hb, (uint32_t)pl.p.Nb, (uint32_t)pl.p.a_boxes};
    if (pl.p.fold) {
      // the fine tensor itself, traversed with stride 2 in w and h: coordinate (2w + b, 2h + a) selects the phase
      uint64_t fdims[5] = {c_in_block, fw, fh, (uint64_t)a->n, (uint64_t)((a->cout + 63) / 64)};
      uint64_t fstr[5] = {2, (uint64_t)a->lddy * 2, fw * a->lddy * 2, fh * fw * a->lddy * 2, 128};
      uint32_t fbox[5] = {64, (uint32_t)pl.p.Wb * 2, (uint32_t)pl.p.Hb * 2, (uint32_t)pl.p.Nb, (uint32_t)pl.p.a_boxes};
      uint32_t fes[5] = {1, 2, 2, 1, 1};
      rc = encode_tmap_bf16(&tmDY, a->dy, 5, fdims, fstr, fbox, CU_TENSOR_MAP_SWIZZLE_128B, fes);
    } else if (pl.p.rowpair) {
      uint32_t box4[4] = {64, (uint32_t)pl.p.Wb, 1, 1};
      rc = encode_tmap_bf16(&tmDY, dyb, 4, dims, str, box4, CU_TENSOR_MAP_SWIZZLE_128B);
    } else {
      rc = encode_tmap_bf16(&tmDY, dyb, 5, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    }
    if (rc) return rc;
  }
  const int xboxw = pl.p.xh ? pl.p.Wb + 2 : pl.p.Wb;
  const int xs = pl.p.xstride, xh = a->h * xs, xw = a->w * xs;     // X extent (2x the dY grid for ConvTranspose)
  rc = encode_act_tmap_ex(&tmX0, a->x0, a->c0, a->n, xh, xw, a->ldx0, (long long)a->ldx0 * xw,
                          (long long)a->ldx0 * xw * xh, xboxw, pl.p.Hb, pl.p.Nb, xs);
  if (rc) return rc;
  if (a->c1 > 0) {
    rc = encode_act_tmap_ex(&tmX1, a->x1, a->c1, a->n, xh, xw, a->ldx1, (long long)a->ldx1 * xw,
                            (long long)a->ldx1 * xw * xh, xboxw, pl.p.Hb, pl.p.Nb, xs);
    if (rc) return rc;
  } else {
    tmX1 = tmX0;
  }
  {
    // (the weight gradients are launched from the autograd engine thread, possibly several at once: set exactly once)
    static std::once_flag attr_once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(attr_once, [] {
      cudaError_t e = cudaFuncSetAttribute(conv_wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(conv_wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(conv_wgrad_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 cudaSharedmemCarveoutMaxShared);
      // Ask for the full 228 KB shared-memory carveout even when a launch needs less: the driver otherwise picks the
      // smallest configuration that fits this kernel (196 KB for 194 KB used), and the memory-bound kernels meant to
      // run next to it on the side-stream schedule (BatchNorm backward, gate) find no shared memory left on the SM.
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(conv_wgrad_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 cudaSharedmemCarveoutMaxShared);
      attr_err = e;
    });
    B2_CHECK_CUDA(attr_err);
  }
  dim3 grid(pl.gy * pl.gz, pl.splits, 1);
  if (pl.p.pair) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(kWgThreads);
    cfg.dynamicSmemBytes = (size_t)pl.smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    B2_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_wgrad_kernel<true>, tmDY, tmX0, tmX1, pl.p));
  } else {
    conv_wgrad_kernel<false><<<grid, kWgThreads, pl.smem_bytes, stream>>>(tmDY, tmX0, tmX1, pl.p);
  }
  B2_LAUNCH_CHECK();
  const long long n4 = (pl.count + 3) / 4;
  if (n4 <= 16384 && pl.splits >= 16)
    wgrad_reduce_wide_kernel<<<(unsigned)((n4 + 31) / 32), 256, 0, stream>>>(pl.p.ws, a->dw, pl.count, pl.splits,
                                                                            a->accumulate);
  else
  wgrad_reduce_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, stream>>>(pl.p.ws, a->dw, pl.count, pl.splits,
                                                                       a->accumulate);
  B2_LAUNCH_CHECK();
  return B2_OK;
}
