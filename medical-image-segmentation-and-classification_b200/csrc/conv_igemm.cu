// b200seg — implicit-GEMM convolution (stride 1, 'same' padding, 1x1 / 3x3) on tcgen05: persistent, warp-specialised.
//
// GEMM view:  D[M = pixels, N = cout] = sum over (tap, channel block)  A_tap[pixels, 64 ch] * W_tap[cout, 64 ch]^T
//   A tiles : one TMA box (64 ch, Wb, Hb, Nb) of the NHWC activation per (tap, channel block); the box origin is
//             shifted by the tap offset and TMA's out-of-bounds zero fill supplies the padding halo.  The box
//             lands in smem as 128 rows of 128 B (K-major, 128B swizzle) == the canonical UMMA A layout.
//             "halo" mode (tiles that are a single image-row segment, W >= 128): ONE box of Wb+2 pixels per
//             (filter row, channel block); the three horizontal taps are three MMAs whose A descriptors start
//             0 / 128 / 256 B into that box, so the activation is fetched 3x instead of 9x.
//   B tiles : TMA box (64 ch, BLOCK_N, 1 or 3 taps) of the packed weights [tap][cout][cin], same layout.
//   D       : 128 x BLOCK_N fp32 accumulators in TMEM, double buffered (2 x BLOCK_N columns).
// One CTA per SM loops over its tiles (fixed n-tile, strided m-tiles):
//   warp 0    TMA producer (smem ring of `stages` A+B slots, full/empty mbarriers)
//   warp 1    TMEM allocator + single-thread tcgen05.mma issuer; tcgen05.commit frees smem slots and publishes
//             a finished accumulator (tmem_full); waits on tmem_empty before overwriting a buffer
//   warps 2-5 epilogue group 0, warps 6-9 epilogue group 1 (used when the drain, not the MMAs, paces a tile: small K;
//             the groups take alternate tiles = alternate TMEM buffers and own one staging tile each):
//             tcgen05.ld -> +bias (+addend) (ReLU) -> bf16 -> swizzled smem tile -> TMA store; BatchNorm sum /
//             sum-of-squares of the ROUNDED output are column sums of that smem tile (16-byte reads), kept in fp64
//             registers across all tiles of the CTA and flushed through shuffles + smem with one fp64 atomic per
//             channel and group at the end.
// Double-M work items (BLOCK_N <= 128, large layers): two consecutive m-tiles share every weight stage — two A slots
// per stage, four accumulators in TMEM, one epilogue group per tile.  The kernel is bound by the bytes each SM pulls
// through the L2 -> SM fabric, and the weight tile is 75 % of them at N <= 128; sharing it is worth 14-29 % per layer.
// Clusters of 2 or 4 CTAs that multicast the weight tiles to each other were built and removed: no change at 2 CTAs,
// slower at 4 (the multicast does not relieve what bounds these tiles).
// A Cout = 64 "row-pair" mode (two output rows per tile, stacked taps, N = 128 MMAs) was built and removed: isolated
// 64->64 @256^2 0.390 -> 0.366 ms, but inside the training step, where the weight gradients load the same L2 -> SM
// fabric, the gain vanished.
// CTA pairs (cta_group::2, IgemmParams::pair): the two CTAs of a 2-cluster share one M = 256 MMA, each holding its own
// 128-pixel activation tile and half of the weight rows, which halves the weight bytes every SM pulls through the
// L2 -> SM fabric without needing a second set of accumulators (the N = 256 layers fill TMEM with two buffers already).
// The epilogue of tile i overlaps the main loop of tile i+1.
//
// Used for fprop (reference nn.Conv2d call sites, see include/b200seg.h) and for dgrad (flipped/transposed
// weight packing).  The K dimension may span two source tensors (elided torch.cat).
#include <stdlib.h>
#include <mutex>

#include "common.cuh"
#include "igemm_util.cuh"

namespace b2 {

static constexpr int kMaxEpiGroups = 2;
static constexpr int kThreads = 64 + 128 * kMaxEpiGroups;   // producer + MMA warps, then 4 epilogue warps per group
static constexpr int kMaxStages = 12;

struct IgemmParams {
  int H, W, N;
  int Wb, Hb, Nb;     // box extents; Wb*Hb*Nb == 128
  int tw, th;         // tiles along W and H
  int taps;           // 1 or 9
  int cb0, cb1;       // 64-channel blocks in source 0 / 1
  int block_n, stages, num_k_iters;
  int cout, n_tiles, m_tiles;
  int halo;
  int dm;             // "double-M" mode: a work item is TWO consecutive m-tiles that share every weight stage (two A
                      // slots per stage, four accumulators in TMEM): halves the weight bytes a CTA pulls through the
                      // L2 -> SM fabric per FLOP.  BLOCK_N <= 128.
  int stride, ksize, pad_h, pad_w;
  int a_stage_bytes, b_stage_bytes, a_tx_bytes;
  int epi_groups;     // 1 or 2 epilogue warp groups (two staging tiles)
  int ctile_bytes;    // bytes of one staging tile (128 x block_n bf16; at least one 64-channel panel in gate mode)
  int debug_skip;     // timing experiments only (B200SEG_DEBUG_SKIP): 1 = no TMA loads, 2 = no MMAs, 4 = no drain
  int fold;           // folded-UpConv launches (AttentionUNet.py:15-27 as four 2x2 phase convolutions) merged into ONE:
                      //   1 = fprop: the phase (a, b) is an extra tile dimension; tile t belongs to phase t / m_tiles_phase,
                      //       uses weight taps 4*phase .. 4*phase+3 with tap offsets (u - (1-a), v - (1-b)) and stores to
                      //       y[n, 2h+a, 2w+b, :] through a 5-D view (b*C + c, w, a, h, n) of the fine grid;
                      //   2 = dgrad: the four phases are ONE K loop of 16 taps, tap o = 4*phase + 2u + v reading the
                      //       (a, b) sub-lattice of dz at offset (u - a, v - b) through the same kind of 5-D view — no
                      //       addend chain, one epilogue per output tile instead of four.
  int fold_c;         // channel count of the fine-grid tensor behind the 5-D view (fprop: Cout, dgrad: C of dz)
  int m_tiles_phase;  // fold == 1: m-tiles per phase
  int fold_il;        // fold == 1: the phase is the INNER tile dimension — tile index t = 8 * pair + 2 * phase + member, so the
                      // four phases of a pair of coarse tiles run back to back (in neighbouring clusters) and the coarse
                      // input is fetched from DRAM once instead of once per phase (128 -> 64 @128^2: 1074 -> 270 MB read);
                      // consecutive tiles (a CTA pair / a double-M item) keep sharing one phase = one set of weights
  uint32_t mg_nt, mg_tw, mg_th, mg_mtp;   // magic multipliers (ceil(2^32 / d)) of n_tiles, tw, th, m_tiles_phase: the tile
                      // decode runs once per tile in every warp role and integer division was 8 % of the epilogue's time
  int wres;           // weight-resident mode: the CTA's whole weight slab (all taps x channel blocks of its single n-tile;
                      // all four phases of a merged UpConv fprop) is loaded into shared memory ONCE and the ring only
                      // carries activations.  The Cout = 64 layers at 256^2 were bound by the L2 -> SM fabric
                      // (64->64: 51 KB of activations + 36 KB of weights per 128-pixel tile at ~10 TB/s chip-wide).
  int wres_bytes;     // bytes of the resident slab (this CTA's half in pair mode)
  int pair;           // CTA-pair mode (2-CTA clusters, kernel instantiation kPair): ONE tcgen05.mma.cta_group::2 with
                      // M = 256 covers the two m-tiles of the pair; each CTA stages its own activation tile and HALF of
                      // the weight rows in its own shared memory (each SM receives half the weight bytes), the rank-0
                      // CTA issues the MMAs, every CTA drains its own 128 accumulator rows
  const float* bias;
  const __nv_bfloat16* addend;
  int add_tma;        // the addend tile is TMA-loaded into the group's staging tile at the START of the tile's drain (same
                      // box and swizzle as the output store) and added in place: per-thread row loads issued after the
                      // accumulator was ready made every 32-column chunk pay a global-memory round trip inside the drain
  int ldadd;
  double* stats;
  double* stats_partial;   // deterministic mode: [gridDim.x * epi_groups][2 * cout] rows, one per (CTA, epilogue group)
  int relu;
  int add_after_act;
  // fused eval-mode attention gate (b2_gate_fused): the GEMM is [g | x] . [s_g W_g ; s_x W_x]^T (+ folded biases), the
  // epilogue turns each accumulator ROW (one pixel, all F_int columns — one thread) into
  //   psi = sigmoid(s1 * (bpsi + sum_f wpsi[f] * relu(acc[f])) + h1)   and stores   out[pixel, :] = x[pixel, :] * psi
  const __nv_bfloat16* gate_x;    // nullptr: ordinary convolution epilogue
  int gate_ldx, gate_c;           // channel stride / channel count of x and out (tmY describes out, 64-channel boxes)
  const float* gate_wpsi;         // [F_int]
  const float* gate_k;            // device scalars: bpsi, scale1, shift1 (three pointers packed below)
  const float* gate_s1;
  const float* gate_h1;
};

// kPair: the CTA-pair variant is a separate instantiation — a kernel that contains cta_group::2 instructions can only
// be launched as (multiples of) 2-CTA clusters, so the single-CTA kernel must not contain them.
template <bool kHasAdd, bool kPair>
__global__ void __launch_bounds__(kThreads, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                  const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmY,
                  const __grid_constant__ CUtensorMap tmAdd, const IgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const bool dm = !kPair && p.dm != 0;                                 // pair mode never runs double-M items
  const int a_slots = dm ? 2 : 1;                                      // activation tiles per stage
  const int nbuf = dm ? 4 : 2;                                         // accumulators in TMEM
  const int stage_bytes = a_slots * p.a_stage_bytes + (p.wres ? 0 : p.b_stage_bytes);
  const int ctile_bytes = p.ctile_bytes;
  uint8_t* ctile0 = smem + p.stages * stage_bytes;                     // per group: 128 x block_n bf16, 1024 B aligned
  uint8_t* wres_base = ctile0 + p.epi_groups * ctile_bytes;            // resident weights (wres mode), 1024 B aligned
  uint8_t* tail = wres_base + p.wres_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tmem_full_bar = empty_bar + kMaxStages;                    // [4]
  uint64_t* tmem_empty_bar = tmem_full_bar + 4;                        // [4]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 4);
  uint64_t* wres_bar = reinterpret_cast<uint64_t*>(tail + 264);        // resident weights have landed
  uint64_t* add_bar = reinterpret_cast<uint64_t*>(tail + 272);         // [kMaxEpiGroups]: a group's addend tile has landed
  float* s_bias0 = reinterpret_cast<float*>(tail + 320);               // [group][256]
  float* s_psi0 = s_bias0 + kMaxEpiGroups * 256;                       // [group][256] (fused gate: psi weights)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // Work items ("super tiles") are numbered n-fastest: item u = (m-group u / n_tiles, n-tile u % n_tiles); the CTA of
  // rank r in its cluster takes m-tile m-group * cluster + r, cluster q takes items q, q + #clusters, ...
  constexpr int C = kPair ? 2 : 1;                                     // CTAs per cluster
  const uint32_t crank = kPair ? cluster_ctarank() : 0u;
  const int cluster_id = (int)blockIdx.x / C;
  const int num_clusters = (int)gridDim.x / C;
  const int per_item = dm ? 2 : C;                                     // m-tiles per work item
  const int total_items = ((p.m_tiles + per_item - 1) / per_item) * p.n_tiles;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);   // pair mode: one multicast commit of the leader's MMAs frees it in both CTAs
    }
    mbar_init(wres_bar, 1);
    for (int b = 0; b < kMaxEpiGroups; ++b) mbar_init(&add_bar[b], 1);
    for (int b = 0; b < 4; ++b) {
      mbar_init(&tmem_full_bar[b], 1);
      mbar_init(&tmem_empty_bar[b], kPair ? 8u : 4u);   // one arrival per epilogue warp (of both CTAs of a pair)
    }
    fence_barrier_init();
    tma_prefetch_desc(&tmA0);
    tma_prefetch_desc(&tmB);
    if (p.cb1 > 0) tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmY);
  }
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < nbuf * p.block_n) tmem_cols <<= 1;
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
  if constexpr (kPair) cluster_sync_all();   // the peer's barriers are initialised before anything can signal them
  tc_fence_after();
  // (B200SEG_PDL) everything above — barrier init, descriptor prefetch, TMEM allocation — may overlap the previous
  // kernel's tail; nothing below may run before that kernel has completed
  pdl_enter();
  const uint32_t tmem_base = *tmem_slot;
  const int cbt = p.cb0 + p.cb1;

  if (warp == 0) {
    // ------------------------------ TMA producer (warp-uniform control flow) ------------------------------
    int stage = 0;
    uint32_t phase = 0;
    // pair mode: the leader's barrier collects the bytes of BOTH CTAs (own A tile + half of B each)
    const uint32_t tx = (uint32_t)(a_slots * p.a_tx_bytes + (p.wres ? 0 : p.b_stage_bytes)) * (uint32_t)C;
    const int b_rows = p.block_n / C;            // weight rows this CTA fetches per tap
    if (p.wres) {
      // weight-resident mode: every weight block the K loop of a tile walks — (phase,) tap group o, channel block cb,
      // in that order, the same boxes the streamed stages use — is fetched once, onto one barrier (n_tiles == 1)
      if (elect_one()) {
        const uint32_t wtx = (uint32_t)p.wres_bytes * (uint32_t)C;
        uint32_t lbar = 0u;
        if constexpr (kPair) {
          lbar = mapa_shared(smem_u32(wres_bar), 0);
          if (crank == 0) mbar_arrive_expect_tx(wres_bar, wtx);
        } else {
          mbar_arrive_expect_tx(wres_bar, wtx);
        }
        (void)lbar;
        const int outer_n = p.halo ? 3 : p.taps;
        const int nph = p.fold == 1 ? 4 : 1;
        int j = 0;
        for (int ph = 0; ph < nph; ++ph) {
          for (int o = 0; o < outer_n; ++o) {
            const int wtap = p.fold == 1 ? ph * 4 + o : (p.halo ? o * 3 : o);
            for (int cb = 0; cb < cbt; ++cb, ++j) {
              uint8_t* sb = wres_base + j * p.b_stage_bytes;
              if constexpr (kPair) tma_load_3d_pair(sb, &tmB, lbar, cb * kKBlock, (int)crank * b_rows, wtap);
              else tma_load_3d(sb, &tmB, wres_bar, cb * kKBlock, 0, wtap);
            }
          }
        }
      }
      __syncwarp();
    }
    for (int item = cluster_id; item < total_items; item += num_clusters) {
      const int m_group = fast_div(item, p.n_tiles, p.mg_nt);
      const int n_tile = item - m_group * p.n_tiles;
      // pixel origin of the item's tile(s); a ragged last item recomputes the last tile (its result is dropped)
      int w0s[2], h0s[2], n0s[2];
      int tph = 0;                                 // fold == 1: the phase of the item's tile(s)
      for (int q = 0; q < a_slots; ++q) {
        int t = m_group * per_item + (dm ? q : (int)crank);
        if (t >= p.m_tiles) t = p.m_tiles - 1;
        if (p.fold == 1) {
          if (p.fold_il) {
            tph = (t >> 1) & 3;
            t = ((t >> 3) << 1) | (t & 1);
          } else {
            tph = fast_div(t, p.m_tiles_phase, p.mg_mtp);
            t -= tph * p.m_tiles_phase;
          }
        }
        const int t1 = fast_div(t, p.tw, p.mg_tw);
        const int tw_i = t - t1 * p.tw;
        const int tn_i = fast_div(t1, p.th, p.mg_th);
        const int th_i = t1 - tn_i * p.th;
        w0s[q] = tw_i * p.Wb;
        h0s[q] = th_i * p.Hb;
        n0s[q] = tn_i * p.Nb;
      }
      const int w0 = w0s[0], h0 = h0s[0], n0 = n0s[0];
      const int outer = p.halo ? 3 : p.taps;      // halo mode: one iteration per (input row, channel block)
      for (int o = 0; o < outer; ++o) {
        int dr = 0, ds = 0, tap0 = o;
        int fa = 0, fb = 0;                        // fold == 2: sub-lattice (a, b) of dz this tap reads
        if (p.fold == 2) {
          fa = o >> 3;
          fb = (o >> 2) & 1;
          dr = ((o >> 1) & 1) - fa;
          ds = (o & 1) - fb;
        } else if (p.fold == 1) {
          dr = (o >> 1) - (1 - (tph >> 1));
          ds = (o & 1) - (1 - (tph & 1));
          tap0 = tph * 4 + o;
        } else if (p.halo) {
          dr = o - 1;
          ds = -1;
          tap0 = o * 3;
        } else {
          dr = o / p.ksize - p.pad_h;
          ds = o % p.ksize - p.pad_w;
        }
        for (int cb = 0; cb < cbt; ++cb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
            uint8_t* sa = smem + stage * stage_bytes;
            uint8_t* sb = sa + a_slots * p.a_stage_bytes;
            // one activation box (4-D NHWC box, or the 5-D sub-lattice view of the merged UpConv dgrad)
            auto load_a = [&](uint8_t* dst, int qw0, int qh0, int qn0, uint32_t lbar) {
              const CUtensorMap* tm = cb < p.cb0 ? &tmA0 : &tmA1;
              const int c = (cb < p.cb0 ? cb : cb - p.cb0) * kKBlock;
              if (p.fold == 2) {
                if constexpr (kPair) tma_load_5d_pair(dst, tm, lbar, fb * p.fold_c + c, qw0 + ds, fa, qh0 + dr, qn0);
                else tma_load_5d(dst, tm, &full_bar[stage], fb * p.fold_c + c, qw0 + ds, fa, qh0 + dr, qn0);
              } else {
                if constexpr (kPair) tma_load_4d_pair(dst, tm, lbar, c, p.stride * qw0 + ds, p.stride * qh0 + dr, qn0);
                else tma_load_4d(dst, tm, &full_bar[stage], c, p.stride * qw0 + ds, p.stride * qh0 + dr, qn0);
              }
            };
            if constexpr (kPair) {
              // both CTAs load into their own smem; completion is counted on the LEADER's barrier, which only the
              // leader arms (its arrive + expect_tx may come after the peer's bytes: the phase needs both)
              const uint32_t lbar = mapa_shared(smem_u32(&full_bar[stage]), 0);
              if (crank == 0) mbar_arrive_expect_tx(&full_bar[stage], tx);
              load_a(sa, w0, h0, n0, lbar);
              if (!p.wres)
                tma_load_3d_pair(sb, &tmB, lbar, cb * kKBlock, n_tile * p.block_n + (int)crank * b_rows, tap0);
            } else {
            if (p.debug_skip & 1) {
              mbar_arrive(&full_bar[stage]);
            } else {
            mbar_arrive_expect_tx(&full_bar[stage], tx);
            load_a(sa, w0, h0, n0, 0u);
            if (dm) load_a(sa + p.a_stage_bytes, w0s[1], h0s[1], n0s[1], 0u);   // second tile of the item
            if (!p.wres) tma_load_3d(sb, &tmB, &full_bar[stage], cb * kKBlock, n_tile * p.block_n, tap0);
            }
            }
          }
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 && !(kPair && crank != 0)) {
    // ------------------------------ MMA issuer (pair mode: the leader CTA only) ------------------------------
    const uint32_t idesc = umma_idesc_bf16(kPair ? 2 * kTileM : kTileM, p.block_n, 0, 0);
    const uint32_t b_tap_step = (uint32_t)(kPair ? p.block_n / 2 : p.block_n) * 8u;   // descriptor units between taps
    const uint64_t desc0 = umma_desc_sw128(0, 16, 1024);          // K-major SW128 descriptor with start address 0
    const uint64_t desc_hi = desc0 & 0xFFFFFFFF00000000ull;
    const uint32_t desc_lo0 = (uint32_t)desc0;
    int stage = 0;
    uint32_t phase = 0;
    int ti = 0;
    const int sub = p.halo ? 3 : 1;
    const int nb_shift = dm ? 2 : 1;             // log2(accumulators in TMEM)
    const uint32_t wres_addr = smem_u32(wres_base);
    if (p.wres) {
      mbar_wait(wres_bar, 0);                    // the resident weights (of both CTAs of a pair) have landed
      tc_fence_after();
    }
    for (int item = cluster_id; item < total_items; item += num_clusters, ++ti) {
      int wres_it0 = 0;                          // wres + merged UpConv fprop: first weight block of the tile's phase
      if (p.wres && p.fold == 1) {
        int t = fast_div(item, p.n_tiles, p.mg_nt) * per_item;
        if (t >= p.m_tiles) t = p.m_tiles - 1;
        wres_it0 = (p.fold_il ? ((t >> 1) & 3) : fast_div(t, p.m_tiles_phase, p.mg_mtp)) * p.num_k_iters;
      }
      // local tile counter lt = a_slots * ti + q  ->  accumulator lt % nbuf, barrier phase (lt / nbuf) & 1
      for (int q = 0; q < a_slots; ++q) {
        const uint32_t lt = (uint32_t)(a_slots * ti + q);
        mbar_wait(&tmem_empty_bar[lt & (nbuf - 1)], ((lt >> nb_shift) & 1u) ^ 1u);
      }
      tc_fence_after();
      for (int it = 0; it < p.num_k_iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_addr = smem_u32(smem + stage * stage_bytes);
          const uint32_t b_addr = p.wres ? wres_addr + (uint32_t)((wres_it0 + it) * p.b_stage_bytes)
                                         : a_addr + a_slots * p.a_stage_bytes;
          // Descriptors differ only in the 14-bit start-address field (bytes >> 4) of the low word, and smem
          // addresses are < 256 KB, so stepping a descriptor is one 32-bit add: +2 per 16-element K step (32 B),
          // +8 per pixel of halo shift (128 B), +8 * BLOCK_N per weight tap.  This keeps the single issuing thread
          // at a few instructions per MMA — it paces the N <= 128 tiles otherwise.
          const int nsub = (p.debug_skip & 2) ? 0 : sub;
          for (int q = 0; q < a_slots; ++q) {
            const uint32_t lt = (uint32_t)(a_slots * ti + q);
            const uint32_t d_tmem = tmem_base + (lt & (uint32_t)(nbuf - 1)) * (uint32_t)p.block_n;
            uint32_t a_lo = desc_lo0 + ((a_addr + (uint32_t)(q * p.a_stage_bytes)) >> 4);
            uint32_t b_lo = desc_lo0 + (b_addr >> 4);
            for (int s = 0; s < nsub; ++s) {     // (a fully unrolled 12-MMA variant measured slower)
              if constexpr (kPair) {
#pragma unroll
                for (int k = 0; k < kKBlock / 16; ++k)
                  umma_bf16_pair(d_tmem, desc_hi | (uint64_t)(a_lo + 2 * k), desc_hi | (uint64_t)(b_lo + 2 * k), idesc,
                                 (it | s | k) != 0 ? 1u : 0u);
              } else {
#pragma unroll
                for (int k = 0; k < kKBlock / 16; ++k)
                  umma_bf16(d_tmem, desc_hi | (uint64_t)(a_lo + 2 * k), desc_hi | (uint64_t)(b_lo + 2 * k), idesc,
                            (it | s | k) != 0 ? 1u : 0u);
              }
              a_lo += 8;
              b_lo += b_tap_step;
            }
          }
          // frees this smem slot (in both CTAs of a pair) when the MMAs have read it
          if constexpr (kPair) umma_commit_pair(&empty_bar[stage], 3);
          else umma_commit(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one()) {
        for (int q = 0; q < a_slots; ++q) {
          uint64_t* fb = &tmem_full_bar[(uint32_t)(a_slots * ti + q) & (uint32_t)(nbuf - 1)];
          if constexpr (kPair) umma_commit_pair(fb, 3);      // both CTAs drain their half of the M = 256 accumulator
          else umma_commit(fb);
        }
      }
      __syncwarp();
    }
  } else if (warp >= 2 && ((warp - 2) >> 2) < p.epi_groups) {
    // ---------------- epilogue: group 0 = warps 2..5, group 1 = warps 6..9 (tiles alternate between groups) ----------------
    const int g = (warp - 2) >> 2;
    const int G = p.epi_groups;
    const int et = (threadIdx.x - 64) & 127;   // 0..127 within the group
    uint8_t* ctile = ctile0 + g * ctile_bytes;
    float* s_bias = s_bias0 + g * 256;
    float* s_psi = s_psi0 + g * 256;
    const int bar_id = 1 + g;
    if (p.stats_partial != nullptr) {
      // the flushes below add into this group's row, and a CTA may never meet some n-tile: zero the row first (after
      // pdl_enter above — the previous finish may read the workspace until then), then sync the group
      double* srow = p.stats_partial + (size_t)(blockIdx.x * G + g) * (2 * p.cout);
      for (int i = et; i < 2 * p.cout; i += 128) srow[i] = 0.0;
      asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
    }
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access
    const int row = quad * 32 + lane;          // accumulator row == pixel within the tile
    const int wl = row % p.Wb;
    const int hl = (row / p.Wb) % p.Hb;
    const int nl = row / (p.Wb * p.Hb);
    const bool relu = p.relu != 0;
    // statistics mapping: a thread owns one 16 B chunk (8 channels) for a slab of `nchunks` rows
    const int nchunks = p.block_n >> 3;        // 4, 8, 16 or 32 chunks per row; 128 / nchunks slabs
    const int schunk = lane % nchunks;         // == et % nchunks (nchunks divides 32)
    const int sgrp = et / nchunks;
    double acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.0;
    // fp32 partial sums of the last few tiles (32 values each, as many as one N = 256 tile contributes): the fp64 pipe
    // is narrow, so the conversion + DADD per channel runs once per 32 rows instead of once per tile
    float fs[8], fq[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) fs[j] = fq[j] = 0.f;
    int fpending = 0;
    auto fold_stats = [&]() {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc[j] += (double)fs[j];
        acc[8 + j] += (double)fq[j];
        fs[j] = fq[j] = 0.f;
      }
      fpending = 0;
    };

    // add the group's partial sums into stats[]: lanes owning the same chunk are combined by shuffles, the four
    // warps through the (idle) staging tile, so each channel costs one fp64 atomic per group and flush
    auto flush_stats = [&](int n_tile_) {
      fold_stats();
      for (int off = nchunks; off < 32; off <<= 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], off);
      }
      if (et == 0) tma_store_wait_read();
      asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");    // staging tile is free
      double* red = reinterpret_cast<double*>(ctile);                 // [warp][sum | sumsq][block_n]
      if (lane < nchunks) {
        double* r0 = red + ((warp - 2) & 3) * 2 * p.block_n + schunk * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          r0[j] = acc[j];
          r0[p.block_n + j] = acc[8 + j];
        }
      }
      asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
      for (int i = et; i < 2 * p.block_n; i += 128) {
        const int which = i / p.block_n, c = i % p.block_n;
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < 4; ++w) v += red[(w * 2 + which) * p.block_n + c];
        const int sidx = which * p.cout + n_tile_ * p.block_n + c;
        if (p.stats_partial != nullptr)      // this thread owns slot sidx of this (CTA, group) row for the whole launch
          p.stats_partial[(size_t)(blockIdx.x * p.epi_groups + g) * (2 * p.cout) + sidx] += v;
        else
          atomicAdd(&p.stats[sidx], v);
      }
      // (the staging tile is next written after another group barrier, see the tile loop)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = 0.0;
    };

    int cur_n_tile = -1;
    uint32_t add_phase = 0;                      // parity of this group's addend barrier
    const int nb_shift = dm ? 2 : 1;             // log2(accumulators in TMEM)
    // ti = local tile counter of this CTA (group g takes ti = g, g + G, ...); double-M: item = ti / 2, tile ti & 1
    for (int ti = g;; ti += G) {
      const int item = cluster_id + (dm ? (ti >> 1) : ti) * num_clusters;
      if (item >= total_items) break;
      const int m_group = fast_div(item, p.n_tiles, p.mg_nt);
      const int n_tile = item - m_group * p.n_tiles;
      const int ch_base = n_tile * p.block_n;
      int t = m_group * per_item + (dm ? (ti & 1) : (int)crank);
      int eph = 0;                                 // fold == 1: phase of this tile
      if (p.fold == 1 && t < p.m_tiles) {
        eph = p.fold_il ? ((t >> 1) & 3) : fast_div(t, p.m_tiles_phase, p.mg_mtp);
      }
      if (t >= p.m_tiles || (p.debug_skip & 4)) {
        // ragged last group: this CTA only kept the pipeline protocol going; hand the accumulator straight back
        const int dbuf = ti & (nbuf - 1);
        mbar_wait(&tmem_full_bar[dbuf], ((uint32_t)ti >> nb_shift) & 1u);
        tc_fence_after();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (kPair) mbar_arrive_remote(&tmem_empty_bar[dbuf], 0);
          else mbar_arrive(&tmem_empty_bar[dbuf]);
        }
        continue;
      }
      if (n_tile != cur_n_tile) {
        // new output-channel slab: flush the statistics kept for the previous one, reload the bias slice
        if (cur_n_tile >= 0 && p.stats != nullptr) flush_stats(cur_n_tile);
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");   // everyone is done reading the old bias slice
        for (int i = et; i < p.block_n; i += 128) {
          s_bias[i] = p.bias ? p.bias[ch_base + i] : 0.f;
          if (p.gate_x != nullptr) s_psi[i] = p.gate_wpsi[i];
        }
        cur_n_tile = n_tile;
      }
      if (p.fold == 1) t = p.fold_il ? (((t >> 3) << 1) | (t & 1)) : t - eph * p.m_tiles_phase;
      const int t1 = fast_div(t, p.tw, p.mg_tw);
      const int tw_i = t - t1 * p.tw;
      const int tn_i = fast_div(t1, p.th, p.mg_th);
      const int th_i = t1 - tn_i * p.th;
      const int w0 = tw_i * p.Wb, h0 = th_i * p.Hb, n0 = tn_i * p.Nb;
      // pixels of the tile that exist (tiles at the right / bottom / batch edge are clipped): row r of the tile is pixel
      // (n0 + r / (Wb Hb), h0 + (r / Wb) % Hb, w0 + r % Wb); all three box extents are powers of two
      const bool tile_full = w0 + p.Wb <= p.W && h0 + p.Hb <= p.H && n0 + p.Nb <= p.N;
      auto row_valid = [&](int r) {
        return tile_full || (w0 + r % p.Wb < p.W && h0 + (r / p.Wb) % p.Hb < p.H && n0 + r / (p.Wb * p.Hb) < p.N);
      };
      const int buf = ti & (nbuf - 1);

      // the group's previous TMA store must have finished READING the staging tile before it is overwritten
      if (et == 0) tma_store_wait_read();
      asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
      if (kHasAdd && p.add_tma) {
        // the addend tile lands in the staging tile while this group waits for the accumulator
        if (et == 0) {
          mbar_arrive_expect_tx(&add_bar[g], (uint32_t)(kTileM * p.block_n * 2));
          for (int pn = 0; pn < (p.block_n >> 6); ++pn)
            tma_load_4d(ctile + pn * (kTileM * 128), &tmAdd, &add_bar[g], ch_base + pn * 64, w0, h0, n0);
        }
      }

      mbar_wait(&tmem_full_bar[buf], ((uint32_t)ti >> nb_shift) & 1u);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * p.block_n);
      const bool valid = row_valid(row);
      const uint32_t row_off = p.block_n >= 64 ? (uint32_t)row * 128u : (uint32_t)row * 64u;
      const uint32_t row_x = p.block_n >= 64 ? (uint32_t)(row & 7) : (uint32_t)((row >> 1) & 3);
      const __nv_bfloat16* arow = nullptr;
      if (kHasAdd) {
        const long long pix = ((long long)(n0 + nl) * p.H + (h0 + hl)) * p.W + (w0 + wl);
        arow = valid ? p.addend + pix * p.ldadd + ch_base : nullptr;
        // The addend rows are plain global loads issued after the accumulator is ready, so every 32-column chunk of a
        // tile used to pay a DRAM round trip inside the drain (the gate's 1x1 dgrad with the direct x gradient as
        // addend ran at 3.7 TB/s where the same launch without addend reaches 5 TB/s).  Pull the rows of the NEXT tile
        // this group will drain into L2 now; its loads then hit L2.
        const int ti2 = ti + G;
        const int item2 = cluster_id + (dm ? (ti2 >> 1) : ti2) * num_clusters;
        if (p.add_tma) {
          mbar_wait(&add_bar[g], add_phase);
          add_phase ^= 1u;
        } else if (item2 < total_items) {
          const int m_group2 = fast_div(item2, p.n_tiles, p.mg_nt);
          const int t2 = m_group2 * per_item + (dm ? (ti2 & 1) : (int)crank);
          if (t2 < p.m_tiles) {
            const int u1 = fast_div(t2, p.tw, p.mg_tw);
            const int u_w = t2 - u1 * p.tw;
            const int u_n = fast_div(u1, p.th, p.mg_th);
            const int u_h = u1 - u_n * p.th;
            const int w2 = u_w * p.Wb + wl, h2 = u_h * p.Hb + hl, n2 = u_n * p.Nb + nl;
            if (w2 < p.W && h2 < p.H && n2 < p.N) {
              const __nv_bfloat16* nrow = p.addend + (((long long)n2 * p.H + h2) * p.W + w2) * p.ldadd +
                                          (item2 - m_group2 * p.n_tiles) * p.block_n;
              for (int c = 0; c < p.block_n; c += 64) asm volatile("prefetch.global.L2 [%0];" ::"l"(nrow + c));
            }
          }
        }
      }
      if (p.gate_x != nullptr) {
        // ---------------- fused attention-gate epilogue (eval mode) ----------------
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");      // s_bias / s_psi of this slab are in place
        float q = 0.f;
        for (int c = 0; c < p.block_n; c += 32) {
          float v[32];
          tmem_ld32(taddr + c, v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 32; ++e) q = fmaf(fmaxf(v[e] + s_bias[c + e], 0.f), s_psi[c + e], q);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (kPair) mbar_arrive_remote(&tmem_empty_bar[buf], 0);
          else mbar_arrive(&tmem_empty_bar[buf]);
        }
        const float qn = fmaf(q + __ldg(p.gate_k), __ldg(p.gate_s1), __ldg(p.gate_h1));
        const float ps = 1.f / (1.f + __expf(-qn));
        const long long pix = ((long long)(n0 + nl) * p.H + (h0 + hl)) * p.W + (w0 + wl);
        const __nv_bfloat16* xrow = valid ? p.gate_x + pix * p.gate_ldx : nullptr;
        for (int pn = 0; pn < (p.gate_c >> 6); ++pn) {
          if (pn > 0) {                      // the previous panel's TMA store must have read the staging tile
            if (et == 0) tma_store_wait_read();
            asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
          }
#pragma unroll
          for (int q8 = 0; q8 < 8; ++q8) {
            uint4 u = xrow != nullptr ? __ldg(reinterpret_cast<const uint4*>(xrow + pn * 64) + q8) : make_uint4(0, 0, 0, 0);
            u.x = pack_bf16x2(bf16lo(u.x) * ps, bf16hi(u.x) * ps);
            u.y = pack_bf16x2(bf16lo(u.y) * ps, bf16hi(u.y) * ps);
            u.z = pack_bf16x2(bf16lo(u.z) * ps, bf16hi(u.z) * ps);
            u.w = pack_bf16x2(bf16lo(u.w) * ps, bf16hi(u.w) * ps);
            *reinterpret_cast<uint4*>(ctile + (uint32_t)row * 128u + (((uint32_t)q8 ^ (uint32_t)(row & 7)) << 4)) = u;
          }
          fence_proxy_async();
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
          if (et == 0) {
            tma_store_4d(&tmY, ctile, pn * 64, w0, h0, n0);
            tma_store_commit();
          }
        }
        continue;
      }
      for (int c = 0; c < p.block_n; c += 32) {
        float v[32];
        tmem_ld32(taddr + c, v);
        // bias slice for these 32 columns (broadcast reads) while the TMEM load is in flight
        float bs[32];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c + q * 4);
          bs[q * 4 + 0] = b4.x; bs[q * 4 + 1] = b4.y; bs[q * 4 + 2] = b4.z; bs[q * 4 + 3] = b4.w;
        }
        // staging address of this row's 16 B chunks: panel (64 channels) + row + swizzled chunk
        const uint32_t cbase = (uint32_t)(c >> 6) * (uint32_t)(kTileM * 128) + row_off;
        const uint32_t chunk0 = (uint32_t)((c & 63) >> 3);
        uint4 au[4];
        if (kHasAdd) {
          if (p.add_tma) {           // the TMA-loaded addend tile has the layout of the output tile: read in place
#pragma unroll
            for (int q = 0; q < 4; ++q)
              au[q] = *reinterpret_cast<const uint4*>(ctile + cbase + (((chunk0 + q) ^ row_x) << 4));
          } else {
#pragma unroll
            for (int q = 0; q < 4; ++q)
              au[q] = arow != nullptr ? __ldg(reinterpret_cast<const uint4*>(arow + c) + q) : make_uint4(0, 0, 0, 0);
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t pk[4];
          const uint32_t aw[4] = {kHasAdd ? au[q].x : 0u, kHasAdd ? au[q].y : 0u, kHasAdd ? au[q].z : 0u,
                                  kHasAdd ? au[q].w : 0u};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int e = q * 8 + 2 * j;
            float a = v[e] + bs[e];
            float b = v[e + 1] + bs[e + 1];
            if (kHasAdd) {
              const float a0 = bf16lo(aw[j]), a1 = bf16hi(aw[j]);
              if (p.add_after_act) {    // x + relu(conv(.)): the addend joins after the activation (on rounded values)
                if (relu) {
                  a = fmaxf(a, 0.f);
                  b = fmaxf(b, 0.f);
                }
                a = bf16_round(a) + a0;
                b = bf16_round(b) + a1;
              } else {
                a += a0;
                b += a1;
                if (relu) {
                  a = fmaxf(a, 0.f);
                  b = fmaxf(b, 0.f);
                }
              }
            } else if (relu) {
              a = fmaxf(a, 0.f);
              b = fmaxf(b, 0.f);
            }
            pk[j] = pack_bf16x2(a, b);
          }
          *reinterpret_cast<uint4*>(ctile + cbase + (((chunk0 + q) ^ row_x) << 4)) =
              make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
      // accumulator drained: hand the TMEM buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (kPair) mbar_arrive_remote(&tmem_empty_bar[buf], 0);    // the leader's MMA thread waits for both CTAs
        else mbar_arrive(&tmem_empty_bar[buf]);
      }
      fence_proxy_async();                       // generic-proxy smem writes -> visible to the TMA store
      asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");

      if (et == 0) {
        if (p.fold == 1) {          // phase (a, b) of the fine grid: 5-D view (b*C + c, w, a, h, n)
          for (int pn = 0; pn < (p.block_n >> 6); ++pn)
            tma_store_5d(&tmY, ctile + pn * (kTileM * 128), (eph & 1) * p.fold_c + ch_base + pn * 64, w0, eph >> 1, h0,
                         n0);
        } else if (p.block_n >= 64) {
          for (int pn = 0; pn < (p.block_n >> 6); ++pn)
            tma_store_4d(&tmY, ctile + pn * (kTileM * 128), ch_base + pn * 64, w0, h0, n0);
        } else {
          tma_store_4d(&tmY, ctile, ch_base, w0, h0, n0);     // 32-channel tile: 64 B rows, 64B-swizzle map
        }
        tma_store_commit();
      }
      if (p.stats != nullptr) {
        // column sums of the ROUNDED outputs (what BatchNorm sees under autocast), 8 channels per thread: rows
        // r_begin .. r_begin + nchunks - 1 of the staged tile, chunk `schunk`
        const int r_begin = sgrp * nchunks;
        if (tile_full) {
          // whole tile valid: batches of rows whose loads are all in flight before the first one is consumed
          if (p.block_n >= 64) {      // nchunks = 8 / 16 / 32, r_begin % 8 == 0: row r_begin + i has swizzle term i & 7
            const uint8_t* base = ctile + (uint32_t)(schunk >> 3) * (uint32_t)(kTileM * 128) + (uint32_t)r_begin * 128u;
            const uint32_t sc7 = (uint32_t)(schunk & 7);
            for (int i0 = 0; i0 < nchunks; i0 += 8) {
              uint4 u[8];
#pragma unroll
              for (int i = 0; i < 8; ++i)
                u[i] = *reinterpret_cast<const uint4*>(base + (uint32_t)(i0 + i) * 128u + ((sc7 ^ (uint32_t)i) << 4));
#pragma unroll
              for (int i = 0; i < 8; ++i) stats_accum(u[i], fs, fq);
            }
          } else {                    // 32-channel tiles: nchunks = 4, 64 B rows, chunk ^= (row >> 1) & 3
            uint4 u[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint32_t r = (uint32_t)(r_begin + i);
              u[i] = *reinterpret_cast<const uint4*>(ctile + r * 64u + ((((uint32_t)schunk) ^ ((r >> 1) & 3u)) << 4));
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) stats_accum(u[i], fs, fq);
          }
        } else {
          for (int r = r_begin; r < r_begin + nchunks; ++r) {
            if (!row_valid(r)) continue;
            stats_accum(*reinterpret_cast<const uint4*>(ctile + ctile_off(p.block_n, r, schunk * 8)), fs, fq);
          }
        }
        if (++fpending * nchunks >= 32) fold_stats();   // every 8, 4, 2, 1 tiles for N = 32, 64, 128, 256
      }
    }
    if (p.stats != nullptr && cur_n_tile >= 0) flush_stats(cur_n_tile);
    if (et == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) cluster_sync_all();   // no CTA leaves while its peer may still signal its barriers
  if (warp == 1) {
    if constexpr (kPair) tmem_dealloc_pair(tmem_base, tmem_cols);
    else tmem_dealloc(tmem_base, tmem_cols);
  }
}

// Tile geometry shared with the wgrad kernel: split `tile_pix` pixels into a (Wb, Hb, Nb) box of power-of-two extents,
// Wb * Hb * Nb == tile_pix.  Any image extent is accepted (the reference is fully convolutional, AttentionUNet.py:86-121:
// 224^2, 320^2, 384^2 ...): tiles at the right / bottom / batch edge are CLIPPED — TMA loads zero-fill the pixels outside
// the tensor (they add nothing to a weight gradient), TMA stores drop them, and the epilogue masks them out of the
// BatchNorm statistics.  For extents that are powers of two or multiples of 128 nothing is clipped.
static int pow2ceil_i(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}
int conv_tile_geometry(int n, int h, int w, int tile_pix, int* Wb, int* Hb, int* Nb, int* tw, int* th, int* tn) {
  B2_REQUIRE(n > 0 && h > 0 && w > 0, B2_ERR_SHAPE, "bad extent n=%d h=%d w=%d", n, h, w);
  int wb = pow2ceil_i(w);
  if (wb > tile_pix) wb = tile_pix;
  const int rows = tile_pix / wb;
  int hb = pow2ceil_i(h);
  if (hb > rows) hb = rows;
  *Wb = wb;
  *Hb = hb;
  *Nb = rows / hb;
  *tw = (w + wb - 1) / wb;
  *th = (h + hb - 1) / hb;
  *tn = (n + *Nb - 1) / *Nb;
  return B2_OK;
}

// General NHWC view: element strides (s_w, s_h, s_n) of the pixel grid, optional traversal stride `es` in w and h
// (box extents are given in LOADED pixels).
int encode_act_tmap_ex(CUtensorMap* tm, const void* base, int c, int n, int h, int w, long long s_w, long long s_h,
                       long long s_n, int Wb, int Hb, int Nb, int es) {
  B2_REQUIRE(s_w % 8 == 0 && s_h % 8 == 0 && s_n % 8 == 0 && c % 8 == 0, B2_ERR_ALIGN,
             "channel count %d / pixel strides must be multiples of 8 elements", c);
  B2_REQUIRE(Wb * es <= 256 && Hb * es <= 256, B2_ERR_SHAPE, "TMA box too large for stride %d", es);
  uint64_t dims[4] = {(uint64_t)c, (uint64_t)w, (uint64_t)h, (uint64_t)n};
  uint64_t str[4] = {2, (uint64_t)s_w * 2, (uint64_t)s_h * 2, (uint64_t)s_n * 2};
  uint32_t box[4] = {64, (uint32_t)(Wb * es), (uint32_t)(Hb * es), (uint32_t)Nb};
  uint32_t est[4] = {1, (uint32_t)es, (uint32_t)es, 1};
  return encode_tmap_bf16(tm, base, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, est);
}

int encode_act_tmap(CUtensorMap* tm, const void* base, int c, int ld, int n, int h, int w, int Wb, int Hb, int Nb) {
  return encode_act_tmap_ex(tm, base, c, n, h, w, ld, (long long)ld * w, (long long)ld * w * h, Wb, Hb, Nb, 1);
}

static int env_int(const char* name, int dflt) { return env_switch(name, dflt); }

static int pick_block_n(int cout, bool wide_rows) {
  const int forced = env_int("B200SEG_BLOCK_N", 0);
  // N = 256 tiles do not leave room for >= 3 pipeline stages in halo mode (3 taps of B per stage)
  if (forced > 0 && cout % forced == 0 && !(forced > 128 && wide_rows)) return forced;
  if (cout % 256 == 0 && !wide_rows) return 256;   // deep layers: halves the activation re-fetch, 96 B/clk smem feed
  if (cout % 128 == 0) return 128;
  if (cout % 64 == 0) return 64;
  if (cout % 32 == 0) return 32;
  return 0;
}

struct GateExtra {            // fused eval-mode attention gate (b2_gate_fused): see IgemmParams::gate_x
  const void* x;
  int ldx, c;
  const float *wpsi, *bpsi, *scale1, *shift1;
};

int conv_c64_try_launch(const b2_conv_args* a, cudaStream_t stream);     // conv_c64.cu

static int conv_igemm_launch(const b2_conv_args* a, cudaStream_t stream, const GateExtra* gate = nullptr) {
  B2_REQUIRE(a != nullptr, B2_ERR_SHAPE, "null args");
  if (gate == nullptr) {
    // Cout = 64 3x3 layers on wide images: the row-streaming kernel (N = 192 MMAs, every input row fetched once)
    const int rc64 = conv_c64_try_launch(a, stream);
    if (rc64 != 0) return rc64 < 0 ? rc64 : B2_OK;
  }
  const int stride = a->stride == 0 ? 1 : a->stride;
  const int out_mul = a->out_mul == 0 ? 1 : a->out_mul;
  B2_REQUIRE(a->ksize >= 1 && a->ksize <= 3, B2_ERR_SHAPE, "ksize %d unsupported (1, 2 or 3)", a->ksize);
  const int fold = a->fold_mode;
  B2_REQUIRE(fold >= 0 && fold <= 2, B2_ERR_SHAPE, "fold_mode %d unsupported", fold);
  if (fold != 0) {
    B2_REQUIRE(gate == nullptr && a->ksize == 2 && a->c1 == 0 && a->addend == nullptr && (a->stride == 0 || a->stride == 1) &&
                   (a->out_mul == 0 || a->out_mul == 1) && (a->in_mul == 0 || a->in_mul == 1) && a->c0 % 64 == 0 &&
                   a->cout % 64 == 0,
               B2_ERR_SHAPE, "merged UpConv launch: plain 2x2 taps, one K source, channels multiples of 64");
    B2_REQUIRE(a->ldx0 == a->c0 && a->ldy == a->cout, B2_ERR_SHAPE, "merged UpConv launch needs dense tensors");
  }
  B2_REQUIRE(stride == 1 || stride == 2, B2_ERR_SHAPE, "stride %d unsupported (1 or 2)", stride);
  const int in_mul = a->in_mul == 0 ? 1 : a->in_mul;
  B2_REQUIRE(a->ksize != 2 || stride == 2 || a->custom_pad != 0 || fold != 0, B2_ERR_SHAPE,
             "ksize 2 needs stride 2 or explicit tap offsets");
  B2_REQUIRE(in_mul >= 1 && (in_mul == 1 || stride == 1) && a->in_off_h >= 0 && a->in_off_h < in_mul &&
                 a->in_off_w >= 0 && a->in_off_w < in_mul,
             B2_ERR_SHAPE, "bad input placement mul=%d off=(%d,%d)", in_mul, a->in_off_h, a->in_off_w);
  B2_REQUIRE(out_mul >= 1 && a->out_off_h >= 0 && a->out_off_h < out_mul && a->out_off_w >= 0 &&
                 a->out_off_w < out_mul,
             B2_ERR_SHAPE, "bad output placement mul=%d off=(%d,%d)", out_mul, a->out_off_h, a->out_off_w);
  B2_REQUIRE(a->n > 0 && a->h > 0 && a->w > 0, B2_ERR_SHAPE, "bad extent n=%d h=%d w=%d", a->n, a->h, a->w);
  B2_REQUIRE(a->c0 > 0 && a->c1 >= 0, B2_ERR_SHAPE, "bad channel counts c0=%d c1=%d", a->c0, a->c1);
  B2_REQUIRE(a->c1 == 0 || a->c0 % 64 == 0, B2_ERR_SHAPE, "c0=%d must be a multiple of 64 when c1>0", a->c0);
  B2_REQUIRE(a->ktot >= a->c0 + a->c1 && a->ktot % 8 == 0, B2_ERR_SHAPE, "ktot=%d inconsistent", a->ktot);
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  p.block_n = pick_block_n(a->cout, a->ksize == 3 && a->w >= kTileM);
  B2_REQUIRE(p.block_n != 0, B2_ERR_SHAPE, "cout=%d must be a multiple of 32", a->cout);
  B2_REQUIRE(a->ldy % 8 == 0 && (reinterpret_cast<uintptr_t>(a->y) & 15) == 0, B2_ERR_ALIGN, "y misaligned");
  B2_REQUIRE(a->addend == nullptr || (a->ldadd % 8 == 0 && (reinterpret_cast<uintptr_t>(a->addend) & 15) == 0),
             B2_ERR_ALIGN, "addend misaligned");
  int tn;
  int rc = conv_tile_geometry(a->n, a->h, a->w, kTileM, &p.Wb, &p.Hb, &p.Nb, &p.tw, &p.th, &tn);
  if (rc) return rc;
  p.H = a->h; p.W = a->w; p.N = a->n;
  p.taps = fold == 2 ? 16 : a->ksize * a->ksize;
  p.fold = fold;
  p.fold_c = fold == 1 ? a->cout : a->c0;
  p.cb0 = (a->c0 + 63) / 64;
  p.cb1 = (a->c1 + 63) / 64;
  const int cbt = p.cb0 + p.cb1;
  p.cout = a->cout;
  p.m_tiles = p.tw * p.th * tn;
  // Small M (batch 1 ... 4 per GPU at the deep levels): with fewer work items than half the SMs every item streams its
  // whole K range of activations anyway, so narrower tiles cost nothing there and put 2-4x as many SMs to work on the
  // weights (a 1024 -> 1024 @16^2 layer at batch 4: 16 -> 64 items).  The fused gate needs F_int in one tile.
  if (gate == nullptr && env_int("B200SEG_BLOCK_N", 0) == 0 && env_int("B200SEG_SMALL_M", 1) != 0) {
    const int slots = num_sms() / 2;               // CTA pairs
    while (p.block_n > 64 && (long long)((p.m_tiles * (fold == 1 ? 4 : 1) + 1) / 2) * (a->cout / p.block_n) * 2 <= slots)
      p.block_n /= 2;
  }
  p.n_tiles = a->cout / p.block_n;
  p.m_tiles_phase = p.m_tiles;
  p.fold_il = (fold == 1 && p.m_tiles % 2 == 0) ? 1 : 0;
  if (fold == 1) p.m_tiles *= 4;                 // the four phases are an extra tile dimension
  p.bias = a->bias;
  p.addend = static_cast<const __nv_bfloat16*>(a->addend);
  p.ldadd = a->ldadd;
  p.stats = a->stats;
  p.relu = a->relu;
  p.add_after_act = (a->addend != nullptr && a->add_after_act) ? 1 : 0;
  p.stride = stride;
  p.ksize = a->ksize;
  p.pad_h = a->custom_pad ? a->pad_h : (a->ksize == 3 ? 1 : 0);
  p.pad_w = a->custom_pad ? a->pad_w : (a->ksize == 3 ? 1 : 0);
  // halo mode: 3x3, tile == one row segment of 128 pixels
  p.halo = (p.taps == 9 && stride == 1 && !a->custom_pad && p.Hb == 1 && p.Nb == 1 && p.Wb == kTileM) ? 1 : 0;
  if (p.halo) {
    p.a_tx_bytes = (kTileM + 2) * 128;
    p.a_stage_bytes = ((p.a_tx_bytes + 1023) / 1024) * 1024;
    p.b_stage_bytes = 3 * p.block_n * 128;
    p.num_k_iters = 3 * cbt;
  } else {
    p.a_tx_bytes = kTileM * 128;
    p.a_stage_bytes = kTileM * 128;
    p.b_stage_bytes = p.block_n * 128;
    p.num_k_iters = p.taps * cbt;
  }
  int ctile_bytes = kTileM * p.block_n * 2;
  if (gate != nullptr) {
    B2_REQUIRE(p.n_tiles == 1 && out_mul == 1 && in_mul == 1 && stride == 1 && a->ksize == 1,
               B2_ERR_SHAPE, "fused gate: F_int=%d must be one tile (32 | 64 | 128 | 256) of a plain 1x1 GEMM", a->cout);
    B2_REQUIRE(gate->c % 64 == 0 && gate->ldx % 8 == 0 && (reinterpret_cast<uintptr_t>(gate->x) & 15) == 0, B2_ERR_SHAPE,
               "fused gate: C=%d must be a multiple of 64, x 16 B aligned", gate->c);
    if (ctile_bytes < kTileM * 128) ctile_bytes = kTileM * 128;       // one 64-channel output panel
    p.gate_x = static_cast<const __nv_bfloat16*>(gate->x);
    p.gate_ldx = gate->ldx;
    p.gate_c = gate->c;
    p.gate_wpsi = gate->wpsi;
    p.gate_k = gate->bpsi;
    p.gate_s1 = gate->scale1;
    p.gate_h1 = gate->shift1;
  }
  p.ctile_bytes = ctile_bytes;
  const int tail_bytes = 320 + 2 * kMaxEpiGroups * 256 * 4 + 192;      // barriers, bias + psi slices, slack
  // Double-M: two consecutive m-tiles per work item share every weight stage (see IgemmParams::dm).  Needs four
  // accumulators in TMEM (BLOCK_N <= 128), two A slots per stage and still >= 2 (>= 3 for thin stages) stages.
  {
    const int want = env_int("B200SEG_DM", 2);      // 0 = off, 1 = only with two epilogue groups, 2 = also with one
    p.dm = 0;
    if (want != 0 && p.block_n <= 128 && p.m_tiles >= env_int("B200SEG_DM_MIN_TILES", 4 * num_sms()) &&
        !(fold == 1 && p.m_tiles_phase % 2 != 0)) {
      const int sb2 = 2 * p.a_stage_bytes + p.b_stage_bytes;
      const int g2 = 232448 - 1024 - tail_bytes - 2 * ctile_bytes, g1 = g2 + ctile_bytes;
      if (g2 / sb2 >= 2 || (want == 2 && g1 / sb2 >= 2)) p.dm = 1;
    }
  }
  // CTA pairs (cta_group::2): B200SEG_PAIR = 0 off, 1 the N = 256 tiles (no room in TMEM for the double-M sharing),
  // 2 (default) every eligible layer (replaces double-M there).  Measured at batch 64 (profiles/r02_conv_layers_pair*):
  // N = 256 layers 1224 -> 1460 ... 1385 -> 1637 TFLOP/s, 64 -> 128 @128^2 944 -> 1218, 64 -> 64 @256^2 853 -> 910;
  // conv_igemm time inside the training step 16.3 -> 14.7 ms.
  p.debug_skip = env_int("B200SEG_DEBUG_SKIP", 0);
  {
    const int want = env_int("B200SEG_PAIR", 2);
    p.pair = 0;
    if (want != 0 && p.m_tiles >= 2 && p.block_n % 16 == 0 && (want >= 2 || p.block_n == 256) &&
        !(fold == 1 && p.m_tiles_phase % 2 != 0) && p.debug_skip == 0) {
      p.pair = 1;
      p.dm = 0;
      p.b_stage_bytes /= 2;          // each CTA of the pair stages half of the weight rows
    }
  }
  int stage_bytes = (p.dm ? 2 : 1) * p.a_stage_bytes + p.b_stage_bytes;
  // Two epilogue groups (two staging tiles) when the accumulator drain, not the MMA, paces a tile: the drain costs
  // about 1750 + 36 * BLOCK_N clocks per tile per group (measured), the MMAs K/16 * BLOCK_N/2.  A second group is
  // not worth giving up pipeline stages for when the main loop is the longer of the two anyway.
  {
    const long long mma_clk = (long long)p.num_k_iters * (p.halo ? 3 : 1) * (kKBlock / 16) * (p.block_n / 2);
    const long long epi_clk = 1750 + 36ll * p.block_n;
    const int forced_g = env_int("B200SEG_EPI_GROUPS", 0);
    p.epi_groups = forced_g > 0 ? (forced_g > kMaxEpiGroups ? kMaxEpiGroups : forced_g)
                                : (mma_clk * 5 < epi_clk * 6 ? 2 : 1);
    if (p.dm) p.epi_groups = 2;        // the two tiles of an item finish together: one group each
    const int budget2 = 232448 - 1024 - tail_bytes - 2 * ctile_bytes;
    if (p.epi_groups == 2 && budget2 / stage_bytes < 2) p.epi_groups = 1;
    // pair-mode N = 256 tiles: two 64 KB staging tiles leave three pipeline stages, which costs more than the second
    // group's drain overlap buys (128->256 @64^2 fprop: 0.164 ms with two groups, 0.125 ms with one)
    if (p.epi_groups == 2 && p.pair && p.block_n == 256 && forced_g == 0 && budget2 / stage_bytes < 4) p.epi_groups = 1;
  }
  // Weight-resident mode (IgemmParams::wres): one n-tile, the whole slab next to >= 4 activation-only stages, and
  // enough tiles per CTA that fetching all weights before the first MMA costs nothing.
  int budget = 232448 - 1024 - tail_bytes - p.epi_groups * ctile_bytes;
  p.wres = 0;
  p.wres_bytes = 0;
  {
    const long long wb = (long long)(fold == 1 ? 4 : 1) * p.num_k_iters * p.b_stage_bytes;
    const int a_only = (p.dm ? 2 : 1) * p.a_stage_bytes;
    if (p.n_tiles == 1 && p.debug_skip == 0 && p.m_tiles >= 4 * num_sms() && wb % 1024 == 0 &&
        (budget - wb) / a_only >= 4) {
      p.wres = 1;
      p.wres_bytes = (int)wb;
      stage_bytes = a_only;
      budget -= (int)wb;
    }
  }
  int stages = budget / stage_bytes;
  if (stages > kMaxStages) stages = kMaxStages;
  if (env_int("B200SEG_MAX_STAGES", 0) >= 2 && stages > env_int("B200SEG_MAX_STAGES", 0))
    stages = env_int("B200SEG_MAX_STAGES", 0);
  B2_REQUIRE(stages >= 2, B2_ERR_SHAPE, "tile configuration does not fit shared memory");
  p.stages = stages;
  const int smem_bytes = stages * stage_bytes + p.epi_groups * ctile_bytes + p.wres_bytes + tail_bytes + 1024;

  CUtensorMap tmA0, tmA1, tmB, tmY;
  const int boxw = p.halo ? p.Wb + 2 : p.Wb;
  const int ih = a->h * stride, iw = a->w * stride;      // extent of the sampled input grid
  if (fold == 2) {
    // dz [n, 2h, 2w, C] as (b*C + c, w, a, h, n): the (a, b) sub-lattices become coordinates of one 5-D map
    const uint64_t Cc = (uint64_t)a->c0, W2 = (uint64_t)a->w, H2 = (uint64_t)a->h;
    uint64_t dims[5] = {2 * Cc, W2, 2, H2, (uint64_t)a->n};
    uint64_t str[5] = {2, 2 * Cc * 2, 2 * W2 * Cc * 2, 4 * W2 * Cc * 2, 4 * H2 * W2 * Cc * 2};
    uint32_t box[5] = {64, (uint32_t)p.Wb, 1, (uint32_t)p.Hb, (uint32_t)p.Nb};
    rc = encode_tmap_bf16(&tmA0, a->x0, 5, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  } else {
    // underlying image is (ih*in_mul) x (iw*in_mul); the operand is its (in_off_h, in_off_w) sub-lattice
    const long long fw = (long long)iw * in_mul, fh = (long long)ih * in_mul;
    const long long off0 = ((long long)a->in_off_h * fw + a->in_off_w) * a->ldx0;
    rc = encode_act_tmap_ex(&tmA0, static_cast<const __nv_bfloat16*>(a->x0) + off0, a->c0, a->n, ih, iw,
                            (long long)in_mul * a->ldx0, (long long)in_mul * fw * a->ldx0, fh * fw * a->ldx0, boxw,
                            p.Hb, p.Nb, stride);
    if (rc) return rc;
  }
  if (a->c1 > 0) {
    B2_REQUIRE(in_mul == 1, B2_ERR_SHAPE, "input placement is not supported with two K sources");
    rc = encode_act_tmap_ex(&tmA1, a->x1, a->c1, a->n, ih, iw, a->ldx1, (long long)a->ldx1 * iw,
                            (long long)a->ldx1 * iw * ih, boxw, p.Hb, p.Nb, stride);
    if (rc) return rc;
  } else {
    tmA1 = tmA0;
  }
  {
    uint64_t dims[3] = {(uint64_t)(a->c0 + a->c1), (uint64_t)a->cout, (uint64_t)(fold == 1 ? 16 : p.taps)};
    uint64_t str[3] = {2, (uint64_t)a->ktot * 2, (uint64_t)a->w_tap_stride * 2};
    // all taps of the stage in one box; pair mode: this CTA's half of the rows
    uint32_t box[3] = {64, (uint32_t)(p.pair ? p.block_n / 2 : p.block_n), p.halo ? 3u : 1u};
    rc = encode_tmap_bf16(&tmB, a->wpk, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  // output pixel grid (possibly a strided sub-lattice of a larger image: ConvTranspose pixel shuffle)
  const long long ow = (long long)a->w * out_mul, oh = (long long)a->h * out_mul;
  const long long y_sw = (long long)out_mul * a->ldy;      // element strides of the output pixel grid
  const long long y_sh = (long long)out_mul * ow * a->ldy;
  const long long y_sn = oh * ow * a->ldy;
  void* y = static_cast<__nv_bfloat16*>(a->y) + ((long long)a->out_off_h * ow + a->out_off_w) * a->ldy;
  if (fold == 1) {                // y [n, 2h, 2w, Cout] as (b*C + c, w, a, h, n)
    B2_REQUIRE(p.block_n >= 64, B2_ERR_SHAPE, "merged UpConv fprop needs cout >= 64");
    const uint64_t Cc = (uint64_t)a->cout, W2 = (uint64_t)a->w, H2 = (uint64_t)a->h;
    uint64_t dims[5] = {2 * Cc, W2, 2, H2, (uint64_t)a->n};
    uint64_t str[5] = {2, 2 * Cc * 2, 2 * W2 * Cc * 2, 4 * W2 * Cc * 2, 4 * H2 * W2 * Cc * 2};
    uint32_t box[5] = {64, (uint32_t)p.Wb, 1, (uint32_t)p.Hb, (uint32_t)p.Nb};
    rc = encode_tmap_bf16(&tmY, a->y, 5, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
  } else if (gate != nullptr) {   // the gate's output has C channels (64-channel boxes), not F_int
    rc = encode_act_tmap_ex(&tmY, y, gate->c, a->n, a->h, a->w, y_sw, y_sh, y_sn, p.Wb, p.Hb, p.Nb, 1);
  } else if (p.block_n >= 64) {
    rc = encode_act_tmap_ex(&tmY, y, a->cout, a->n, a->h, a->w, y_sw, y_sh, y_sn, p.Wb, p.Hb, p.Nb, 1);
  } else {
    // 32-channel tiles are staged as 64 B rows with chunk ^= (row >> 1) & 3 == TMA's 64B swizzle
    uint64_t dims[4] = {(uint64_t)a->cout, (uint64_t)a->w, (uint64_t)a->h, (uint64_t)a->n};
    uint64_t str[4] = {2, (uint64_t)y_sw * 2, (uint64_t)y_sh * 2, (uint64_t)y_sn * 2};
    uint32_t box[4] = {32, (uint32_t)p.Wb, (uint32_t)p.Hb, (uint32_t)p.Nb};
    rc = encode_tmap_bf16(&tmY, y, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B);
  }
  if (rc) return rc;
  CUtensorMap tmAdd = tmY;
  p.add_tma = 0;
  if (a->addend != nullptr && p.block_n >= 64 && fold == 0 && gate == nullptr && out_mul == 1 && a->cout % 64 == 0) {
    rc = encode_act_tmap_ex(&tmAdd, a->addend, a->cout, a->n, a->h, a->w, a->ldadd, (long long)a->ldadd * a->w,
                            (long long)a->ldadd * a->w * a->h, p.Wb, p.Hb, p.Nb, 1);
    if (rc) return rc;
    p.add_tma = 1;
  }
  {
    // forward runs on the caller's thread, backward on the autograd engine's: set the attributes exactly once
    static std::once_flag attr_once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(attr_once, [] {
      cudaError_t e = cudaFuncSetAttribute(conv_igemm_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_igemm_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_igemm_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_igemm_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
      attr_err = e;
    });
    B2_CHECK_CUDA(attr_err);
  }
  // persistent grid: one CTA per SM.  When the number of clusters is a multiple of n_tiles every CTA keeps one n-tile
  // for its whole life and its BN statistics stay in registers; otherwise they are flushed whenever the slab changes.
  const int C = p.pair ? 2 : 1;        // CTAs per cluster: pair mode launches 2-CTA clusters
  int clusters = num_sms() / C;
  if (p.pair) {
    static std::mutex mc_mu;
    static int max_pairs = 0;
    std::lock_guard<std::mutex> mc_lock(mc_mu);
    if (max_pairs == 0) {
      cudaLaunchConfig_t qc = {};
      qc.gridDim = dim3((unsigned)(num_sms() / 2 * 2));
      qc.blockDim = dim3(kThreads);
      qc.dynamicSmemBytes = 232448;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = 2;
      qa[0].val.clusterDim.y = 1;
      qa[0].val.clusterDim.z = 1;
      qc.attrs = qa;
      qc.numAttrs = 1;
      int n = 0;
      B2_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&n, conv_igemm_kernel<false, false>, &qc));
      B2_REQUIRE(n > 0, B2_ERR_CUDA, "no cluster of 2 CTAs can be resident");
      max_pairs = n;
    }
    if (clusters > max_pairs) clusters = max_pairs;
  }
  const int per_item = p.dm ? 2 : C;
  const long long total = (long long)((p.m_tiles + per_item - 1) / per_item) * p.n_tiles;
  B2_REQUIRE(total < (1ll << 31), B2_ERR_SHAPE, "too many tiles");
  {
    // magic multipliers of the tile decode (fast_div): exact while dividend * divisor < 2^32
    auto magic = [](int d) { return d <= 1 ? 0u : (uint32_t)(((1ull << 32) + (uint64_t)d - 1) / (uint64_t)d); };
    // one condition per division of the decode: items / n_tiles; tiles (of one phase) / tw; (tiles / tw) / th; and, for
    // the merged UpConv fprop without interleaved phases only, tiles / m_tiles_phase
    const long long lim = 1ll << 32;
    const long long tiles1 = p.fold == 1 ? p.m_tiles_phase : p.m_tiles;
    const bool ok_nt = p.n_tiles <= 1 || total * p.n_tiles < lim;
    const bool ok_tw = p.tw <= 1 || tiles1 * p.tw < lim;
    const bool ok_th = p.th <= 1 || (tiles1 / (p.tw > 0 ? p.tw : 1) + 1) * p.th < lim;
    const bool ok_ph = !(p.fold == 1 && !p.fold_il) || (long long)p.m_tiles * p.m_tiles_phase < lim;
    B2_REQUIRE(ok_nt && ok_tw && ok_th && ok_ph, B2_ERR_SHAPE,
               "too many tiles for the tile decode (items %lld, n_tiles %d, m_tiles %d, tw %d, th %d)", total, p.n_tiles,
               p.m_tiles, p.tw, p.th);
    p.mg_nt = magic(p.n_tiles);
    p.mg_tw = magic(p.tw);
    p.mg_th = magic(p.th);
    p.mg_mtp = magic(p.m_tiles_phase);
  }
  if (clusters > total) clusters = (int)total;
  if (clusters > p.n_tiles && (total / clusters) >= 16) clusters = (clusters / p.n_tiles) * p.n_tiles;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(clusters * C));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = (size_t)smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // programmatic dependent launch (common.cuh): the kernel waits after its prologue; size rule on the output tensor
  if (pdl_allowed((long long)p.m_tiles * 128 * p.cout * 2)) {
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
  }
  DetBuf det;
  det.partial = nullptr;
  const long long det_rows = (long long)clusters * C * p.epi_groups;
  if (p.stats != nullptr) {
    rc = det_begin(&det, det_rows, 2 * p.cout, stream);
    if (rc) return rc;
  }
  p.stats_partial = det.partial;
  if (p.pair) {
    if (p.addend != nullptr)
      B2_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_igemm_kernel<true, true>, tmA0, tmA1, tmB, tmY, tmAdd, p));
    else
      B2_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_igemm_kernel<false, true>, tmA0, tmA1, tmB, tmY, tmAdd, p));
  } else if (p.addend != nullptr) {
    B2_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_igemm_kernel<true, false>, tmA0, tmA1, tmB, tmY, tmAdd, p));
  } else {
    B2_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_igemm_kernel<false, false>, tmA0, tmA1, tmB, tmY, tmAdd, p));
  }
  B2_LAUNCH_CHECK();
  if (det.partial) return det_finish(det.partial, det_rows, 2 * p.cout, 2 * p.cout, p.stats, stream);
  return B2_OK;
}

}  // namespace b2

extern "C" int b2_conv_fprop(const b2_conv_args* a, b2_stream_t stream) {
  int rc = b2_arch_check();
  if (rc) return rc;
  return b2::conv_igemm_launch(a, static_cast<cudaStream_t>(stream));
}

extern "C" int b2_conv_dgrad(const b2_conv_args* a, b2_stream_t stream) {
  int rc = b2_arch_check();
  if (rc) return rc;
  return b2::conv_igemm_launch(a, static_cast<cudaStream_t>(stream));
}

// Eval-mode attention gate in ONE launch (AttentionUNet.py:48-54 with the three BatchNorms folded):
//   out = x * sigmoid(s1 * (bpsi + wpsi . relu([g | x] . W^T + bias)) + h1)
extern "C" int b2_gate_fused(const b2_gate_args* g, b2_stream_t stream) {
  int rc = b2_arch_check();
  if (rc) return rc;
  B2_REQUIRE(g != nullptr && g->c > 0 && g->fint > 0, B2_ERR_SHAPE, "bad gate args");
  b2_conv_args a;
  memset(&a, 0, sizeof(a));
  a.n = g->n; a.h = g->h; a.w = g->w; a.ksize = 1;
  a.x0 = g->g; a.c0 = g->c; a.ldx0 = g->ldg;
  a.x1 = g->x; a.c1 = g->c; a.ldx1 = g->ldx;
  a.wpk = g->wpk; a.ktot = 2 * g->c; a.w_tap_stride = (int64_t)g->fint * 2 * g->c;
  a.cout = g->fint;
  a.y = g->out; a.ldy = g->ldo;
  a.bias = g->bias;
  b2::GateExtra gx;
  gx.x = g->x; gx.ldx = g->ldx; gx.c = g->c;
  gx.wpsi = g->wpsi; gx.bpsi = g->bpsi; gx.scale1 = g->scale1; gx.shift1 = g->shift1;
  return b2::conv_igemm_launch(&a, static_cast<cudaStream_t>(stream), &gx);
}
