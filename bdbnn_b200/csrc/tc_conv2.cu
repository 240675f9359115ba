// Persistent, warp-specialised tcgen05 implicit-GEMM conv (forward and dgrad), version 2.
//
// Why (measured on B200, profiles/r1_*): the one-tile-per-CTA kernel in tc_conv.cu is bound by
// L2->SM traffic and per-CTA latency, not by HBM or the tensor pipe: every 128-pixel tile re-reads
// the whole [BN x 9*C] weight slab and nine shifted activation boxes from L2 (1.0-1.4 GB per layer).
// Here one CTA per SM stays resident and each work item is a SUPER TILE of up to four 128-row M tiles
// (four TMEM accumulators) that
//   * share every weight stage  -> weight traffic / 4
//   * (halo mode) share ONE activation patch per 64-channel K block: the patch holds the super
//     tile's pixels in padded-width raster order plus the halo rows; tap (dh,dw) of M tile j is the
//     same swizzled patch viewed from row j*128 + (dh-dh_min)*PW + (dw-dw_min) — the UMMA descriptor
//     start address simply moves by whole 128-byte rows (absolute-address swizzle, base_offset 0).
//     Activation traffic drops from 9 boxes per tile to ~1.2 patches per 4 tiles.
//   * overlap roles across work items: warp 4 = TMA producer, warp 5 = MMA issuer, warps 0-3 =
//     epilogue; with BN <= 64 the eight accumulators form two buffers so the epilogue of item i
//     overlaps the MMAs of item i+1.
// Non-halo mode (small images, stride-2 forward) keeps per-tap boxes but still shares weight stages.
#include "tc_common.cuh"

namespace bdbnn {

// Warp roles: warps 0..7 = epilogue (two groups of four; group g = warp / 4 handles the 32-column blocks cb with
// (cb & 1) == g, both groups read every TMEM lane quadrant warp % 4), warp 8 = TMA producer, warp 9 = MMA issuer.
// Two epilogue groups double the loads / stores in flight per SM: with four warps the dgrad epilogue of the
// 56x56 layers (reads the STE mask and the shortcut gradient, writes gx: 0.5 GB per launch) was latency-bound
// at ~16 KB in flight per SM and left the MMA pipe idle more than half of the kernel (ncu: tensor pipe 17 %).
constexpr int kTc2Threads = 320;
constexpr int kEpiWarps = 8;

struct TcConv2Params {
  int32_t OW, OH, NIMG;
  int32_t halo;
  // non-halo tile box: BNI images x BH rows x BW(=OW) cols per M tile
  int32_t BW, BH, BNI, tiles_h, n_mtiles;
  // halo geometry: super tile = HBNI image blocks of IB padded rows (IB = (rows + dh_span) * PW when
  // HBNI > 1) or SH image rows of one image; patch box = [HBNI][PH][PW][64]
  int32_t PW, PH, SH, IB, HBNI, dh_min, dw_min, supers_per_img;
  uint32_t patch_bytes;
  int32_t n_supers, n_ntiles;
  int32_t Kc, n_kb, a_halves, in_step;
  int32_t n_taps;
  int8_t tap_dh[kMaxTaps], tap_dw[kMaxTaps];
  uint8_t tap_b[kMaxTaps];
  int32_t out_step, out_off_h, out_off_w, OHf, OWf;
  int32_t Nout, BN, NB, TS;
  int32_t stages;
  int32_t cg;                // CTAs per MMA: 1, or 2 (CTA pair, M = 256 cta_group::2 MMAs; b_bytes = half the N tile)
  int32_t dbg;               // BDBNN_TC_DBG experiment bits: 1 = no global stores, 2 = no TMEM loads, 4 = no MMAs
  uint32_t stage_bytes, b_bytes;
  int32_t fmt;               // BDBNN_FMT_* or -1 (fp8)
  int32_t row_bytes;         // bytes per pixel row of a K block: 128 (16-bit x 64 ch, fp8 x 128 ch) or 64 (fp8 x 64 ch)
  int32_t kb_elems;          // channels per K block
  const uint32_t* amax_bits;
  const float* add;
  const float* alpha;
  const uint32_t* mask;
  float* out;
  int16_t* out_i16;          // MODE 0: write the exact integer accumulator as int16 (y = alpha * int, |int| <= taps*Kc)
  double* bn_sums;           // MODE 0: per-channel sum / sum of squares of the result [2*Nout] (or NULL)
  uint32_t* bn_ymax;         // MODE 0: per-channel max|result| bits [Nout]
  // MODE 1 (dgrad whose result gx IS the gradient gz of the BatchNorm unit that produced this conv's input):
  // accumulate that unit's backward statistics here — bn_sums = [sum gz | sum gz*yhat], bn_ymax = max|gz| —
  // with yhat = (alpha*y_int - mean)*invstd read from the producer's int16 conv result (same pixel grid, Nout ch).
  const int16_t* st_y;
  const float* st_alpha;
  const float* st_mean;
  const float* st_invstd;
  long long* trace;          // optional clock64 trace of CTA 0 (bdbnn_debug_trace), else NULL
};

constexpr int kMaxStatCh = 512;   // channels the in-kernel BatchNorm statistics can hold per CTA

// role r (0 producer, 1 mma, 2 epilogue) appends (event id, clock) pairs to its 2048-entry lane.
#define BDBNN_TR(r, ev)                                                           \
  do {                                                                            \
    if (p.trace != nullptr && blockIdx.x == 0 && tr_n < 1023) {                   \
      p.trace[(r) * 2048 + 2 * tr_n] = (ev);                                      \
      p.trace[(r) * 2048 + 2 * tr_n + 1] = clock64();                             \
      ++tr_n;                                                                     \
    }                                                                             \
  } while (0)

struct SuperGeom {
  int n0, h0, ntl;  // first image, first output row, M tiles in use
};

__device__ __forceinline__ SuperGeom super_geom(const TcConv2Params& p, int sup) {
  SuperGeom g;
  if (p.halo) {
    if (p.HBNI > 1 || p.supers_per_img == 1) {
      g.n0 = sup * p.HBNI;
      g.h0 = 0;
      const int imgs = min(p.HBNI, p.NIMG - g.n0);
      g.ntl = (imgs * p.IB + kTileM - 1) / kTileM;
    } else {
      g.n0 = sup / p.supers_per_img;
      g.h0 = (sup - g.n0 * p.supers_per_img) * p.SH;
      const int rows = min(p.SH, p.OH - g.h0);
      g.ntl = (rows * p.PW + kTileM - 1) / kTileM;
    }
  } else {
    const int t0 = sup * p.TS;
    g.n0 = 0; g.h0 = 0;
    g.ntl = min(p.TS, p.n_mtiles - t0);
  }
  if (g.ntl > p.TS) g.ntl = p.TS;
  return g;
}

// CG = 1: one CTA per work item (super tile x N tile).  CG = 2: a CTA PAIR (2-CTA cluster) per TWO adjacent super
// tiles of the same N tile, executed as M = 256 tcgen05.mma.cta_group::2 instructions issued by the leader CTA:
// each CTA stages its own activation patch / boxes (A) and HALF of the weight tile (B rows rank*BN/2 ...), so
// per unit of work every SM fetches half the B bytes from shared memory — the measured limiter of the SS-mode
// MMAs (DESIGN.md §5 finding 3).  Barriers the MMA thread waits on live in the leader; the peer's TMA loads
// complete_tx on them (cta_group::2 TMA form) and its epilogue warps arrive on them through shared::cluster.
// BST (MODE 1 only): accumulate the producing unit's BatchNorm backward statistics in the epilogue (see params).
template <int MODE, int CG, bool BST = false>
__global__ void __launch_bounds__(kTc2Threads, 1)
tc_conv2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const TcConv2Params p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kMaxStages], empty_bar[kMaxStages];
  __shared__ __align__(8) uint64_t pfull_bar[2], pempty_bar[2];
  __shared__ __align__(8) uint64_t tfull_bar[2], tempty_bar[2];
  __shared__ uint32_t tmem_slot;
  __shared__ uint32_t tap_shift_rows[kMaxTaps];   // halo: row offset of tap i inside the patch
  // BatchNorm statistics of this CTA's output rows (MODE 0 with p.bn_sums), flushed once.  The warps' fp32 partials
  // meet in fp64, where their sum is exact while they span fewer than ~29 binary orders of magnitude, and otherwise
  // rounds in the last fp64 bits only: the order the atomics arrive in (and the order of the per-CTA fp64 atomics
  // below) then almost never reaches the fp32 mean / variance.  fp32 shared atomics changed those in the last bit
  // from run to run, and in a binarised network a last-bit difference flips signs downstream.
  constexpr bool kStats = MODE == 0 || BST;
  __shared__ double stat_sum[kStats ? kMaxStatCh : 1], stat_sq[kStats ? kMaxStatCh : 1];
  __shared__ uint32_t stat_max[kStats ? kMaxStatCh : 1];
  const bool do_stats = kStats && p.bn_sums != nullptr;   // MODE 0: statistics of y; MODE 1 (BST): backward statistics of gz
  if (do_stats)
    for (int i = threadIdx.x; i < p.Nout; i += blockDim.x) { stat_sum[i] = 0.0; stat_sq[i] = 0.0; stat_max[i] = 0u; }

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < p.n_taps)
    tap_shift_rows[threadIdx.x] = uint32_t((p.tap_dh[threadIdx.x] - p.dh_min) * p.PW +
                                           (p.tap_dw[threadIdx.x] - p.dw_min));
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t ring_base = smem_base + (p.halo ? 2u * p.patch_bytes : 0u);
  const int kb_total = p.n_kb * p.a_halves;
  const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;        // 0 = leader of the pair
  const int cta_w = int(blockIdx.x) / CG, n_ctas_w = int(gridDim.x) / CG;   // work-item walkers (CTAs or pairs)
  const int n_sup_w = (p.n_supers + CG - 1) / CG;                // super tiles (CG=2: pairs of them) to walk
  const int n_work = n_sup_w * p.n_ntiles;
  // super tile this CTA (r = rank) or its peer handles in work item w; a missing odd super is a clamped duplicate
  auto sup_of = [&](int w, uint32_t r) { const int sp = w / p.n_ntiles; return min(sp * CG + int(r), p.n_supers - 1); };
  auto is_dup = [&](int w, uint32_t r) { const int sp = w / p.n_ntiles; return sp * CG + int(r) >= p.n_supers; };

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&pfull_bar[s]), 1);
      mbar_init(smem_u32(&pempty_bar[s]), 1);
      mbar_init(smem_u32(&tfull_bar[s]), 1);
      mbar_init(smem_u32(&tempty_bar[s]), kEpiWarps * CG);   // one arrive per epilogue warp (of both CTAs)
    }
    fence_barrier_init();
  }
  if (warp == kEpiWarps && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
  }
  if (CG == 2) {
    // both CTAs of the pair are running and their barriers initialised before the pair-wide TMEM allocation and
    // before anything signals a peer barrier
    __syncthreads();
    cluster_sync_all();
  }
  if (warp == kEpiWarps + 1) {
    if (CG == 2) tmem_alloc_cg2(smem_u32(&tmem_slot), 512);
    else tmem_alloc(smem_u32(&tmem_slot), 512);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_slot;

  if (warp == kEpiWarps) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      uint32_t it = 0, pcount = 0;
      uint32_t stage = 0, phase = 0;          // ring position, advanced incrementally (this is one thread: no divisions
      int tr_n = 0;                           // by run-time values inside the loops)
      const uint32_t patch_tx = uint32_t(p.PW * p.PH * p.HBNI) * uint32_t(p.row_bytes);
      for (int w = cta_w; w < n_work; w += n_ctas_w) {
        const int nt = w % p.n_ntiles;
        const int sup = sup_of(w, rank);
        const SuperGeom g = super_geom(p, sup);
        const int ntl_peer = CG == 2 ? super_geom(p, sup_of(w, rank ^ 1u)).ntl : 0;
        const int nn0 = nt * p.BN + int(rank) * (p.BN / CG);        // this CTA's rows of the weight tile
        const int t0_n = p.halo ? 0 : (sup * p.TS) / p.tiles_h, t0_h = p.halo ? 0 : sup * p.TS - t0_n * p.tiles_h;
        for (int kb = 0; kb < kb_total; ++kb) {
          const int kbb = kb >= p.n_kb ? kb - p.n_kb : kb;
          if (p.halo) {
            const uint32_t pa = pcount & 1u;
            BDBNN_TR(0, 0);
            mbar_wait(smem_u32(&pempty_bar[pa]), ((pcount >> 1) & 1u) ^ 1u);
            BDBNN_TR(0, 1);
            const uint32_t pb = smem_u32(&pfull_bar[pa]);
            if (CG == 2) {
              if (rank == 0) mbar_expect_tx(pb, 2u * patch_tx);          // both CTAs' patches land on the leader's barrier
              tma_load_4d_cg2(smem_base + pa * p.patch_bytes, &tmA, mapa_shared(pb, 0), kb * p.kb_elems, p.dw_min,
                              g.h0 + p.dh_min, g.n0);
            } else {
              mbar_expect_tx(pb, patch_tx);
              tma_load_4d(smem_base + pa * p.patch_bytes, &tmA, pb, kb * p.kb_elems, p.dw_min, g.h0 + p.dh_min, g.n0);
            }
            ++pcount;
          }
          for (int ti = 0; ti < p.n_taps; ++ti, ++it, stage = stage + 1 == uint32_t(p.stages) ? (phase ^= 1u, 0u) : stage + 1) {
            mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
            const uint32_t fb_local = smem_u32(&full_bar[stage]);
            const uint32_t fb = CG == 2 ? mapa_shared(fb_local, 0) : fb_local;
            const uint32_t dst = ring_base + stage * p.stage_bytes;
            const uint32_t box_tx = uint32_t(p.BNI * p.BH * p.BW) * uint32_t(p.row_bytes);
            if (rank == 0) {
              uint32_t tx = p.b_bytes * uint32_t(CG);
              if (!p.halo) tx += uint32_t(g.ntl + ntl_peer) * box_tx;
              mbar_expect_tx(fb_local, tx);
            }
            if (!p.halo) {
              int tile_n = t0_n, tile_h = t0_h;              // tile sup * TS + j, advanced without dividing
              for (int j = 0; j < g.ntl; ++j, tile_h + 1 == p.tiles_h ? (tile_h = 0, ++tile_n) : ++tile_h) {
                const uint32_t d = dst + p.b_bytes + uint32_t(j) * (kTileM * uint32_t(p.row_bytes));
                if (CG == 2)
                  tma_load_4d_cg2(d, &tmA, fb, kb * p.kb_elems, p.tap_dw[ti], tile_h * p.BH * p.in_step + p.tap_dh[ti],
                                  tile_n * p.BNI);
                else
                  tma_load_4d(d, &tmA, fb, kb * p.kb_elems, p.tap_dw[ti], tile_h * p.BH * p.in_step + p.tap_dh[ti],
                              tile_n * p.BNI);
              }
            }
            if (CG == 2) tma_load_2d_cg2(dst, &tmB, fb, p.tap_b[ti] * p.Kc + kbb * p.kb_elems, nn0);
            else tma_load_2d(dst, &tmB, fb, p.tap_b[ti] * p.Kc + kbb * p.kb_elems, nn0);
          }
          BDBNN_TR(0, 2);
        }
      }
    }
  } else if (warp == kEpiWarps + 1) {
    // ================================ MMA issuer ================================
    if (lane == 0 && rank == 0) {
      const bool f8 = p.fmt < 0;
      const uint32_t idesc = f8 ? make_idesc_f8(kTileM * CG, uint32_t(p.BN))
                                : make_idesc_bf16(kTileM * CG, uint32_t(p.BN), uint32_t(p.fmt));
      const uint32_t desc_hi = kmajor_hi(uint32_t(p.row_bytes));
      const uint32_t row16 = uint32_t(p.row_bytes) >> 4;          // descriptor-address units per pixel row
      const int k_steps = p.row_bytes / 32;
      uint32_t it = 0, pcount = 0, wcount = 0;
      uint32_t stage = 0, phase = 0;
      int tr_n = 0;
      auto commit = [&](uint32_t bar) { if (CG == 2) umma_commit_cg2(bar); else umma_commit(bar); };
      for (int w = cta_w; w < n_work; w += n_ctas_w, ++wcount) {
        int ntl = super_geom(p, sup_of(w, 0)).ntl;
        if (CG == 2) ntl = max(ntl, super_geom(p, sup_of(w, 1)).ntl);   // the peer's extra tiles cost this CTA garbage MMAs
        const uint32_t buf = wcount % uint32_t(p.NB);
        BDBNN_TR(1, 0);
        mbar_wait(smem_u32(&tempty_bar[buf]), ((wcount / uint32_t(p.NB)) & 1u) ^ 1u);
        tc_fence_after();
        BDBNN_TR(1, 1);
        const uint32_t acc0 = tmem_d + buf * uint32_t(p.TS * p.BN);
        bool first = true;
        for (int kb = 0; kb < kb_total; ++kb) {
          uint32_t patch = 0, pa = 0;
          if (p.halo) {
            pa = pcount & 1u;
            mbar_wait(smem_u32(&pfull_bar[pa]), (pcount >> 1) & 1u);
            tc_fence_after();
            patch = smem_base + pa * p.patch_bytes;
            ++pcount;
            BDBNN_TR(1, 2);
          }
          for (int ti = 0; ti < p.n_taps; ++ti, ++it, stage = stage + 1 == uint32_t(p.stages) ? (phase ^= 1u, 0u) : stage + 1) {
            mbar_wait(smem_u32(&full_bar[stage]), phase);
            tc_fence_after();
            if (ti == 0) BDBNN_TR(1, 3);
            const uint32_t b_src = ring_base + stage * p.stage_bytes;
            const uint32_t b_lo = kmajor_lo(b_src);
            // the low descriptor word advances by row_bytes/16 per pixel row, 128 rows per M tile
            uint32_t a_lo = p.halo ? kmajor_lo(patch) + tap_shift_rows[ti] * row16 : kmajor_lo(b_src + p.b_bytes);
            uint32_t acc = acc0;
            if (!(p.dbg & 4)) {
              for (int j = 0; j < ntl; ++j, a_lo += kTileM * row16, acc += uint32_t(p.BN)) {
                if (CG == 2) {
                  for (int k = 0; k < k_steps; ++k) {
                    if (f8) umma_split_cg2<1>(acc, a_lo + 2u * k, desc_hi, b_lo + 2u * k, desc_hi, idesc, (!first || k > 0) ? 1u : 0u);
                    else    umma_split_cg2<0>(acc, a_lo + 2u * k, desc_hi, b_lo + 2u * k, desc_hi, idesc, (!first || k > 0) ? 1u : 0u);
                  }
                } else if (f8) {
                  for (int k = 0; k < k_steps; ++k)
                    umma_f8_split(acc, a_lo + 2u * k, desc_hi, b_lo + 2u * k, desc_hi, idesc, (!first || k > 0) ? 1u : 0u);
                } else if (p.row_bytes == 128) {
                  umma_bf16_k4(acc, a_lo, b_lo, desc_hi, idesc, first ? 0u : 1u);
                } else {
                  for (int k = 0; k < k_steps; ++k)
                    umma_bf16_split(acc, a_lo + 2u * k, desc_hi, b_lo + 2u * k, desc_hi, idesc, (!first || k > 0) ? 1u : 0u);
                }
              }
            }
            first = false;
            commit(smem_u32(&empty_bar[stage]));
          }
          if (p.halo) commit(smem_u32(&pempty_bar[pa]));
        }
        commit(smem_u32(&tfull_bar[buf]));
        BDBNN_TR(1, 4);
      }
    }
  } else {
    // ================================ epilogue (warps 0..7) ================================
    const int quad = warp & 3;        // TMEM lane quadrant = rows quad*32 .. quad*32+31 of every M tile
    const int grp = warp >> 2;        // column-block parity this warp handles
    const int mask_words = (p.Nout + 31) >> 5;
    const float post = p.amax_bits ? amax_pow2_scale(__ldg(p.amax_bits), true) : 1.0f;
    uint32_t wcount = 0;
    int tr_n = (threadIdx.x == 0) ? 0 : 100000;
    // 4 KB per-warp staging tile behind the TMA ring (generic-proxy only, never touched by TMA/UMMA)
    uint8_t* stage_warp = smem_raw + (ring_base - smem_u32(smem_raw)) + size_t(p.stages) * p.stage_bytes +
                          size_t(warp) * 4096;
    // BatchNorm statistics: each lane keeps (sum, sum of squares, max|.|) of the 4 channels it stores for
    // every 32-column block of the N tile, across tiles and work items, and flushes them to shared memory
    // only when the N tile changes or the CTA is done (per-block shuffles + atomics cost 25-35 % of the
    // forward kernels when done per 32x32 block).
    constexpr int kAcc = kStats ? 4 : 1;             // this group's 32-column blocks of the widest N tile (256)
    float4 acc_s[kAcc], acc_q[kAcc], acc_m[kAcc];
#pragma unroll
    for (int cb = 0; cb < kAcc; ++cb) acc_s[cb] = acc_q[cb] = acc_m[cb] = make_float4(0.f, 0.f, 0.f, 0.f);
    int acc_nn0 = -1;
    auto flush_stats = [&]() {
      if (!do_stats || acc_nn0 < 0) return;
#pragma unroll
      for (int ca = 0; ca < kAcc; ++ca) {
        const int cb = 2 * ca + grp;                   // the column block accumulator `ca` belongs to
        if (cb * 32 >= p.BN) break;
        float4 ss = acc_s[ca], sq = acc_q[ca], mx = acc_m[ca];
        // lanes cq, cq+8, cq+16, cq+24 hold the same 4 channels for different rows
#pragma unroll
        for (int d = 8; d <= 16; d <<= 1) {
          ss.x += __shfl_xor_sync(0xffffffffu, ss.x, d); ss.y += __shfl_xor_sync(0xffffffffu, ss.y, d);
          ss.z += __shfl_xor_sync(0xffffffffu, ss.z, d); ss.w += __shfl_xor_sync(0xffffffffu, ss.w, d);
          sq.x += __shfl_xor_sync(0xffffffffu, sq.x, d); sq.y += __shfl_xor_sync(0xffffffffu, sq.y, d);
          sq.z += __shfl_xor_sync(0xffffffffu, sq.z, d); sq.w += __shfl_xor_sync(0xffffffffu, sq.w, d);
          mx.x = fmaxf(mx.x, __shfl_xor_sync(0xffffffffu, mx.x, d)); mx.y = fmaxf(mx.y, __shfl_xor_sync(0xffffffffu, mx.y, d));
          mx.z = fmaxf(mx.z, __shfl_xor_sync(0xffffffffu, mx.z, d)); mx.w = fmaxf(mx.w, __shfl_xor_sync(0xffffffffu, mx.w, d));
        }
        if (lane < 8) {
          const int ch = acc_nn0 + cb * 32 + lane * 4;
          atomicAdd(&stat_sum[ch], double(ss.x)); atomicAdd(&stat_sum[ch + 1], double(ss.y));
          atomicAdd(&stat_sum[ch + 2], double(ss.z)); atomicAdd(&stat_sum[ch + 3], double(ss.w));
          atomicAdd(&stat_sq[ch], double(sq.x)); atomicAdd(&stat_sq[ch + 1], double(sq.y));
          atomicAdd(&stat_sq[ch + 2], double(sq.z)); atomicAdd(&stat_sq[ch + 3], double(sq.w));
          atomicMax(&stat_max[ch], __float_as_uint(mx.x)); atomicMax(&stat_max[ch + 1], __float_as_uint(mx.y));
          atomicMax(&stat_max[ch + 2], __float_as_uint(mx.z)); atomicMax(&stat_max[ch + 3], __float_as_uint(mx.w));
        }
        acc_s[ca] = acc_q[ca] = acc_m[ca] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    for (int w = cta_w; w < n_work; w += n_ctas_w, ++wcount) {
      const int nt = w % p.n_ntiles;
      const int sup = sup_of(w, rank);
      const bool dup = is_dup(w, rank);          // odd super-tile count: this CTA only shadows the leader's last item
      const SuperGeom g = super_geom(p, sup);
      const int nn0 = nt * p.BN;
      if (do_stats && nn0 != acc_nn0) {
        flush_stats();
        acc_nn0 = nn0;
      }
      const uint32_t buf = wcount % uint32_t(p.NB);
      BDBNN_TR(2, 0);
      mbar_wait(smem_u32(&tfull_bar[buf]), (wcount / uint32_t(p.NB)) & 1u);
      tc_fence_after();
      BDBNN_TR(2, 1);
      for (int j = 0; j < g.ntl; ++j) {
        const int m = j * kTileM + quad * 32 + lane;
        int ni, hi, wi;
        bool valid;
        if (p.halo) {
          const int blk = (p.HBNI > 1 || p.supers_per_img == 1) ? m / p.IB : 0;
          const int rem = m - blk * p.IB;
          hi = rem / p.PW;
          wi = rem - hi * p.PW;
          ni = g.n0 + blk;
          hi += g.h0;
          valid = wi < p.OW && hi < p.OH && ni < p.NIMG && blk < p.HBNI &&
                  (p.HBNI > 1 || p.supers_per_img == 1 || hi < g.h0 + p.SH);
        } else {
          const int t = sup * p.TS + j;
          const int tile_n = t / p.tiles_h, tile_h = t - tile_n * p.tiles_h;
          const int r = quad * 32 + lane;
          wi = r % p.BW;
          const int q = r / p.BW;
          hi = tile_h * p.BH + q % p.BH;
          const int nl = q / p.BH;
          ni = tile_n * p.BNI + nl;
          valid = nl < p.BNI && hi < p.OH && ni < p.NIMG;
        }
        const int oh = hi * p.out_step + p.out_off_h, ow = wi * p.out_step + p.out_off_w;
        valid = valid && oh < p.OHf && ow < p.OWf;
        const int64_t pix = (int64_t(ni) * p.OHf + oh) * p.OWf + ow;
        const uint32_t tbase = tmem_d + (uint32_t(quad * 32) << 16) + buf * uint32_t(p.TS * p.BN) + uint32_t(j * p.BN);
        if ((p.dbg & 1) || dup) valid = false;
        if (p.dbg & 2) continue;
        // Row offsets/validity of this warp's 32 rows are exchanged by shuffle in the store phase.
        const int64_t row_off = valid ? pix * p.Nout + nn0 : int64_t(-1);
#pragma unroll
        for (int ca = 0; ca < 4; ++ca) {
          const int cb = 2 * ca + grp;
          const int c0 = cb * 32;
          if (c0 >= p.BN) break;
          uint32_t v[32];
          tmem_ld32(tbase + uint32_t(c0), v);
          uint32_t word = 0;
          if (MODE == 1 && valid) word = __ldg(p.mask + pix * mask_words + ((nn0 + c0) >> 5));
          tmem_ld_wait();
          // (1) scale/mask and park the 32x32 fp32 block in this warp's swizzled staging tile:
          //     row r = lane, 16-byte chunk c at r*128 + ((c ^ (r&7)) * 16)  (4 wavefronts per STS.128)
          __syncwarp();
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const int q = c * 4;
            float4 o;
            if (MODE == 0) {
              if (p.out_i16 != nullptr) {      // raw integers; alpha is applied to the statistics only (below)
                o = make_float4(__uint_as_float(v[q]), __uint_as_float(v[q + 1]), __uint_as_float(v[q + 2]),
                                __uint_as_float(v[q + 3]));
              } else {
                const float4 a = __ldg(reinterpret_cast<const float4*>(p.alpha + nn0 + c0 + q));
                o = make_float4(__uint_as_float(v[q]) * a.x, __uint_as_float(v[q + 1]) * a.y,
                                __uint_as_float(v[q + 2]) * a.z, __uint_as_float(v[q + 3]) * a.w);
              }
            } else {
              o = make_float4(((word >> q) & 1u) ? __uint_as_float(v[q]) * post : 0.0f,
                              ((word >> (q + 1)) & 1u) ? __uint_as_float(v[q + 1]) * post : 0.0f,
                              ((word >> (q + 2)) & 1u) ? __uint_as_float(v[q + 2]) * post : 0.0f,
                              ((word >> (q + 3)) & 1u) ? __uint_as_float(v[q + 3]) * post : 0.0f);
            }
            *reinterpret_cast<float4*>(stage_warp + lane * 128 + ((c ^ (lane & 7)) << 4)) = o;
          }
          __syncwarp();
          // (2) read back transposed: one instruction stores 4 complete 128-byte rows (8 lanes per row).
          //     Row offsets come by shuffle; the optional additive tensor is fetched for all 8 row groups
          //     up front so its latency is paid once per block, not once per store.
          int64_t offs[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) offs[i] = __shfl_sync(0xffffffffu, row_off, 4 * i + (lane >> 3));
          const int cq = lane & 7;
          float4 a16 = make_float4(1.f, 1.f, 1.f, 1.f);
          if (MODE == 0 && p.out_i16 != nullptr)
            a16 = __ldg(reinterpret_cast<const float4*>(p.alpha + nn0 + c0 + cq * 4));
          float4 st_a = make_float4(0.f, 0.f, 0.f, 0.f), st_b = st_a;      // yhat = y_int * st_a - st_b
          if (BST && do_stats) {
            const int ch = nn0 + c0 + cq * 4;
            const float4 al = __ldg(reinterpret_cast<const float4*>(p.st_alpha + ch));
            const float4 mu = __ldg(reinterpret_cast<const float4*>(p.st_mean + ch));
            const float4 is = __ldg(reinterpret_cast<const float4*>(p.st_invstd + ch));
            st_a = make_float4(al.x * is.x, al.y * is.y, al.z * is.z, al.w * is.w);
            st_b = make_float4(mu.x * is.x, mu.y * is.y, mu.z * is.z, mu.w * is.w);
          }
          float4 addv[8];
          if (MODE == 1 && p.add != nullptr) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              addv[i] = offs[i] >= 0 ? *reinterpret_cast<const float4*>(p.add + offs[i] + c0 + cq * 4)   // may alias out
                                     : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          uint2 yv[BST ? 8 : 1];        // producer's y_int for the 8 row groups: all loads in flight before the stores
          if (BST && do_stats) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              yv[i] = offs[i] >= 0 ? __ldg(reinterpret_cast<const uint2*>(p.st_y + offs[i] + c0 + cq * 4)) : make_uint2(0u, 0u);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = 4 * i + (lane >> 3);
            float4 o = *reinterpret_cast<const float4*>(stage_warp + r * 128 + ((cq ^ (r & 7)) << 4));
            if (MODE == 1 && p.add != nullptr) {
              o.x += addv[i].x; o.y += addv[i].y; o.z += addv[i].z; o.w += addv[i].w;
            }
            if (offs[i] >= 0) {
              if (MODE == 0 && p.out_i16 != nullptr) {
                // exact: |o| <= 9 * 512 fits int16; 8 lanes write one 64-byte row segment
                uint2 pk;
                pk.x = (uint32_t(int(o.x)) & 0xffffu) | (uint32_t(int(o.y)) << 16);
                pk.y = (uint32_t(int(o.z)) & 0xffffu) | (uint32_t(int(o.w)) << 16);
                *reinterpret_cast<uint2*>(p.out_i16 + offs[i] + c0 + cq * 4) = pk;
                o.x *= a16.x; o.y *= a16.y; o.z *= a16.z; o.w *= a16.w;      // y = alpha * int for the statistics
              } else {
                *reinterpret_cast<float4*>(p.out + offs[i] + c0 + cq * 4) = o;
              }
              if (do_stats) {
                float4& ss = acc_s[kStats ? ca : 0]; float4& sq = acc_q[kStats ? ca : 0];
                float4& mx = acc_m[kStats ? ca : 0];
                ss.x += o.x; ss.y += o.y; ss.z += o.z; ss.w += o.w;
                if (BST) {            // sum gz * yhat of the producing BatchNorm unit
                  const uint2 yr = yv[BST ? i : 0];
                  sq.x += o.x * fmaf(float(int16_t(yr.x & 0xffffu)), st_a.x, -st_b.x);
                  sq.y += o.y * fmaf(float(int16_t(yr.x >> 16)), st_a.y, -st_b.y);
                  sq.z += o.z * fmaf(float(int16_t(yr.y & 0xffffu)), st_a.z, -st_b.z);
                  sq.w += o.w * fmaf(float(int16_t(yr.y >> 16)), st_a.w, -st_b.w);
                } else {
                sq.x += o.x * o.x; sq.y += o.y * o.y; sq.z += o.z * o.z; sq.w += o.w * o.w;
                }
                mx.x = fmaxf(mx.x, fabsf(o.x)); mx.y = fmaxf(mx.y, fabsf(o.y));
                mx.z = fmaxf(mx.z, fabsf(o.z)); mx.w = fmaxf(mx.w, fabsf(o.w));
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      BDBNN_TR(2, 2);
      if (lane == 0) {
        if (CG == 2) mbar_arrive_cluster(mapa_shared(smem_u32(&tempty_bar[buf]), 0));   // the leader's MMA thread waits
        else mbar_arrive(smem_u32(&tempty_bar[buf]));
      }
    }
    flush_stats();
  }
  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();          // nobody leaves (or frees TMEM) while the pair's MMAs / commits may be in flight
  if (do_stats) {
    // one fp64 atomic per channel per CTA; channels this CTA never touched hold zeros
    for (int i = threadIdx.x; i < p.Nout; i += blockDim.x) {
      if (stat_max[i] != 0u || stat_sum[i] != 0.0 || stat_sq[i] != 0.0) {
        atomicAdd(p.bn_sums + i, stat_sum[i]);
        atomicAdd(p.bn_sums + p.Nout + i, stat_sq[i]);
        atomicMax(p.bn_ymax + i, stat_max[i]);
      }
    }
  }
  if (warp == kEpiWarps + 1) {
    __syncwarp();
    tc_fence_after();
    if (CG == 2) tmem_dealloc_cg2(tmem_d, 512);
    else tmem_dealloc(tmem_d, 512);
  }
}

// Host-only planning probe (bdbnn_debug_conv_plan): when set, launch_tc_conv2 fills it with the tiling it
// chose and returns before creating tensor maps or touching CUDA.
thread_local int32_t* g_plan_sink = nullptr;
void set_conv_plan_sink(int32_t* sink) { g_plan_sink = sink; }

static long long* g_trace = nullptr;
void set_tc_trace(long long* buf) { g_trace = buf; }
long long* get_tc_trace() { return g_trace; }

// mode: 0 = alpha epilogue (forward), 1 = STE-mask epilogue (dgrad)
int launch_tc_conv2(const TcConvLaunch& L, int mode, cudaStream_t st) {
  if (L.n_taps <= 0) return BDBNN_ERR_UNSUPPORTED;
  if (L.win ? (L.Kc != 32 || L.fmt < 0) : (L.Kc % 64 != 0)) return BDBNN_ERR_UNSUPPORTED;
  const bool f8 = L.fmt < 0;
  const int esize = f8 ? 1 : 2;
  // K block: 64 16-bit channels (128-byte rows); fp8: 128 or 64 bytes; stem windows: 32 halves (64-byte rows)
  const int kb_elems = L.win ? 32 : (f8 ? (L.Kc % 128 == 0 ? 128 : 64) : 64);
  const uint32_t row_bytes = uint32_t(kb_elems * esize);
  if (L.Nout != 64 && L.Nout % 128 != 0) return BDBNN_ERR_UNSUPPORTED;
  TcConv2Params p;
  memset(&p, 0, sizeof(p));
  p.OW = L.OW; p.OH = L.OH; p.NIMG = L.NIMG;
  p.Kc = L.Kc; p.n_kb = L.Kc / kb_elems; p.a_halves = L.a_halves; p.in_step = L.in_step;
  p.row_bytes = int(row_bytes); p.kb_elems = kb_elems;
  p.n_taps = L.n_taps;
  memcpy(p.tap_dh, L.dh, sizeof(p.tap_dh));
  memcpy(p.tap_dw, L.dw, sizeof(p.tap_dw));
  memcpy(p.tap_b, L.tb, sizeof(p.tap_b));
  p.out_step = L.out_step; p.out_off_h = L.off_h; p.out_off_w = L.off_w; p.OHf = L.OHf; p.OWf = L.OWf;
  p.Nout = L.Nout;
  // dgrad of the wide layers (Nout = Cin >= 256): 256-wide N tiles — per K step the two M tiles fetch
  // 2 x (4 KB A + 8 KB B) from shared memory instead of 4 x (4 + 4) KB for the same work (SS-mode MMAs are
  // bound by that fetch, DESIGN.md section 5 finding 3).  BDBNN_TC_BN256=0 restores 128.
  static const int bn256 = [] { const char* e = getenv("BDBNN_TC_BN256"); return e ? atoi(e) : 3; }();   // 1 dgrad, 2 fwd8, 3 both (default)
  // forward: the fp8 layers with Cout >= 256 (bit 1 of the knob)
  // CTA pairs (cta_group::2): each CTA stages half of the N tile, so the widest tile (256) costs a CTA what a
  // 128-wide one costs alone — use it whenever the channel count allows.  BDBNN_TC_CG2=0: single-CTA MMAs.
  // Measured on B200 (profiles/r2_cg2_ablation.txt): correct, but a pair MMA costs more than two independent ones
  // on these shapes (layer1 N=64: MMA pipeline 193 us vs 150 us; layer3 dgrad N=256: 82 vs 68 us) -> default off.
  static const int cg2_env = [] { const char* e = getenv("BDBNN_TC_CG2"); return e ? atoi(e) : 0; }();
  p.cg = cg2_env ? 2 : 1;
  const bool wide = L.Nout % 256 == 0 && (p.cg == 2 || (mode == 1 && !f8 && (bn256 & 1)) || (mode == 0 && f8 && (bn256 & 2)));
  p.BN = wide ? 256 : (L.Nout >= 128 ? 128 : 64);
  p.n_ntiles = L.Nout / p.BN;
  // 512 TMEM columns = NB buffers x TS accumulators x BN columns.  BDBNN_TC_TS128 picks the BN=128 split:
  // 4 = four tiles sharing each weight stage, single buffer (epilogue exposed);
  // 2 = two tiles, double-buffered (epilogue overlaps the next item's MMAs, weights re-read twice as often)
  // Measured (ResNet-18 N=256): TS=2 wins while the weight slab per item is small (K <= 128 channels:
  // layer2 fwd 0.109 -> 0.097 ms, stride-2 fwd 0.081 -> 0.058), TS=4 wins for K >= 256 (layers 3, 4).
  static const int ts128 = [] { const char* e = getenv("BDBNN_TC_TS128"); return e ? atoi(e) : 0; }();
  const int ts_auto = (L.Kc * L.a_halves <= 128) ? 2 : 4;
  // 256-wide N tiles: ONE M tile per work item and two accumulator buffers (BDBNN_TC_TS256=2: two tiles, one buffer).
  // The 14x14 / 7x7 layers have 128-196 two-tile items for 148 CTAs — one item per CTA, nothing to overlap its
  // epilogue with (ncu: epilogue warps 59 % of the samples waiting for the accumulator, producer / MMA warps done
  // early); with one-tile items a CTA's second item runs under the first one's epilogue: dgrad 2.08 -> 2.00 ms per
  // step at twice the weight traffic per pixel (forward unchanged).
  static const int ts256 = [] { const char* e = getenv("BDBNN_TC_TS256"); return e ? atoi(e) : 1; }();
  p.TS = p.BN == 256 ? (ts256 == 1 ? 1 : 2) : (p.BN == 64 ? 4 : (ts128 == 4 ? 4 : (ts128 == 2 ? 2 : ts_auto)));
  p.NB = 512 / (p.TS * p.BN);
  p.alpha = L.alpha; p.mask = L.mask; p.out = L.out;
  p.out_i16 = mode == 0 ? L.out_i16 : nullptr;
  if (L.out_i16 && (mode != 0 || L.n_taps * L.Kc * L.a_halves > 32767)) return BDBNN_ERR_UNSUPPORTED;
  p.fmt = L.fmt; p.amax_bits = L.amax_bits; p.add = L.add;
  p.bn_sums = L.Nout <= kMaxStatCh ? L.bn_sums : nullptr;
  p.bn_ymax = L.bn_ymax;
  if (L.bn_sums && !p.bn_sums) return BDBNN_ERR_UNSUPPORTED;
  p.st_y = L.st_y; p.st_alpha = L.st_alpha; p.st_mean = L.st_mean; p.st_invstd = L.st_invstd;
  if (mode == 1 && L.bn_sums && !(L.st_y && L.st_alpha && L.st_mean && L.st_invstd && L.out_step == 1))
    return BDBNN_ERR_UNSUPPORTED;
  p.b_bytes = uint32_t(p.BN / p.cg) * row_bytes;       // rows of the weight tile THIS CTA stages

  int dh0 = 127, dh1 = -127, dw0 = 127, dw1 = -127;
  for (int i = 0; i < p.n_taps; ++i) {
    dh0 = min(dh0, int(p.tap_dh[i])); dh1 = max(dh1, int(p.tap_dh[i]));
    dw0 = min(dw0, int(p.tap_dw[i])); dw1 = max(dw1, int(p.tap_dw[i]));
  }
  const int dh_span = dh1 - dh0, dw_span = dw1 - dw0;
  // BDBNN_TC_PW8=1 (experiment): pad the patch width to a multiple of 8 pixel rows so that the dh row shifts of
  // the tap views stay aligned to the 8-row swizzle atoms
  static const int pw8_env = [] { const char* e = getenv("BDBNN_TC_PW8"); return e ? atoi(e) : 0; }();
  int PW = L.OW + dw_span;
  if (pw8_env && !L.win) PW = (PW + 7) & ~7;
  const int super_rows = p.TS * kTileM;  // padded rows per super tile
  CUtensorMap tmA, tmB;
  int rc;
  // BDBNN_TC_HALO_SMALL=1 (experimental, off): halo patches also for images of <= 128 pixels (several whole
  // images per super tile).  The 7x7 layers then fetch one patch per K block instead of one box per tap
  // (box mode: 2.3 MB of activation traffic per work item against 0.6 MB of weights), at 57 % instead of
  // 77 % row utilisation; to be measured.
  static const int halo_small = [] { const char* e = getenv("BDBNN_TC_HALO_SMALL"); return e ? atoi(e) : 0; }();
  if (L.in_step == 1 && (L.OH * L.OW > kTileM || (halo_small && !L.win && L.OH * L.OW >= 16)) && PW <= 256 &&
      PW * (1 + dh_span) <= super_rows) {
    p.halo = 1;
    p.PW = PW; p.dh_min = dh0; p.dw_min = dw0;
    const int img_block = (L.OH + dh_span) * PW;      // whole image incl. halo rows, padded raster
    if (img_block <= super_rows) {
      p.HBNI = super_rows / img_block;
      if (p.HBNI > L.NIMG) p.HBNI = L.NIMG;
      if (p.HBNI > 256) p.HBNI = 256;
      p.IB = img_block; p.SH = L.OH; p.PH = L.OH + dh_span; p.supers_per_img = 1;
      p.n_supers = (L.NIMG + p.HBNI - 1) / p.HBNI;
    } else {
      p.HBNI = 1;
      p.SH = super_rows / PW;
      if (p.SH > 256 - dh_span) p.SH = 256 - dh_span;
      p.PH = p.SH + dh_span;
      p.IB = super_rows;                               // single block: m / IB == 0 for every row
      p.supers_per_img = (L.OH + p.SH - 1) / p.SH;
      if (p.supers_per_img == 1) { p.IB = p.PH * PW > super_rows ? p.PH * PW : super_rows; }
      p.n_supers = L.NIMG * p.supers_per_img;
    }
    const uint32_t rows = uint32_t(super_rows + dh_span * PW + dw_span);
    p.patch_bytes = (rows * row_bytes + 1023u) & ~1023u;
    if (uint32_t(p.PW * p.PH * p.HBNI) * row_bytes > p.patch_bytes) return BDBNN_ERR_UNSUPPORTED;
    p.stage_bytes = (p.b_bytes + 1023u) & ~1023u;
    rc = g_plan_sink ? BDBNN_OK
                     : make_act_map(&tmA, L.A, L.NIMG, L.IH, L.IW, L.Kc * L.a_halves, kb_elems, p.PW, p.PH, p.HBNI, 1, esize);
  } else {
    p.halo = 0;
    p.BW = L.OW;
    if (L.OW > kTileM) return BDBNN_ERR_UNSUPPORTED;
    if (L.OH * L.OW <= kTileM) {
      p.BH = L.OH;
      p.BNI = kTileM / (L.OH * L.OW);
      if (p.BNI > L.NIMG) p.BNI = L.NIMG;
      if (p.BNI > 256) p.BNI = 256;
    } else {
      p.BH = kTileM / L.OW;
      p.BNI = 1;
    }
    p.tiles_h = (L.OH + p.BH - 1) / p.BH;
    p.n_mtiles = p.tiles_h * ((L.NIMG + p.BNI - 1) / p.BNI);
    p.n_supers = (p.n_mtiles + p.TS - 1) / p.TS;
    p.stage_bytes = (p.b_bytes + uint32_t(p.TS) * kTileM * row_bytes + 1023u) & ~1023u;
    if (g_plan_sink)
      rc = BDBNN_OK;
    else if (L.win)
      rc = make_window_map(&tmA, L.A, L.NIMG, L.IH, L.IW, kb_elems, L.win_stride, L.win_row_stride, L.win_img_stride,
                           p.BW, p.BH, p.BNI, L.in_step);
    else
      rc = make_act_map(&tmA, L.A, L.NIMG, L.IH, L.IW, L.Kc * L.a_halves, kb_elems, p.BW, p.BH, p.BNI, L.in_step, esize);
  }
  if (rc) return rc;
  rc = g_plan_sink ? BDBNN_OK : make_weight_map(&tmB, L.B, L.Nout, L.b_taps * L.Kc, kb_elems, p.BN / p.cg, esize);
  if (rc) return rc;
  const uint32_t kStaging = uint32_t(kEpiWarps) * 4096u;   // epilogue transpose tiles
  const uint32_t fixed = (p.halo ? 2u * p.patch_bytes : 0u) + kStaging;
  // 227 KB per CTA minus static shared memory (barriers; MODE 0 also holds 10 KB of BN statistics)
  const bool bst = mode == 1 && p.bn_sums != nullptr;
  const uint32_t budget = 224u * 1024u - 1024u - ((mode == 0 || bst) ? (2u * 8u + 4u) * kMaxStatCh : 0u);
  if (fixed + 2u * p.stage_bytes > budget) return BDBNN_ERR_UNSUPPORTED;
  int stages = int((budget - fixed) / p.stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  p.stages = stages;
  const size_t smem = size_t(fixed) + size_t(stages) * p.stage_bytes + 1024;
  static const int dbg_env = [] { const char* e = getenv("BDBNN_TC_DBG"); return e ? atoi(e) : 0; }();
  p.dbg = dbg_env;
  p.trace = g_trace;
  const int n_work = ((p.n_supers + p.cg - 1) / p.cg) * p.n_ntiles;      // work items of a CTA (pair)
  int grid = num_sms() / p.cg;
  if (grid > n_work) grid = n_work;
  grid *= p.cg;
  if (g_plan_sink) {
    const int32_t v[12] = {1, p.halo, p.TS, p.NB, p.BN, p.n_ntiles, p.n_supers, stages, int32_t(smem), grid,
                           int32_t(p.stage_bytes), int32_t(p.halo ? p.patch_bytes : 0)};
    memcpy(g_plan_sink, v, sizeof(v));
    return BDBNN_OK;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(unsigned(grid)); cfg.blockDim = dim3(kTc2Threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = unsigned(p.cg); attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  auto launch = [&](auto kern) -> int {
    BDBNN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    BDBNN_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, p));
    return BDBNN_OK;
  };
  if (mode == 0) rc = p.cg == 2 ? launch(tc_conv2_kernel<0, 2>) : launch(tc_conv2_kernel<0, 1>);
  else if (bst)  rc = p.cg == 2 ? launch(tc_conv2_kernel<1, 2, true>) : launch(tc_conv2_kernel<1, 1, true>);
  else           rc = p.cg == 2 ? launch(tc_conv2_kernel<1, 2>) : launch(tc_conv2_kernel<1, 1>);
  if (rc) return rc;
  return check_launch("tc_conv2_kernel");
}

}  // namespace bdbnn
