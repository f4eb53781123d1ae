// Implicit-GEMM convolution / linear / dgrad / wgrad on Blackwell tensor cores.
//
//   fprop : D[pixel, co]   = sum_{tap, ci}  X[pixel + tap, ci] * Wp[co, tap, ci]
//           A = X  tile, TMA 4-D box (64 ch, tw, th, nb) over NHWC   -> smem [128 px][64 ch], K-major, SWIZZLE_128B
//           B = Wp tile, TMA 3-D box (64 ci, 1 tap, BN co)           -> smem [BN co][64 ci],  K-major, SWIZZLE_128B
//           padding = TMA out-of-bounds zero fill (negative / overflowing box coordinates).
//   wgrad : D[co, ci]      = sum_{pixel}    dY[pixel, co] * X[pixel + tap, ci]           (one tap per work item)
//           A = dY tile(s), B = X tile(s): same boxes, consumed as MN-major operands (the pixel axis is K).
//
// One persistent CTA per SM, 6 warps: warp 0 = TMA producer (one lane), warp 1 = tcgen05.mma issuer (one lane) and
// TMEM owner, warps 2..5 = epilogue (TMEM -> registers -> fused epilogue -> global).  Two TMEM accumulator stages so
// the epilogue of tile i overlaps the main loop of tile i+1.
#include "common.cuh"
#include "ptx.cuh"
#include "conv_epilogue.cuh"

namespace sgb {

static constexpr int kWgradThreads = 192;                // wgrad: warps 0 producer, 1 MMA, 2..5 epilogue
static constexpr int kThreads = 128 + kEpiThreads;       // warps 0..3: producer / MMA / aux producer / (idle), warps 4..11: epilogue teams
static constexpr int kTileM = 128;          // pixels (fprop) or output channels (wgrad) per tile = TMEM lanes
static constexpr int kBlockK = 64;          // bf16 elements per 128-byte swizzle row
static constexpr int kABytes = kTileM * kBlockK * 2;  // 16 KiB

struct FpropArgs {
  int B, H, W, Cin, Cout, taps, KW, pad_h, pad_w;
  int tw, th, nb;                 // tile box: tw*th*nb == 128
  int tiles_w, tiles_h, tiles_b, tiles_n, num_tiles;
  int kblocks;                    // ceil(Cin / 64)
  int BN;                         // output-channel tile (multiple of 16, <= 256)
  int w_mode;                     // 0: shared weights [Cout][taps][Cin]; 1: per-image [B][N][K]; 2: per-image MN-major [B][K][N]
  int stages;
  int use_tma;                    // epilogue through staging tiles + TMA tensor stores
  int epi_nbuf;                   // staging tiles per epilogue team (2: a store overlaps the next chunk's conversion)
  int b_resident;                 // 1: every weight tile of this CTA's channel tile stays in shared memory (loaded once)
  int aux_kind, aux_tw, aux_th;   // residual (1) / mask (2) tile staged by TMA; its box is aux_tw x aux_th x nb pixels
  int aux_depth;                  // aux tiles per epilogue team (ring filled by the aux producer warp)
  int out_sub;                    // 2: store only even (h, w) outputs at (h/2, w/2) -> stride-2 convolution (Inception reduction blocks)
  uint32_t tmem_cols;
  EpiArgs e;
};

template <int F>      // epilogue variant (conv_epilogue.cuh: kEpi* bits fixed at compile time; -1 = run-time flags)
__global__ void __launch_bounds__(kThreads, 1)
conv_fprop_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmAux, const FpropArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t epi_stage_base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // two 16 KiB staging tiles when use_tma
  const uint32_t aux_stage_base = epi_stage_base + (p.use_tma ? 2u * p.epi_nbuf * kEpiStageBytes : 0u);   // + two aux tiles when aux_kind
  const uint32_t b_bytes = (uint32_t)p.BN * kBlockK * 2;  // same size for K-major [BN][64] and MN-major (BN/64) x [64][64]
  const uint32_t bres_base = aux_stage_base + (p.aux_kind ? 2u * p.aux_depth * kEpiStageBytes : 0u);     // resident weight tiles [tap][kb]
  const uint32_t smem_base = bres_base + (p.b_resident ? (uint32_t)(p.taps * p.kblocks) * b_bytes : 0u);
  const uint32_t stage_bytes = kABytes + (p.b_resident ? 0u : b_bytes);  // multiple of 1024 because BN % 8 == 0 -> b_bytes % 1024 == 0
  const uint32_t bar_base = smem_base + (uint32_t)p.stages * stage_bytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (p.stages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * p.stages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * p.stages + 2 + a); };
  const uint32_t holder = bar_base + 8u * (2 * p.stages + 4);
  const uint32_t bres_bar = bar_base + 8u * (2 * p.stages + 6);
  auto aux_full = [&](int team, int slot) { return bar_base + 8u * (2 * p.stages + 8 + team * p.aux_depth + slot); };
  auto aux_empty = [&](int team, int slot) { return bar_base + 8u * (2 * p.stages + 8 + (2 + team) * p.aux_depth + slot); };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), kEpiThreads);
      for (int sl = 0; sl < p.aux_depth; ++sl) { mbar_init(aux_full(a, sl), 1); mbar_init(aux_empty(a, sl), 1); }
    }
    mbar_init(bres_bar, 1);
    fence_barrier_init();
    if (p.use_tma) tma_prefetch_desc(&tmY);
  }
  if (warp == 1) {
    tmem_alloc(holder, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(holder));

  const int kiters = p.taps * p.kblocks;

  if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------- TMA producer
      uint32_t it = 0;
      if (p.b_resident) {       // tiles_n == 1: the whole (small) filter is fetched once per CTA instead of once per tile
        mbar_arrive_expect_tx(bres_bar, (uint32_t)(p.taps * p.kblocks) * b_bytes);
        for (int tap = 0; tap < p.taps; ++tap)
          for (int kb = 0; kb < p.kblocks; ++kb)
            tma_load_3d(bres_base + (uint32_t)(tap * p.kblocks + kb) * b_bytes, &tmB, bres_bar, kb * kBlockK, tap, 0);
      }
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        int t = tile;
        const int nt = t % p.tiles_n; t /= p.tiles_n;
        const int wt = t % p.tiles_w; t /= p.tiles_w;
        const int ht = t % p.tiles_h; t /= p.tiles_h;
        const int bt = t;
        const int n0 = nt * p.BN, w0 = wt * p.tw, h0 = ht * p.th, b0 = bt * p.nb;
        for (int tap = 0; tap < p.taps; ++tap) {
          const int dh = tap / p.KW - p.pad_h, dw = tap % p.KW - p.pad_w;
          for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
            const int s = it % p.stages;
            const uint32_t ph = (it / p.stages) & 1;
            mbar_wait(empty_bar(s), ph ^ 1);
            mbar_arrive_expect_tx(full_bar(s), stage_bytes);
            const uint32_t sa = smem_base + s * stage_bytes;
            tma_load_4d(sa, &tmA, full_bar(s), kb * kBlockK, w0 + dw, h0 + dh, b0);
            if (p.b_resident) {
            } else if (p.w_mode == 0) {
              tma_load_3d(sa + kABytes, &tmB, full_bar(s), kb * kBlockK, tap, n0);
            } else if (p.w_mode == 1) {
              tma_load_3d(sa + kABytes, &tmB, full_bar(s), kb * kBlockK, b0, n0);
            } else {
              for (int j = 0; j < p.BN / 64; ++j)
                tma_load_3d(sa + kABytes + j * 8192, &tmB, full_bar(s), n0 + j * 64, kb * kBlockK, b0);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ------------------------------------------------------------- MMA issuer
      const bool b_mn = (p.w_mode == 2);
      const uint32_t idesc = make_idesc_bf16(kTileM, p.BN, 0, b_mn ? 1 : 0);
      uint32_t it = 0, tcount = 0;
      if (p.b_resident) { mbar_wait(bres_bar, 0); tc_fence_after(); }
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++tcount) {
        const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
        mbar_wait(tempty_bar(a), aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + a * p.BN;
        for (int k = 0; k < kiters; ++k, ++it) {
          const int s = it % p.stages;
          const uint32_t ph = (it / p.stages) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t sa = smem_base + s * stage_bytes;
          const uint64_t adesc = make_sdesc_sw128(sa, 16, 1024);
          // K-major B: rows = output channels, +32 B per 16-wide K step.
          // MN-major B: (BN/64) atoms of [64 k-rows][64 n] 8 KiB apart (LBO), 8-row groups 1 KiB apart (SBO), +2 KiB per K step.
          const uint32_t sb = p.b_resident ? bres_base + (uint32_t)k * b_bytes : sa + kABytes;     // k = tap * kblocks + kb
          const uint64_t bdesc = b_mn ? make_sdesc_sw128(sb, 8192, 1024) : make_sdesc_sw128(sb, 16, 1024);
          const uint32_t bstep = b_mn ? 128u : 2u;
#pragma unroll
          for (int kk = 0; kk < kBlockK / 16; ++kk) {
            // A: advance 16 bf16 = 32 bytes along K inside the swizzle row: +2 in the (addr >> 4) field
            umma_f16_ss(d_tmem, adesc + 2 * kk, bdesc + bstep * kk, idesc, (k > 0 || kk > 0) ? 1u : 0u);
          }
          umma_commit(empty_bar(s));  // smem slot reusable once these MMAs retire
        }
        umma_commit(tfull_bar(a));    // accumulator complete
      }
    }
  } else if (warp == 2) {
    if (lane == 0 && p.aux_kind) {
      // ------------------------------------------------------------- aux producer: residual / mask boxes, in the order the
      // two epilogue teams consume their chunks (team = chunk & 1), up to aux_depth boxes ahead per team
      const bool half = p.aux_kind == 1 && p.e.res_up2;
      const uint32_t bytes = (uint32_t)(p.aux_tw * p.aux_th * p.nb) * 128u;
      uint32_t cnt[2] = {0u, 0u};
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        int t = tile;
        const int nt = t % p.tiles_n; t /= p.tiles_n;
        const int wt = t % p.tiles_w; t /= p.tiles_w;
        const int ht = t % p.tiles_h; t /= p.tiles_h;
        const int c1 = half ? (wt * p.tw) >> 1 : wt * p.tw, c2 = half ? (ht * p.th) >> 1 : ht * p.th, c3 = t * p.nb;
        for (int cc = 0; cc * 64 < p.BN; ++cc) {
          const int nbase = nt * p.BN + cc * 64;
          if (nbase >= p.e.Cout) break;
          const int team = cc & 1;
          const uint32_t slot = cnt[team] % (uint32_t)p.aux_depth;
          mbar_wait(aux_empty(team, slot), ((cnt[team] / (uint32_t)p.aux_depth) & 1u) ^ 1u);
          mbar_arrive_expect_tx(aux_full(team, slot), bytes);
          tma_load_4d(aux_stage_base + (uint32_t)(team * p.aux_depth + slot) * kEpiStageBytes, &tmAux, aux_full(team, slot), nbase, c1, c2, c3);
          ++cnt[team];
        }
      }
    }
  } else if (warp >= 4) {
    // --------------------------------------------------------------- epilogue: 8 warps, TMEM lane quadrant = warp % 4;
    // team = which 64-channel chunks (even / odd)
    const int q = warp & 3;
    const int team = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const bool leader = (q == 0) && (lane == 0);
    const int wi = row % p.tw, hi = (row / p.tw) % p.th, bi = row / (p.tw * p.th);
    const bool vec_ok = epi_vec_ok(p.e);
    const float alpha = p.e.alpha_ptr ? p.e.alpha * __ldg(p.e.alpha_ptr) : p.e.alpha;
    const uint32_t stage = epi_stage_base + team * p.epi_nbuf * kEpiStageBytes;
    uint32_t aux_cnt = 0, sbuf = 0;
    EpiAux aux;
    aux.kind = p.aux_kind; aux.ring = aux_stage_base + (uint32_t)(team * p.aux_depth) * kEpiStageBytes;
    aux.full0 = aux_full(team, 0); aux.empty0 = aux_empty(team, 0); aux.depth = p.aux_depth; aux.cnt = &aux_cnt;
    const bool aux_half = p.aux_kind == 1 && p.e.res_up2;
    aux.arow = aux_half ? ((bi * p.aux_th + (p.aux_th == p.th ? hi : (hi >> 1))) * p.aux_tw + (wi >> 1)) : row;
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++tcount) {
      int t = tile;
      const int nt = t % p.tiles_n; t /= p.tiles_n;
      const int wt = t % p.tiles_w; t /= p.tiles_w;
      const int ht = t % p.tiles_h; t /= p.tiles_h;
      const int bt = t;
      const int n0 = nt * p.BN;
      const int w = wt * p.tw + wi, h = ht * p.th + hi, b = bt * p.nb + bi;
      const bool valid = (w < p.W) && (h < p.H) && (b < p.B) && (p.out_sub == 1 || (((w | h) & 1) == 0));
      const long long pix = p.out_sub == 1 ? ((long long)b * p.H + h) * p.W + w
                                           : ((long long)b * ((p.H + 1) >> 1) + (h >> 1)) * ((p.W + 1) >> 1) + (w >> 1);
      const long long rpix = p.e.res_up2 ? (((long long)b * (p.H >> 1) + (h >> 1)) * (p.W >> 1) + (w >> 1)) : pix;

      const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
      mbar_wait(tfull_bar(a), aph);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + a * p.BN;
      if constexpr (F >= 0 && (F & kEpiSmStats) != 0) {
        epilogue_tile_smstats(p.e, t_row, p.BN, n0, valid, pix, alpha, team, nt * 2 + team);
      } else if (F >= 0 || p.use_tma) {          // (the host picks a compile-time variant only for staged stores)
        epilogue_tile_tma<F>(p.e, &tmY, t_row, p.BN, n0, wt * p.tw, ht * p.th, bt * p.nb, valid, pix, rpix, alpha, stage, team, row,
                             leader, 2, p.aux_kind ? &aux : nullptr, p.epi_nbuf == 2 ? &sbuf : nullptr);
      } else if (team == 0) {
        epilogue_row<F>(p.e, t_row, p.BN, n0, valid, pix, rpix, alpha, vec_ok);
      }
      tc_fence_before();
      mbar_arrive(tempty_bar(a));
    }
    if (p.use_tma && leader) bulk_wait_all();   // staging tiles must outlive the last tensor store
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------ wgrad
struct WgradArgs {
  int B, H, W, Cin, Cout, taps, KW, pad_h, pad_w;
  int tw, th, nb;
  int tiles_w, tiles_h, tiles_b, pix_tiles;  // pix_tiles = tiles_w*tiles_h*tiles_b
  int tiles_m, tiles_n;                      // over Cout (128) and Cin (BN)
  int BN;                                    // 64 or 128 (input-channel tile)
  int groups, tiles_per_group;               // independent pixel groups (1, or B for per-image outputs)
  int splits, tiles_per_split;               // K-splits inside a group
  int num_items;                             // tiles_m*tiles_n*taps*groups*splits
  int stages;
  uint32_t tmem_cols;
  float* dw;
  long long dw_group_stride;
  float* dbias;                              // optional: sum over pixels of dy (bias gradient), from a constant-ones B operand
};

__global__ void __launch_bounds__(kWgradThreads, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap tmDY, const __grid_constant__ CUtensorMap tmX, const WgradArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t ones_base = (smem_u32(smem_raw) + 1023u) & ~1023u;          // 16 KiB of bf16 1.0 when dbias (any swizzle of ones is ones)
  const uint32_t smem_base = ones_base + (p.dbias ? (uint32_t)kABytes : 0u);
  const uint32_t a_bytes = 2 * kABytes;                       // two 64-channel boxes -> M = 128
  const uint32_t b_bytes = (uint32_t)(p.BN / 64) * kABytes;   // BN/64 boxes
  const uint32_t stage_bytes = a_bytes + b_bytes;
  const uint32_t bar_base = smem_base + (uint32_t)p.stages * stage_bytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (p.stages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * p.stages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * p.stages + 2 + a); };
  const uint32_t holder = bar_base + 8u * (2 * p.stages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (p.dbias) {
    for (uint32_t i = threadIdx.x; i < (uint32_t)kABytes / 16u; i += kWgradThreads)
      st_shared_v4(ones_base + i * 16u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    fence_proxy_async_smem();                 // generic-proxy writes -> visible to the tensor core's operand reads
  }
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmDY);
    tma_prefetch_desc(&tmX);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(holder, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(holder));

  // work item -> (m tile, n tile, tap, split); n fastest so neighbouring CTAs share the dY tiles in L2
  auto decode = [&](int item, int& mt, int& nt, int& tap, int& grp, int& pt_begin, int& pt_end) {
    int t = item;
    nt = t % p.tiles_n; t /= p.tiles_n;
    tap = t % p.taps; t /= p.taps;
    mt = t % p.tiles_m; t /= p.tiles_m;
    const int sp = t % p.splits; t /= p.splits;
    grp = t;
    const int g0 = grp * p.tiles_per_group;
    pt_begin = g0 + sp * p.tiles_per_split;
    pt_end = min(pt_begin + p.tiles_per_split, g0 + p.tiles_per_group);
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (int item = blockIdx.x; item < p.num_items; item += gridDim.x) {
        int mt, nt, tap, grp, pb, pe;
        decode(item, mt, nt, tap, grp, pb, pe);
        const int dh = tap / p.KW - p.pad_h, dw = tap % p.KW - p.pad_w;
        for (int pt = pb; pt < pe; ++pt, ++it) {
          int t = pt;
          const int wt = t % p.tiles_w; t /= p.tiles_w;
          const int ht = t % p.tiles_h; t /= p.tiles_h;
          const int bt = t;
          const int w0 = wt * p.tw, h0 = ht * p.th, b0 = bt * p.nb;
          const int s = it % p.stages;
          const uint32_t ph = (it / p.stages) & 1;
          mbar_wait(empty_bar(s), ph ^ 1);
          mbar_arrive_expect_tx(full_bar(s), stage_bytes);
          const uint32_t sa = smem_base + s * stage_bytes;
          tma_load_4d(sa, &tmDY, full_bar(s), mt * 128, w0, h0, b0);
          tma_load_4d(sa + kABytes, &tmDY, full_bar(s), mt * 128 + 64, w0, h0, b0);
          for (int j = 0; j < p.BN / 64; ++j)
            tma_load_4d(sa + a_bytes + j * kABytes, &tmX, full_bar(s), nt * p.BN + j * 64, w0 + dw, h0 + dh, b0);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(kTileM, p.BN, 1, 1);  // both operands MN-major
      const uint32_t idesc_ones = make_idesc_bf16(kTileM, 16, 1, 1);
      const uint64_t ones_desc = make_sdesc_sw128(ones_base, kABytes, 1024);
      uint32_t it = 0, tcount = 0;
      for (int item = blockIdx.x; item < p.num_items; item += gridDim.x, ++tcount) {
        int mt, nt, tap, grp, pb, pe;
        decode(item, mt, nt, tap, grp, pb, pe);
        const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
        mbar_wait(tempty_bar(a), aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + a * p.BN;
        // bias gradient: the (first input-channel tile, first tap) items also multiply dY^T by a block of ones
        const bool with_bias = p.dbias != nullptr && nt == 0 && tap == 0;
        const uint32_t d_bias = tmem_base + 2 * p.BN + a * 16;
        for (int pt = pb; pt < pe; ++pt, ++it) {
          const int s = it % p.stages;
          const uint32_t ph = (it / p.stages) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t sa = smem_base + s * stage_bytes;
          // MN-major: 64-wide MN atoms are kABytes apart (LBO), 8-row K groups are 1024 B apart (SBO)
          const uint64_t adesc = make_sdesc_sw128(sa, kABytes, 1024);
          const uint64_t bdesc = make_sdesc_sw128(sa + a_bytes, kABytes, 1024);
#pragma unroll
          for (int kk = 0; kk < kTileM / 16; ++kk) {
            // 16 pixels (K) = two 8-row groups = 2048 bytes -> +128 in the (addr >> 4) field
            umma_f16_ss(d_tmem, adesc + 128 * kk, bdesc + 128 * kk, idesc, (pt > pb || kk > 0) ? 1u : 0u);
          }
          if (with_bias) {
#pragma unroll
            for (int kk = 0; kk < kTileM / 16; ++kk)
              umma_f16_ss(d_bias, adesc + 128 * kk, ones_desc + 128 * kk, idesc_ones, (pt > pb || kk > 0) ? 1u : 0u);
          }
          umma_commit(empty_bar(s));
        }
        umma_commit(tfull_bar(a));
      }
    }
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    uint32_t tcount = 0;
    for (int item = blockIdx.x; item < p.num_items; item += gridDim.x, ++tcount) {
      int mt, nt, tap, grp, pb, pe;
      decode(item, mt, nt, tap, grp, pb, pe);
      const int co = mt * 128 + row;
      const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
      mbar_wait(tfull_bar(a), aph);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + a * p.BN;
      float* dst = p.dw + grp * p.dw_group_stride + ((long long)co * p.taps + tap) * p.Cin;
      if (p.dbias != nullptr && nt == 0 && tap == 0) {      // warp-uniform: column 0 of the ones-product = sum over this item's pixels
        uint32_t v[16];
        __syncwarp();
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + 2 * p.BN + a * 16, v);
        tmem_ld_wait();
        if (pe > pb && co < p.Cout) atomicAdd(p.dbias + co, __uint_as_float(v[0]));
      }
      for (int c0 = 0; c0 < p.BN; c0 += 16) {
        uint32_t v[16];
        __syncwarp();
        tmem_ld16(t_row + c0, v);
        tmem_ld_wait();
        if (pe <= pb || co >= p.Cout) continue;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int ci = nt * p.BN + c0 + j;
          if (ci < p.Cin) atomicAdd(dst + ci, __uint_as_float(v[j]));
        }
      }
      tc_fence_before();
      mbar_arrive(tempty_bar(a));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------ host side
static inline uint32_t pow2_cols(int need) {
  uint32_t c = 32;
  while ((int)c < need) c <<= 1;
  return c;
}

// Tile box over (W, H, B) with tw*th*nb == 128. Power-of-two splits; edges are masked / zero-filled.
static void pick_tile(int H, int W, int B, int& tw, int& th, int& nb) {
  tw = 1;
  while (tw < W && tw < 128) tw <<= 1;   // smallest power of two >= W, capped at 128
  if (tw > 16 && (W % tw) != 0) {        // ragged widths (Inception): prefer narrower tiles to limit waste
    while (tw > 16 && (W % tw) != 0) tw >>= 1;
  }
  th = 1;
  while (th < H && tw * th < 128) th <<= 1;
  nb = 128 / (tw * th);
  (void)B;
}

void fill_epi(EpiArgs& e, const sgb_conv_desc* d) {
  e.H = d->H; e.W = d->W; e.Cout = d->Cout;
  e.alpha = d->alpha; e.alpha_ptr = d->alpha_ptr; e.bias = d->bias;
  e.residual = (const bf16*)d->residual; e.res_cstride = d->res_cstride; e.res_up2 = d->res_up2; e.res_after = d->res_after_mask;
  e.res_scale = d->res_scale != 0.f ? d->res_scale : 1.f;
  e.mask = (const bf16*)d->mask; e.mask_cstride = d->mask_cstride; e.relu = d->relu;
  e.y = d->y; e.y_cstride = d->y_cstride; e.y_fp32 = d->y_fp32;
  e.mask_bits = (const unsigned long long*)d->mask_bits;
  e.relu_bits = (unsigned long long*)d->relu_bits;
  e.sm_mode = d->sm_mode; e.sm_parts = 0; e.sm_stats = d->sm_stats; e.sm_delta = d->sm_delta;
}

static int make_act_tmap(CUtensorMap* m, const void* base, int B, int H, int W, int C, long long cstride, int tw, int th,
                         int nb) {
  uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)B};
  uint64_t strides[3] = {(uint64_t)cstride * 2, (uint64_t)cstride * 2 * W, (uint64_t)cstride * 2 * W * H};
  uint32_t box[4] = {64, (uint32_t)tw, (uint32_t)th, (uint32_t)nb};
  return make_tmap_bf16(m, base, 4, dims, strides, box);
}

}  // namespace sgb

using namespace sgb;

namespace sgb {
bool wgrad3x3_c64_eligible(const sgb_wgrad_desc* d);
int launch_wgrad3x3_c64(const sgb_wgrad_desc* d, cudaStream_t stream);
bool conv3x3_rows_eligible(const sgb_conv_desc* d);
int launch_conv3x3_rows(const sgb_conv_desc* d, cudaStream_t stream);
}  // namespace sgb

// The staged-store epilogue serves the output-heavy layers: K = taps * Cin up to this.  Longer-K layers store directly and
// keep the shared memory of the staging tiles for operand stages.
static constexpr int kEpiTmaMaxK = 640;
static constexpr int kAuxDepth = 2;       // aux ring tiles per epilogue team (profiles/r02_aux_depth_sweep.txt: 3 is no faster)

template <int F>
static int launch_fprop(int grid, size_t smem, cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmY,
                        const CUtensorMap& tmAux, const FpropArgs& p) {
  static bool attr_set = false;
  if (!attr_set) {
    SGB_CUDA(cudaFuncSetAttribute(conv_fprop_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  conv_fprop_kernel<F><<<grid, kThreads, smem, stream>>>(tmA, tmB, tmY, tmAux, p);
  SGB_LAUNCH_CHECK();
  return SGB_OK;
}

static int pick_bn(const sgb_conv_desc* d, long long pixel_tiles) {
  int BN;
  if (d->Cout <= 16) BN = 16;
  else if (d->Cout <= 32) BN = 32;
  else if (d->Cout <= 64) BN = 64;
  else if (d->Cout <= 128 || d->Cout % 256 != 0) BN = 128;
  else BN = 256;
  // 128-wide N tiles only when both halves of every 256-wide tile find an idle SM: an N = 128 tile takes nearly as long as an
  // N = 256 one (the MMA is bound by the shared-memory fetch of the A tile: 712 vs 1381 TFLOP/s on 3x3 128 / 256 channels), so
  // splitting pays only while tiles256 <= SMs / 2 (r02, B = 32: 3x3 256->256 @32x32 ran 557 TFLOP/s as 512 N = 128 tiles)
  {
    long long tiles256 = pixel_tiles * ((d->Cout + 255) / 256);
    if (BN == 256 && 2LL * tiles256 <= sm_count()) BN = 128;
  }
  if (d->w_mode == 2 && BN < 64) BN = 64;  // MN-major B is staged in 64-wide atoms
  return BN;
}

extern "C" int sgb_conv_softmax_parts(const sgb_conv_desc* d) {
  if (!d || d->Cout <= 0) return 0;
  int tw, th, nb;
  pick_tile(d->H, d->W, d->B, tw, th, nb);
  const long long pixel_tiles = (long long)((d->W + tw - 1) / tw) * ((d->H + th - 1) / th) * ((d->B + nb - 1) / nb);
  const int BN = pick_bn(d, pixel_tiles);
  return 2 * ((d->Cout + BN - 1) / BN);
}

extern "C" int sgb_conv_fprop(const sgb_conv_desc* d, sgb_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  SGB_REQUIRE(d && d->x && d->w && d->y);
  SGB_REQUIRE(d->B > 0 && d->H > 0 && d->W > 0 && d->Cin > 0 && d->Cout > 0 && d->KH > 0 && d->KW > 0);
  SGB_REQUIRE(d->Cin % 8 == 0 && d->x_cstride % 8 == 0 && d->x_cstride >= d->Cin);
  SGB_REQUIRE(((uintptr_t)d->x & 15) == 0 && ((uintptr_t)d->w & 15) == 0 && ((uintptr_t)d->y & 15) == 0);
  SGB_REQUIRE(!d->res_up2 || (d->H % 2 == 0 && d->W % 2 == 0));
  SGB_REQUIRE(d->w_mode >= 0 && d->w_mode <= 2);
  SGB_REQUIRE(d->w_mode == 0 || (d->KH == 1 && d->KW == 1 && d->H * d->W >= 128));
  SGB_REQUIRE(d->w_mode != 2 || d->Cout % 8 == 0);
  SGB_REQUIRE(((uintptr_t)d->bias & 15) == 0 && ((uintptr_t)d->residual & 15) == 0 && ((uintptr_t)d->mask & 15) == 0);
  // bit-plane ReLU masks: whole 64-channel words, vector epilogue paths only
  SGB_REQUIRE(!d->mask_bits || (!d->mask && d->Cout % 64 == 0 && !d->y_fp32 && d->out_sub != 2 && ((uintptr_t)d->mask_bits & 7) == 0));
  SGB_REQUIRE(!d->relu_bits || (d->relu && d->Cout % 64 == 0 && !d->y_fp32 && d->out_sub != 2 && d->y_cstride % 8 == 0 &&
                                ((uintptr_t)d->relu_bits & 7) == 0));
  SGB_REQUIRE(!(d->mask_bits || d->relu_bits) || ((!d->residual || d->res_cstride % 8 == 0) && d->y_cstride % 8 == 0));
  // attention softmax inside the epilogue: plain bf16 GEMM tiles only
  SGB_REQUIRE(d->sm_mode >= 0 && d->sm_mode <= 3);
  SGB_REQUIRE(!d->sm_mode || (d->Cout % 64 == 0 && !d->y_fp32 && d->out_sub != 2 && !d->bias && !d->residual && !d->mask && !d->mask_bits &&
                              !d->relu && d->KH == 1 && d->KW == 1 && d->Cin <= kEpiTmaMaxK && d->y_cstride % 8 == 0));
  SGB_REQUIRE(d->sm_mode != 1 || d->sm_stats);
  SGB_REQUIRE(d->sm_mode != 2 || d->sm_stats);
  SGB_REQUIRE(d->sm_mode != 3 || (d->sm_delta && d->sm_p && d->sm_p_cstride % 8 == 0 && ((uintptr_t)d->sm_p & 15) == 0));
  // wide, few-channel 3x3 layers: halo-row kernel (umma_conv3x3.cu)
  if (d->Hin <= 0 && d->Win <= 0 && d->out_sub != 2 && conv3x3_rows_eligible(d)) return launch_conv3x3_rows(d, stream);

  FpropArgs p;
  p.B = d->B; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.Cout = d->Cout;
  p.taps = d->KH * d->KW; p.KW = d->KW; p.pad_h = d->pad_h; p.pad_w = d->pad_w;
  pick_tile(d->H, d->W, d->B, p.tw, p.th, p.nb);
  p.tiles_w = (d->W + p.tw - 1) / p.tw;
  p.tiles_h = (d->H + p.th - 1) / p.th;
  p.tiles_b = (d->B + p.nb - 1) / p.nb;
  const int BN = pick_bn(d, p.tiles_w * p.tiles_h * p.tiles_b);
  p.BN = BN;
  p.w_mode = d->w_mode;
  p.tiles_n = (d->Cout + BN - 1) / BN;
  p.num_tiles = p.tiles_n * p.tiles_w * p.tiles_h * p.tiles_b;
  p.kblocks = (d->Cin + kBlockK - 1) / kBlockK;
  const int Hin = d->Hin > 0 ? d->Hin : d->H, Win = d->Win > 0 ? d->Win : d->W;
  p.out_sub = d->out_sub == 2 ? 2 : 1;
  SGB_REQUIRE(p.out_sub == 1 || (!d->residual && !d->mask));
  fill_epi(p.e, d);
  p.e.sm_parts = 2 * p.tiles_n;
  p.use_tma = (p.out_sub == 1 && epi_can_stage(p.e, BN) && p.taps * d->Cin <= kEpiTmaMaxK) ? 1 : 0;
  // auxiliary epilogue operand through TMA: exactly one of residual / mask, bf16 NHWC with 16-byte aligned channel stride
  p.aux_kind = 0; p.aux_tw = p.tw; p.aux_th = p.th;
  if (p.use_tma && (d->residual != nullptr || d->mask != nullptr)) {   // (mask_bits are 8-byte direct loads)
    // one operand rides TMA: the mask when both are present (full-resolution tile; the residual of such launches is the
    // quarter-size pooled-skip gradient, whose direct 16-byte loads are shared by 2x2 pixel neighbours through L1)
    if (d->mask) p.aux_kind = 2;
    else if (!d->residual) p.aux_kind = 0;                       // bit-plane mask only: nothing to stage
    else if (!d->res_up2) p.aux_kind = 1;
    else if (p.tw >= 2) { p.aux_kind = 1; p.aux_tw = p.tw / 2; p.aux_th = p.th >= 2 ? p.th / 2 : 1; }
  }
  if (d->sm_mode) {
    SGB_REQUIRE(p.use_tma);                                            // (the softmax variants exist only for the staged-store epilogue)
    if (d->sm_mode == 3) p.aux_kind = 3;                               // P tile of the softmax backward
  }
  // short-K layers (one or two K blocks per tile) are store bound: their (small) filter stays resident in shared memory and the
  // space of the B halves of the ring buys more staging tiles per epilogue team = more store bytes in flight
  const uint32_t b_tile = (uint32_t)BN * kBlockK * 2;
  const int kt = p.taps * p.kblocks;
  p.b_resident = (d->w_mode == 0 && p.tiles_n == 1 && kt <= 2 && kt * b_tile <= 64u * 1024u) ? 1 : 0;
  const uint32_t stage_bytes = kABytes + (p.b_resident ? 0u : b_tile);
  p.epi_nbuf = (p.use_tma && kt <= 2) ? 2 : 1;
  p.aux_depth = p.aux_kind ? kAuxDepth : 1;
  auto ring_kb = [&](int nbuf) { return 216 - (p.use_tma ? 32 * nbuf : 0) - (p.aux_kind ? 32 * p.aux_depth : 0) - (p.b_resident ? (int)(kt * b_tile / 1024) : 0); };
  // keep >= 3 operand ring stages: give back aux depth first, then staging tiles
  while (p.aux_kind && p.aux_depth > 1 && ring_kb(p.epi_nbuf) * 1024 < (int)(3 * stage_bytes)) --p.aux_depth;
  while (p.epi_nbuf > 1 && ring_kb(p.epi_nbuf) * 1024 < (int)(3 * stage_bytes)) --p.epi_nbuf;
  int stages = ring_kb(p.epi_nbuf) * 1024 / (int)stage_bytes;
  if (stages > 8) stages = 8;
  if (stages < 2) stages = 2;
  p.stages = stages;
  p.tmem_cols = pow2_cols(2 * BN);

  CUtensorMap tmA, tmB;
  int rc = make_act_tmap(&tmA, d->x, d->B, Hin, Win, d->Cin, d->x_cstride, p.tw, p.th, p.nb);
  if (rc) return rc;
  if (d->w_mode == 0) {
    uint64_t dims[3] = {(uint64_t)d->Cin, (uint64_t)p.taps, (uint64_t)d->Cout};
    uint64_t strides[2] = {(uint64_t)d->Cin * 2, (uint64_t)d->Cin * 2 * p.taps};
    uint32_t box[3] = {64, 1, (uint32_t)BN};
    rc = make_tmap_bf16(&tmB, d->w, 3, dims, strides, box);
  } else if (d->w_mode == 1) {  // per-image [B][N = Cout][K = Cin]
    uint64_t dims[3] = {(uint64_t)d->Cin, (uint64_t)d->B, (uint64_t)d->Cout};
    uint64_t strides[2] = {(uint64_t)d->Cin * 2 * d->Cout, (uint64_t)d->Cin * 2};
    uint32_t box[3] = {64, 1, (uint32_t)BN};
    rc = make_tmap_bf16(&tmB, d->w, 3, dims, strides, box);
  } else {                      // per-image [B][K = Cin][N = Cout], N contiguous
    uint64_t dims[3] = {(uint64_t)d->Cout, (uint64_t)d->Cin, (uint64_t)d->B};
    uint64_t strides[2] = {(uint64_t)d->Cout * 2, (uint64_t)d->Cout * 2 * d->Cin};
    uint32_t box[3] = {64, 64, 1};
    rc = make_tmap_bf16(&tmB, d->w, 3, dims, strides, box);
  }
  if (rc) return rc;
  CUtensorMap tmY = tmA;
  if (p.use_tma) {
    rc = make_act_tmap(&tmY, d->y, d->B, d->H, d->W, d->Cout, d->y_cstride, p.tw, p.th, p.nb);
    if (rc) return rc;
  }
  CUtensorMap tmAux = tmA;
  if (p.aux_kind) {
    const bool half = (p.aux_kind == 1 && d->res_up2);
    const void* ap = p.aux_kind == 1 ? d->residual : (p.aux_kind == 3 ? d->sm_p : d->mask);
    const long long acs = p.aux_kind == 1 ? d->res_cstride : (p.aux_kind == 3 ? d->sm_p_cstride : d->mask_cstride);
    rc = make_act_tmap(&tmAux, ap, d->B, half ? d->H / 2 : d->H, half ? d->W / 2 : d->W, d->Cout, acs, p.aux_tw, p.aux_th, p.nb);
    if (rc) return rc;
  }
  const size_t smem = (size_t)stages * stage_bytes + (p.use_tma ? 2 * p.epi_nbuf * kEpiStageBytes : 0) + (p.aux_kind ? 2 * p.aux_depth * kEpiStageBytes : 0) +
                      (p.b_resident ? (size_t)kt * b_tile : 0) + 1024 + 8 * (2 * stages + 8 + 4 * kAuxDepth) + 16;
  int grid = p.num_tiles < sm_count() ? p.num_tiles : sm_count();
  // the hot epilogue shapes of the training step get compile-time variants; everything else takes the general kernel
  int f = p.use_tma ? epi_flags_of(p.e) : -1;
  SGB_REQUIRE(!d->sm_mode || f == (kEpiFull | (d->sm_mode == 1 ? kEpiSmStats : d->sm_mode == 2 ? kEpiSmApply : kEpiSmBwd)));
  if (f >= 0 && p.aux_kind == 1) f |= kEpiAuxRes;
  if (f >= 0 && p.aux_kind == 2) f |= kEpiAuxMask;
#define SGB_FPROP_CASE(FLAGS) \
  case (FLAGS): return launch_fprop<(FLAGS)>(grid, smem, stream, tmA, tmB, tmY, tmAux, p);
  switch (f) {
    SGB_FPROP_CASE(kEpiFull)                                                          // dgrad / attention GEMMs
    SGB_FPROP_CASE(kEpiFull | kEpiBias)                                               // generator convs
    SGB_FPROP_CASE(kEpiFull | kEpiBias | kEpiRelu)                                    // discriminator convs (no backward expected)
    SGB_FPROP_CASE(kEpiFull | kEpiBias | kEpiRelu | kEpiBitsOut)                      // ... writing the ReLU bit plane
    SGB_FPROP_CASE(kEpiFull | kEpiResPre | kEpiAuxRes)                                // concat-skip dgrad
    SGB_FPROP_CASE(kEpiFull | kEpiBias | kEpiResPre | kEpiAuxRes)                     // block output + skip
    SGB_FPROP_CASE(kEpiFull | kEpiBias | kEpiRelu | kEpiResPre | kEpiAuxRes)          // ... with the next block's ReLU
    SGB_FPROP_CASE(kEpiFull | kEpiBias | kEpiRelu | kEpiResPre | kEpiAuxRes | kEpiBitsOut)
    SGB_FPROP_CASE(kEpiFull | kEpiMask | kEpiMaskBits)                                // dgrad through a ReLU (bit plane)
    SGB_FPROP_CASE(kEpiFull | kEpiMask | kEpiMaskBits | kEpiResPre | kEpiAuxRes)      // fused block entry (bit plane + pooled-skip gradient)
    SGB_FPROP_CASE(kEpiFull | kEpiMask | kEpiAuxMask)                                 // dgrad through a ReLU (bf16 mask tile)
    SGB_FPROP_CASE(kEpiFull | kEpiMask | kEpiResPre | kEpiAuxMask)                    // fused block entry (bf16 mask tile)
    SGB_FPROP_CASE(kEpiFull | kEpiSmStats)                                            // attention: row (max, sum exp) partials of theta . phi^T
    SGB_FPROP_CASE(kEpiFull | kEpiSmApply)                                            // attention: P = softmax(theta . phi^T) written directly
    SGB_FPROP_CASE(kEpiFull | kEpiSmBwd)                                              // attention: dS = P * (do . g^T - delta)
    default: return launch_fprop<-1>(grid, smem, stream, tmA, tmB, tmY, tmAux, p);
  }
#undef SGB_FPROP_CASE
}

extern "C" int sgb_conv_wgrad_fuses_dbias(const sgb_wgrad_desc* d) {
  if (!d) return 0;
  if (wgrad3x3_c64_eligible(d)) return 1;
  return d->per_image ? 0 : 1;          // generic kernel: constant-ones B operand on its (first channel tile, first tap) items
}

extern "C" int sgb_conv_wgrad(const sgb_wgrad_desc* d, sgb_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  SGB_REQUIRE(d && d->x && d->dy && d->dw);
  SGB_REQUIRE(d->B > 0 && d->H > 0 && d->W > 0 && d->Cin > 0 && d->Cout > 0 && d->KH > 0 && d->KW > 0);
  SGB_REQUIRE(d->Cin % 8 == 0 && d->x_cstride % 8 == 0 && d->Cout % 8 == 0 && d->dy_cstride % 8 == 0);
  SGB_REQUIRE(((uintptr_t)d->x & 15) == 0 && ((uintptr_t)d->dy & 15) == 0);
  if (wgrad3x3_c64_eligible(d)) return launch_wgrad3x3_c64(d, stream);
  SGB_REQUIRE(d->dbias == nullptr || !d->per_image);

  WgradArgs p;
  p.B = d->B; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.Cout = d->Cout;
  p.taps = d->KH * d->KW; p.KW = d->KW; p.pad_h = d->pad_h; p.pad_w = d->pad_w;
  pick_tile(d->H, d->W, d->B, p.tw, p.th, p.nb);
  p.tiles_w = (d->W + p.tw - 1) / p.tw;
  p.tiles_h = (d->H + p.th - 1) / p.th;
  p.tiles_b = (d->B + p.nb - 1) / p.nb;
  p.pix_tiles = p.tiles_w * p.tiles_h * p.tiles_b;
  p.BN = (d->Cin <= 64) ? 64 : 128;
  p.tiles_m = (d->Cout + 127) / 128;
  p.tiles_n = (d->Cin + p.BN - 1) / p.BN;
  p.groups = d->per_image ? d->B : 1;
  SGB_REQUIRE(!d->per_image || (p.nb == 1));
  p.tiles_per_group = p.pix_tiles / p.groups;
  p.dw_group_stride = (long long)d->Cout * p.taps * d->Cin;
  const int base_items = p.tiles_m * p.tiles_n * p.taps * p.groups;
  // K-splits: the persistent grid runs ceil(items / SMs) rounds of one item (= tiles_per_split pixel tiles + a drain) each, so
  // pick the split count that minimises rounds x (tiles_per_split + drain); r02 ncu: 9 taps x 33 splits = 297 items ran as
  // 148 + 148 + 1 and left the SMs idle for a third of the launch.
  {
    const int sms = sm_count();
    const int max_splits = p.tiles_per_group < (4 * sms + base_items - 1) / base_items ? p.tiles_per_group : (4 * sms + base_items - 1) / base_items;
    const long long drain = 2;                      // accumulator drain (fp32 red.add of a 128 x BN block) in pixel-tile units
    long long best_cost = -1;
    int best = 1;
    for (int s = 1; s <= (max_splits < 1 ? 1 : max_splits); ++s) {
      const int tps = (p.tiles_per_group + s - 1) / s;
      const int eff = (p.tiles_per_group + tps - 1) / tps;
      const long long rounds = ((long long)base_items * eff + sms - 1) / sms;
      const long long cost = rounds * (tps + drain);
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = s; }
    }
    // near-ties go to MORE splits: concurrent items of one split read the same dY / X tiles at the same moment (36 CTAs on
    // one set of L2 lines for a 256 -> 256 filter), more splits = more distinct streams and drains hidden behind the next item
    // (r02: 3x3 512->512 @16x16 ran 807 TF/s with 1 split x 144 items and 968 TF/s with 3 x 144)
    for (int s = best + 1; s <= (max_splits < 1 ? 1 : max_splits); ++s) {
      const int tps = (p.tiles_per_group + s - 1) / s;
      const int eff = (p.tiles_per_group + tps - 1) / tps;
      const long long rounds = ((long long)base_items * eff + sms - 1) / sms;
      if (50 * rounds * (tps + drain) <= 51 * best_cost) best = s;
    }
    p.tiles_per_split = (p.tiles_per_group + best - 1) / best;
    p.splits = (p.tiles_per_group + p.tiles_per_split - 1) / p.tiles_per_split;
  }
  p.num_items = base_items * p.splits;
  const uint32_t stage_bytes = 2 * kABytes + (p.BN / 64) * kABytes;
  int stages = (int)(((d->dbias ? 224 - 16 : 200) * 1024) / stage_bytes);   // the ones slab must not cost a pipeline stage
  if (stages > 6) stages = 6;
  p.stages = stages;
  p.tmem_cols = pow2_cols(2 * p.BN + (d->dbias ? 32 : 0));
  p.dw = d->dw;
  p.dbias = d->dbias;
  if (d->dbias && !d->accumulate) SGB_CUDA(cudaMemsetAsync(d->dbias, 0, sizeof(float) * (size_t)d->Cout, stream));

  if (!d->accumulate)
    SGB_CUDA(cudaMemsetAsync(d->dw, 0, sizeof(float) * (size_t)d->Cout * p.taps * d->Cin * (d->per_image ? d->B : 1), stream));

  CUtensorMap tmDY, tmX;
  int rc = make_act_tmap(&tmDY, d->dy, d->B, d->H, d->W, d->Cout, d->dy_cstride, p.tw, p.th, p.nb);
  if (rc) return rc;
  rc = make_act_tmap(&tmX, d->x, d->B, d->H, d->W, d->Cin, d->x_cstride, p.tw, p.th, p.nb);
  if (rc) return rc;

  const size_t smem = (size_t)stages * stage_bytes + (d->dbias ? kABytes : 0) + 1024 + 8 * (2 * stages + 4) + 16;
  static bool attr_set = false;
  if (!attr_set) {
    SGB_CUDA(cudaFuncSetAttribute(conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  int grid = p.num_items < sm_count() ? p.num_items : sm_count();
  conv_wgrad_kernel<<<grid, kWgradThreads, smem, stream>>>(tmDY, tmX, p);
  SGB_LAUNCH_CHECK();
  return SGB_OK;
}
