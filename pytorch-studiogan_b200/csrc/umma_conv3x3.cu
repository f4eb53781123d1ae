// 3x3 / pad 1 convolution for wide feature maps with few channels (W % 128 == 0, Cin <= 128): the layers of
// BigGAN-Deep at 128x128 / 256x256, where the generic per-tap kernel is bound by L2 -> smem traffic (each output tile
// re-fetches its input 9x and the whole filter once).  This variant stages HALO ROWS once and forms all nine taps from
// shared memory:
//   work item   = two adjacent output rows x 128 pixels x BN channels (two TMEM accumulators, M = 128 each)
//   A staging   = 4 input rows (h0-1 .. h0+2) of 130 pixels x 64 channels per K block, one TMA box each
//                 (OOB rows / columns zero-filled = padding); tap (kh, kw) of output row j reads row buffer kh + j at a
//                 start address advanced by kw pixels (kw * 128 B): rows stay 128 B apart, and the 128-byte swizzle is a
//                 function of the absolute shared-memory address, so a row-shifted descriptor addresses exactly what TMA wrote
//   B staging   = filter taps; RESIDENT in smem for the whole persistent CTA when they fit (C = 64: 72 KiB), else a ring
//   L2 traffic  = 33 KiB per 128 output pixels at C = 64 (was 216 KiB), 210 KiB at C = 128 (was 576 KiB)
// Warps: 0 = A producer, 1 = MMA issuer + TMEM owner, 2..5 = epilogue, 6 = B producer.
#include "common.cuh"
#include "ptx.cuh"
#include "conv_epilogue.cuh"

namespace sgb {

static constexpr int kRowPix = 130;
static constexpr int kRowLoadBytes = kRowPix * 128;   // 16640
static constexpr int kRowBufBytes = 17 * 1024;        // 17408, keeps every row buffer 1024-byte aligned
static constexpr int kRowsThreads = 128 + kEpiThreads;  // warps 0: A producer, 1: MMA, 2: B producer, 3: idle, 4..11: epilogue

struct RowsArgs {
  int B, H, W, Cin, Cout;
  int kblocks, BN, tiles_n, segs, hpairs, num_tiles;
  int resident, a_stages, b_stages;
  int use_tma, epi_bufs;   // TMA-store epilogue; 2 staging tiles: team t owns output row t, 1: team 0 handles both rows
  uint32_t tmem_cols;
  EpiArgs e;
};

template <int F>      // epilogue variant, see conv_epilogue.cuh
__global__ void __launch_bounds__(kRowsThreads, 1)
conv3x3_rows_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmY, const RowsArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t epi_stage_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_base = epi_stage_base + (p.use_tma ? (uint32_t)p.epi_bufs * kEpiStageBytes : 0u);
  const uint32_t a_stage_bytes = 4 * kRowBufBytes;
  const uint32_t b_tile_bytes = (uint32_t)p.BN * 128u;
  const uint32_t a_base = smem_base;
  const uint32_t b_base = a_base + (uint32_t)p.a_stages * a_stage_bytes;
  const uint32_t b_total = p.resident ? 9u * p.kblocks * b_tile_bytes : (uint32_t)p.b_stages * b_tile_bytes;
  const uint32_t bar_base = b_base + b_total;
  const int nb = p.resident ? 1 : p.b_stages;
  auto a_full = [&](int s) { return bar_base + 8u * s; };
  auto a_empty = [&](int s) { return bar_base + 8u * (p.a_stages + s); };
  auto b_full = [&](int s) { return bar_base + 8u * (2 * p.a_stages + s); };
  auto b_empty = [&](int s) { return bar_base + 8u * (2 * p.a_stages + nb + s); };
  auto tfull = [&](int a) { return bar_base + 8u * (2 * p.a_stages + 2 * nb + a); };
  auto tempty = [&](int a) { return bar_base + 8u * (2 * p.a_stages + 2 * nb + 2 + a); };
  const uint32_t holder = bar_base + 8u * (2 * p.a_stages + 2 * nb + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < p.a_stages; ++s) { mbar_init(a_full(s), 1); mbar_init(a_empty(s), 1); }
    for (int s = 0; s < nb; ++s) { mbar_init(b_full(s), 1); mbar_init(b_empty(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull(a), 1); mbar_init(tempty(a), kEpiThreads); }
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

  auto decode = [&](int tile, int& nt, int& ws, int& hp, int& b) {
    int t = tile;
    nt = t % p.tiles_n; t /= p.tiles_n;
    ws = t % p.segs; t /= p.segs;
    hp = t % p.hpairs; t /= p.hpairs;
    b = t;
  };

  if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------- A producer: four halo rows per K block
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        int nt, ws, hp, b;
        decode(tile, nt, ws, hp, b);
        const int w0 = ws * 128, h0 = hp * 2;
        for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
          const int s = it % p.a_stages;
          mbar_wait(a_empty(s), ((it / p.a_stages) & 1) ^ 1);
          mbar_arrive_expect_tx(a_full(s), 4 * kRowLoadBytes);
          const uint32_t sa = a_base + s * a_stage_bytes;
          for (int r = 0; r < 4; ++r) tma_load_4d(sa + r * kRowBufBytes, &tmA, a_full(s), kb * 64, w0 - 1, h0 - 1 + r, b);
        }
      }
    }
  } else if (warp == 2) {
    if (lane == 0) {
      // ------------------------------------------------------------- B producer: filter taps (resident or ring)
      if (p.resident) {
        mbar_arrive_expect_tx(b_full(0), 9u * p.kblocks * b_tile_bytes);
        // resident order [kb][kw][kh]: the taps (kh, kw) and (kh + 1, kw) are adjacent, so one N = 2 BN operand covers both
        for (int tap = 0; tap < 9; ++tap)
          for (int kb = 0; kb < p.kblocks; ++kb)
            tma_load_3d(b_base + ((kb * 3 + tap % 3) * 3 + tap / 3) * b_tile_bytes, &tmB, b_full(0), kb * 64, tap, 0);
      } else {
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
          int nt, ws, hp, b;
          decode(tile, nt, ws, hp, b);
          for (int kb = 0; kb < p.kblocks; ++kb)
            for (int tap = 0; tap < 9; ++tap, ++it) {
              const int s = it % p.b_stages;
              mbar_wait(b_empty(s), ((it / p.b_stages) & 1) ^ 1);
              mbar_arrive_expect_tx(b_full(s), b_tile_bytes);
              tma_load_3d(b_base + s * b_tile_bytes, &tmB, b_full(s), kb * 64, tap, nt * p.BN);
            }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ------------------------------------------------------------- MMA issuer
      const uint32_t idesc = make_idesc_bf16(128, p.BN, 0, 0);
      if (p.resident) { mbar_wait(b_full(0), 0); tc_fence_after(); }
      uint32_t ita = 0, itb = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++tcount) {
        const uint32_t as = tcount & 1, aph = (tcount >> 1) & 1;
        mbar_wait(tempty(as), aph ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < p.kblocks; ++kb, ++ita) {
          const int sa_i = ita % p.a_stages;
          mbar_wait(a_full(sa_i), (ita / p.a_stages) & 1);
          tc_fence_after();
          const uint32_t sa = a_base + sa_i * a_stage_bytes;
          if (p.resident) {
            // Halo row r feeds output row 1 through tap row r - 1 and output row 0 through tap row r.  For r = 1, 2 both exist:
            // ONE MMA with B = [W(r-1, kw); W(r, kw)] (N = 2 BN) writes the [row 1 | row 0] accumulator pair, so the A
            // operand (the dominant shared-memory read at N = 64) is fetched once instead of twice.
            const uint32_t d_pair = tmem_base + as * 2 * p.BN;
            const uint32_t idesc2 = make_idesc_bf16(128, 2 * p.BN, 0, 0);
            for (int r = 1; r <= 2; ++r)
              for (int kw = 0; kw < 3; ++kw) {
                const uint64_t bdesc = make_sdesc_sw128(b_base + ((kb * 3 + kw) * 3 + (r - 1)) * b_tile_bytes, 16, 1024);
                const uint64_t adesc = make_sdesc_sw128(sa + r * kRowBufBytes + kw * 128, 16, 1024);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                  umma_f16_ss(d_pair, adesc + 2 * kk, bdesc + 2 * kk, idesc2, (kb > 0 || r > 1 || kw > 0 || kk > 0) ? 1u : 0u);
              }
            for (int e = 0; e < 2; ++e)          // r = 0: tap row 0 -> output row 0;  r = 3: tap row 2 -> output row 1
              for (int kw = 0; kw < 3; ++kw) {
                const uint64_t bdesc = make_sdesc_sw128(b_base + ((kb * 3 + kw) * 3 + (e ? 2 : 0)) * b_tile_bytes, 16, 1024);
                const uint64_t adesc = make_sdesc_sw128(sa + (e ? 3 : 0) * kRowBufBytes + kw * 128, 16, 1024);
                const uint32_t d_one = d_pair + (e ? 0 : p.BN);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) umma_f16_ss(d_one, adesc + 2 * kk, bdesc + 2 * kk, idesc, 1u);
              }
            umma_commit(a_empty(sa_i));
            continue;
          }
          for (int tap = 0; tap < 9; ++tap) {          // filter ring (the resident case was handled above)
            const int kh = tap / 3, kw = tap % 3;
            const int sb = itb % p.b_stages;
            mbar_wait(b_full(sb), (itb / p.b_stages) & 1);
            tc_fence_after();
            const uint64_t bdesc = make_sdesc_sw128(b_base + sb * b_tile_bytes, 16, 1024);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const uint64_t adesc = make_sdesc_sw128(sa + (kh + j) * kRowBufBytes + kw * 128, 16, 1024);
              const uint32_t d_tmem = tmem_base + (as * 2 + j) * p.BN;
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_f16_ss(d_tmem, adesc + 2 * kk, bdesc + 2 * kk, idesc, (kb > 0 || tap > 0 || kk > 0) ? 1u : 0u);
            }
            umma_commit(b_empty(sb));
            ++itb;
          }
          umma_commit(a_empty(sa_i));
        }
        umma_commit(tfull(as));
      }
    }
  } else if (warp >= 4) {
    // --------------------------------------------------------------- epilogue: 8 warps (two teams)
    const int q = warp & 3;
    const int team = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const bool leader = (q == 0) && (lane == 0);
    const bool vec_ok = epi_vec_ok(p.e);
    const float alpha = p.e.alpha_ptr ? p.e.alpha * __ldg(p.e.alpha_ptr) : p.e.alpha;
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++tcount) {
      int nt, ws, hp, b;
      decode(tile, nt, ws, hp, b);
      const int w = ws * 128 + row;
      const uint32_t as = tcount & 1, aph = (tcount >> 1) & 1;
      mbar_wait(tfull(as), aph);
      tc_fence_after();
#pragma unroll 1
      for (int j = 0; j < 2; ++j) {
        const int h = hp * 2 + j;
        const long long pix = ((long long)b * p.H + h) * p.W + w;
        const long long rpix = p.e.res_up2 ? (((long long)b * (p.H >> 1) + (h >> 1)) * (p.W >> 1) + (w >> 1)) : pix;
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (as * 2 + (p.resident ? 1 - j : j)) * p.BN;
        if (F >= 0 || p.use_tma) {               // (the host picks a compile-time variant only for staged stores)
          // team t owns output row t.  epi_bufs == 2: both teams stage + TMA-store; epi_bufs == 1 (no room for a second
          // staging tile, C = 64): team 0 stages + TMA-stores row 0 while team 1 writes row 1 with direct 16-byte stores
          // (one full 128-byte line per thread at C = 64) -- two rows drain concurrently instead of back to back.
          if (team == j) {
            if (p.epi_bufs == 2 || team == 0) {
              const uint32_t stage = epi_stage_base + ((p.epi_bufs == 2) ? team : 0) * kEpiStageBytes;
              // one team covers every chunk of its row: run the chunk loop for both parities on the team's own barrier
              epilogue_tile_tma<F>(p.e, &tmY, t_row, p.BN, nt * p.BN, ws * 128, h, b, true, pix, rpix, alpha, stage, team, row, leader, 1);
            } else {
              epilogue_row<F>(p.e, t_row, p.BN, nt * p.BN, true, pix, rpix, alpha, vec_ok);
            }
          }
        } else if (team == 0) {
          epilogue_row<F>(p.e, t_row, p.BN, nt * p.BN, true, pix, rpix, alpha, vec_ok);
        }
      }
      tc_fence_before();
      mbar_arrive(tempty(as));
    }
    if (p.use_tma && leader) bulk_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

void fill_epi(EpiArgs& e, const sgb_conv_desc* d);

template <int F>
static int launch_rows(int grid, size_t smem, cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmY,
                       const RowsArgs& p) {
  static bool attr_set = false;
  if (!attr_set) {
    SGB_CUDA(cudaFuncSetAttribute(conv3x3_rows_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  conv3x3_rows_kernel<F><<<grid, kRowsThreads, smem, stream>>>(tmA, tmB, tmY, p);
  SGB_LAUNCH_CHECK();
  return SGB_OK;
}

bool conv3x3_rows_eligible(const sgb_conv_desc* d) {
  return d->KH == 3 && d->KW == 3 && d->pad_h == 1 && d->pad_w == 1 && d->w_mode == 0 && d->W % 128 == 0 && d->H % 2 == 0 &&
         d->Cin % 64 == 0 && d->Cin <= 128 && d->Cout % 8 == 0;
}

int launch_conv3x3_rows(const sgb_conv_desc* d, cudaStream_t stream) {
  RowsArgs p;
  p.B = d->B; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.Cout = d->Cout;
  p.kblocks = d->Cin / 64;
  p.BN = d->Cout <= 128 ? (d->Cout + 15) / 16 * 16 : 128;   // Cout = 8 (padded image channels) runs as one N = 16 tile
  p.tiles_n = (d->Cout + p.BN - 1) / p.BN;
  p.segs = d->W / 128;
  p.hpairs = d->H / 2;
  p.num_tiles = p.tiles_n * p.segs * p.hpairs * d->B;
  fill_epi(p.e, d);
  const uint32_t b_tile = p.BN * 128u;
  const uint32_t budget = 227u * 1024u - 2048u;
  const uint32_t a_stage = 4 * kRowBufBytes;
  const uint32_t resident_bytes = 9u * p.kblocks * b_tile;
  p.use_tma = epi_can_stage(p.e, p.BN) ? 1 : 0;
  p.epi_bufs = 2;
  p.resident = (p.tiles_n == 1 && resident_bytes + 2 * a_stage + (p.use_tma ? kEpiStageBytes : 0) <= budget) ? 1 : 0;
  if (p.resident) {
    if (p.use_tma && resident_bytes + 2 * a_stage + 2 * kEpiStageBytes > budget) p.epi_bufs = 1;
    const uint32_t epi_bytes = p.use_tma ? p.epi_bufs * kEpiStageBytes : 0;
    p.a_stages = (int)((budget - resident_bytes - epi_bytes) / a_stage);
    if (p.a_stages > 3) p.a_stages = 3;
    p.b_stages = 1;
  } else {
    p.a_stages = 2;
    const uint32_t epi_bytes = p.use_tma ? p.epi_bufs * kEpiStageBytes : 0;
    p.b_stages = (int)((budget - 2 * a_stage - epi_bytes) / b_tile);
    if (p.b_stages > 6) p.b_stages = 6;
    if (p.b_stages < 2) return SGB_ERR_UNSUPPORTED;
  }
  uint32_t cols = 32;
  while ((int)cols < 4 * p.BN) cols <<= 1;
  p.tmem_cols = cols;

  CUtensorMap tmA, tmB;
  {
    uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)d->W, (uint64_t)d->H, (uint64_t)d->B};
    uint64_t strides[3] = {(uint64_t)d->x_cstride * 2, (uint64_t)d->x_cstride * 2 * d->W, (uint64_t)d->x_cstride * 2 * d->W * d->H};
    uint32_t box[4] = {64, (uint32_t)kRowPix, 1, 1};
    int rc = make_tmap_bf16(&tmA, d->x, 4, dims, strides, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)d->Cin, 9, (uint64_t)d->Cout};
    uint64_t strides[2] = {(uint64_t)d->Cin * 2, (uint64_t)d->Cin * 2 * 9};
    uint32_t box[3] = {64, 1, (uint32_t)p.BN};
    int rc = make_tmap_bf16(&tmB, d->w, 3, dims, strides, box);
    if (rc) return rc;
  }
  CUtensorMap tmY = tmA;
  if (p.use_tma) {
    uint64_t dims[4] = {(uint64_t)d->Cout, (uint64_t)d->W, (uint64_t)d->H, (uint64_t)d->B};
    uint64_t strides[3] = {(uint64_t)d->y_cstride * 2, (uint64_t)d->y_cstride * 2 * d->W, (uint64_t)d->y_cstride * 2 * d->W * d->H};
    uint32_t box[4] = {64, 128, 1, 1};
    int rc = make_tmap_bf16(&tmY, d->y, 4, dims, strides, box);
    if (rc) return rc;
  }
  const int nb = p.resident ? 1 : p.b_stages;
  const size_t smem = (size_t)p.a_stages * a_stage + (p.resident ? resident_bytes : p.b_stages * b_tile) +
                      (p.use_tma ? p.epi_bufs * kEpiStageBytes : 0) + 1024 +
                      8 * (2 * p.a_stages + 2 * nb + 4) + 16;
  const int grid = p.num_tiles < sm_count() ? p.num_tiles : sm_count();
  const int f = p.use_tma ? epi_flags_of(p.e) : -1;
  switch (f) {
    case kEpiFull | kEpiBias: return launch_rows<kEpiFull | kEpiBias>(grid, smem, stream, tmA, tmB, tmY, p);                        // generator 3x3
    case kEpiFull | kEpiBias | kEpiRelu: return launch_rows<kEpiFull | kEpiBias | kEpiRelu>(grid, smem, stream, tmA, tmB, tmY, p);    // discriminator 3x3
    case kEpiFull | kEpiBias | kEpiRelu | kEpiBitsOut:
      return launch_rows<kEpiFull | kEpiBias | kEpiRelu | kEpiBitsOut>(grid, smem, stream, tmA, tmB, tmY, p);                         // ... writing the ReLU bit plane
    case kEpiFull | kEpiMask: return launch_rows<kEpiFull | kEpiMask>(grid, smem, stream, tmA, tmB, tmY, p);                        // dgrad through a ReLU (bf16 mask)
    case kEpiFull | kEpiMask | kEpiMaskBits:
      return launch_rows<kEpiFull | kEpiMask | kEpiMaskBits>(grid, smem, stream, tmA, tmB, tmY, p);                                   // dgrad through a ReLU (bit plane)
    case kEpiFull: return launch_rows<kEpiFull>(grid, smem, stream, tmA, tmB, tmY, p);                                              // plain dgrad
    default: return launch_rows<-1>(grid, smem, stream, tmA, tmB, tmY, p);
  }
}

}  // namespace sgb
