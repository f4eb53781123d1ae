// Fused conv epilogue shared by the tcgen05 conv kernels: TMEM accumulator row -> alpha, bias, residual (optionally read
// from a half-resolution tensor = nearest x2 upsample), ReLU, ReLU-mask, post-mask residual -> bf16 / fp32 NHWC store.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace sgb {

struct EpiArgs {
  int H, W, Cout;
  float alpha;
  const float* alpha_ptr;
  const float* bias;
  const bf16* residual; long long res_cstride; int res_up2; int res_after; float res_scale;
  const bf16* mask; long long mask_cstride;
  int relu;
  void* y; long long y_cstride; int y_fp32;
  // ReLU masks as bit planes (Cout % 64 == 0): one 64-bit word per (pixel, 64-channel chunk), bit j = channel 64 * chunk + j.
  // mask_bits replaces ``mask`` (1/16 of its bytes); relu_bits is written by a relu epilogue for the consumer's backward.
  const unsigned long long* mask_bits;
  unsigned long long* relu_bits;
  // Row softmax of the attention map inside the GEMM epilogues (one thread = one query row of the tile):
  //   sm_mode 1: no output; per row and per (channel tile, team) the partial (max, sum exp) of its columns -> sm_stats
  //   sm_mode 2: y = exp(acc - m) / l with (m, l) merged from the row's sm_parts partials
  //   sm_mode 3: y = P * (acc - delta[row]) (softmax backward; P arrives through the aux TMA ring, kind 3)
  int sm_mode, sm_parts;
  float* sm_stats;            // [rows][sm_parts][2]
  const float* sm_delta;      // [rows]
};

// 16 accumulator values -> 16 mask bits (value > 0)
__device__ __forceinline__ uint32_t positive_bits16(const float (&f)[16]) {
  uint32_t b = 0u;
#pragma unroll
  for (int j = 0; j < 16; ++j) b |= (f[j] > 0.f) ? (1u << j) : 0u;
  return b;
}
// The same 16 bits from the PACKED bf16 pairs of a post-ReLU piece (every half is +0 or a positive value <= 0x7F80): adding
// 0x7FFF to a half sets its bit 15 iff it is non-zero without carrying into its neighbour; PRMT gathers the four flag bytes of
// two words, one multiply moves the four flags into a nibble.  27 integer instructions per piece instead of 40
// (FSETP + SEL per element + adds) -- the bit plane is paid for by write-bound layers (r02: 1x1 32->128 @256x256 +1.2 ms).
__device__ __forceinline__ uint32_t positive_bits16_packed(const uint32_t (&w)[8]) {
  uint32_t bits = 0u;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t ta = w[2 * k] + 0x7FFF7FFFu, tb = w[2 * k + 1] + 0x7FFF7FFFu;
    const uint32_t flags = __byte_perm(ta, tb, 0x7531) & 0x80808080u;      // bits 7 / 15 / 23 / 31 = elements 4k .. 4k+3
    bits |= ((flags * 0x00204081u) >> 28) << (4 * k);
  }
  return bits;
}
__device__ __forceinline__ void apply_bits16(float (&f)[16], uint32_t mb) {
#pragma unroll
  for (int j = 0; j < 16; ++j) f[j] = ((mb >> j) & 1u) ? f[j] : 0.f;
}

__device__ __forceinline__ float bf16_bits_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_bits_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

// Operand alignment of the vector epilogue paths: whole 8-channel units, 16-byte aligned rows of every bf16 operand.
__host__ __device__ inline bool epi_vec_ok(const EpiArgs& p) {
  return (p.Cout % 8 == 0) && (p.y_cstride % 8 == 0) && (p.residual == nullptr || p.res_cstride % 8 == 0) &&
         (p.mask == nullptr || p.mask_cstride % 8 == 0);
}
// A launch can stage its output tile in shared memory and write it with TMA tensor stores: bf16 output, whole 64-channel
// chunks per tile, aligned operands.
__host__ __device__ inline bool epi_can_stage(const EpiArgs& p, int BN) {
  return !p.y_fp32 && (BN % 64 == 0) && epi_vec_ok(p);
}

// One 16-column piece of the epilogue.  Every store path runs the same steps in the same order (alpha, [softmax], bias,
// residual, ReLU, mask, post-mask residual, pack), so their outputs are bit-identical; where a bf16 operand comes from (the
// aux ring in shared memory, __ldg, or zeros past a ragged channel tail) is the caller's choice.
__device__ __forceinline__ void piece_bias(float (&f)[16], const float* bias, int nvalid) {
  const float4* bp = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (4 * j < nvalid) {
      const float4 bb = __ldg(bp + j);
      f[4 * j + 0] += bb.x; f[4 * j + 1] += bb.y; f[4 * j + 2] += bb.z; f[4 * j + 3] += bb.w;
    }
  }
}
// f += rs * r for the 16 bf16 values of two 16-byte units
__device__ __forceinline__ void piece_res_fma(float (&f)[16], uint4 r0, uint4 r1, float rs) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const uint4 r = j ? r1 : r0;
    f[8 * j + 0] = fmaf(bf16_bits_lo(r.x), rs, f[8 * j + 0]); f[8 * j + 1] = fmaf(bf16_bits_hi(r.x), rs, f[8 * j + 1]);
    f[8 * j + 2] = fmaf(bf16_bits_lo(r.y), rs, f[8 * j + 2]); f[8 * j + 3] = fmaf(bf16_bits_hi(r.y), rs, f[8 * j + 3]);
    f[8 * j + 4] = fmaf(bf16_bits_lo(r.z), rs, f[8 * j + 4]); f[8 * j + 5] = fmaf(bf16_bits_hi(r.z), rs, f[8 * j + 5]);
    f[8 * j + 6] = fmaf(bf16_bits_lo(r.w), rs, f[8 * j + 6]); f[8 * j + 7] = fmaf(bf16_bits_hi(r.w), rs, f[8 * j + 7]);
  }
}
// f = (m > 0) ? f : 0 for the 16 bf16 mask values of two 16-byte units
__device__ __forceinline__ void piece_mask_bf16(float (&f)[16], uint4 m0, uint4 m1) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const uint4 m = j ? m1 : m0;
    f[8 * j + 0] = bf16_bits_lo(m.x) > 0.f ? f[8 * j + 0] : 0.f;
    f[8 * j + 1] = bf16_bits_hi(m.x) > 0.f ? f[8 * j + 1] : 0.f;
    f[8 * j + 2] = bf16_bits_lo(m.y) > 0.f ? f[8 * j + 2] : 0.f;
    f[8 * j + 3] = bf16_bits_hi(m.y) > 0.f ? f[8 * j + 3] : 0.f;
    f[8 * j + 4] = bf16_bits_lo(m.z) > 0.f ? f[8 * j + 4] : 0.f;
    f[8 * j + 5] = bf16_bits_hi(m.z) > 0.f ? f[8 * j + 5] : 0.f;
    f[8 * j + 6] = bf16_bits_lo(m.w) > 0.f ? f[8 * j + 6] : 0.f;
    f[8 * j + 7] = bf16_bits_hi(m.w) > 0.f ? f[8 * j + 7] : 0.f;
  }
}
__device__ __forceinline__ void piece_pack(const float (&f)[16], uint32_t (&w)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) w[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
}

// -------------------------------------------------------------------------------------------------------------------
// Epilogue v2 (bf16 NHWC output, channel tile a multiple of 64): two teams of four warps take alternate 64-channel
// chunks; a team converts its 128 x 64 chunk into a SWIZZLE_128B staging tile in shared memory and one thread issues
// a TMA tensor store (full 128-byte lines, asynchronous, out-of-range rows / channels clipped by the hardware).  This
// replaces 16-byte-per-lane strided global stores, which bound every wide 1x1 layer (K = 64..128) at ~1/6 of HBM speed.
// -------------------------------------------------------------------------------------------------------------------
static constexpr int kEpiThreads = 256;           // 8 epilogue warps

// Optional auxiliary operand of the epilogue (the residual OR the ReLU-mask tensor) staged by TMA: one SWIZZLE_128B box of
// the same pixels (or of the half-resolution source pixels for the nearest-x2 residual) per 64-channel chunk.  The boxes are
// fetched by a dedicated producer warp into a per-team ring of ``depth`` tiles (full / empty mbarriers), in the order the team
// consumes its chunks, so their ~1-2 us latency under load overlaps ``depth`` chunks of epilogue work instead of one.
struct EpiAux {
  int kind;                 // 1 residual, 2 mask
  uint32_t ring;            // this team's first aux tile (1024-byte aligned), tiles 16 KiB apart
  uint32_t full0, empty0;   // this team's first full / empty mbarrier (8 bytes apart per slot)
  int depth;                // ring slots per team
  uint32_t* cnt;            // per-thread count of chunks consumed by this team
  int arow;                 // aux-tile row this thread reads
};

__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 r;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}
static constexpr int kEpiStageBytes = 128 * 128;  // one 128-row x 64-channel bf16 chunk

// Compile-time epilogue variants.  The per-piece loop below runs on 2 warps per scheduler with little latency hiding, so
// every run-time test of "is there a bias / residual / mask / ragged channel tail" costs issue slots on the critical path of
// the memory-bound layers (ncu, r01: ~150 SASS instructions per 16-column piece).  F >= 0 fixes those questions at compile
// time (bit 0 bias, 1 ReLU, 2 residual before the activation, 3 residual after the mask, 4 mask, 5 Cout % 64 == 0 and every
// 16-byte alignment holds); F < 0 is the fully general run-time version.
static constexpr int kEpiBias = 1, kEpiRelu = 2, kEpiResPre = 4, kEpiResPost = 8, kEpiMask = 16, kEpiFull = 32;
// ... bit 6: the mask is a bit plane (mask_bits), 7 / 8: the residual / the bf16 mask tile arrives through the aux TMA ring,
// 9: the ReLU epilogue also writes its bit plane (relu_bits).  r02 ncu of the fused block-entry dgrad (mask + residual): with these
// three questions left to run time the compiler if-converts both sides of each and the piece loop issues 12 instructions per
// output element (the bias-only variant: 2).
static constexpr int kEpiMaskBits = 64, kEpiAuxRes = 128, kEpiAuxMask = 256, kEpiBitsOut = 512;
// attention: bit 10 softmax statistics (no store), 11 softmax apply, 12 softmax backward (P tile through the aux ring)
static constexpr int kEpiSmStats = 1024, kEpiSmApply = 2048, kEpiSmBwd = 4096;

__host__ __device__ inline int epi_flags_of(const EpiArgs& p) {
  int f = 0;
  if (p.bias) f |= kEpiBias;
  if (p.relu) f |= kEpiRelu;
  if (p.residual) f |= p.res_after ? kEpiResPost : kEpiResPre;
  if (p.mask || p.mask_bits) f |= kEpiMask;
  if (p.mask_bits) f |= kEpiMaskBits;
  if (p.relu && p.relu_bits) f |= kEpiBitsOut;
  if (p.Cout % 64 == 0) f |= kEpiFull;
  if (p.sm_mode == 1) f |= kEpiSmStats;
  if (p.sm_mode == 2) f |= kEpiSmApply;
  if (p.sm_mode == 3) f |= kEpiSmBwd;
  return f;
}

// 2^x on the SFU (ex2.approx: 2^-22 relative error, far below the bf16 rounding of the softmax output); the accurate exp2f
// costs ~10 instructions per element and made the softmax epilogues issue bound (r02: 0.88 ms per score-GEMM pass)
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Softmax statistics of one accumulator tile (sm_mode 1): this thread's row, the 64-column chunks of its team; the running
// (max, sum exp) pair is kept in registers and stored once -- nothing else leaves the SM.
__device__ __forceinline__ void epilogue_tile_smstats(const EpiArgs& p, uint32_t t_row, int BN, int n0, bool valid, long long pix,
                                                      float alpha, int team, int part) {
  float m = -INFINITY, l = 0.f;
  constexpr float kLog2e = 1.4426950408889634f;
  for (int cc = team; cc * 64 < BN; cc += 2) {
    if (n0 + cc * 64 >= p.Cout) break;
#pragma unroll 1
    for (int s0 = 0; s0 < 4; s0 += 2) {
      uint32_t v[2][16];
      __syncwarp();
      tmem_ld16(t_row + cc * 64 + s0 * 16, v[0]);
      tmem_ld16(t_row + cc * 64 + (s0 + 1) * 16, v[1]);
      tmem_ld_wait();
      float pm = -INFINITY;
#pragma unroll
      for (int q = 0; q < 2; ++q)
#pragma unroll
        for (int j = 0; j < 16; ++j) pm = fmaxf(pm, __uint_as_float(v[q][j]) * alpha);
      const float mn = fmaxf(m, pm);
      float acc = 0.f;
#pragma unroll
      const float a2 = alpha * kLog2e, mn2 = -mn * kLog2e;
      for (int q = 0; q < 2; ++q)
#pragma unroll
        for (int j = 0; j < 16; ++j) acc += fast_ex2(fmaf(__uint_as_float(v[q][j]), a2, mn2));
      l = l * fast_ex2((m - mn) * kLog2e) + acc;
      m = mn;
    }
  }
  if (valid) {
    float2* dst = reinterpret_cast<float2*>(p.sm_stats) + pix * p.sm_parts + part;
    *dst = make_float2(m, l);
  }
}

// Direct-store epilogue.  One thread = one accumulator row (TMEM lane); t_row: TMEM address of this warp's lane quadrant at
// the accumulator's first column.  All 32 lanes of the warp must call this (tcgen05.ld is warp-collective); stores are
// predicated by valid.  F < 0: run-time flags, bf16 or fp32 output, scalar path for a ragged / unaligned channel tail.
// F >= 0 (bf16 output, Cout % 64 == 0, 16-byte aligned operands): two 16-column pieces per TMEM wait.  Used by the halo-row
// kernel's second output row at C = 64 (no room for a second staging tile): one full 128-byte line per thread and piece pair.
template <int F>
__device__ __forceinline__ void epilogue_row(const EpiArgs& p, uint32_t t_row, int BN, int n0, bool valid, long long pix,
                                             long long rpix, float alpha, bool vec_ok) {
  static_assert(F < 0 || (F & kEpiFull), "compile-time variants have a full channel tile");
  constexpr int NP = F >= 0 ? 2 : 1;
  const bool has_bias = F < 0 ? p.bias != nullptr : (F & kEpiBias) != 0;
  const bool do_relu = F < 0 ? p.relu != 0 : (F & kEpiRelu) != 0;
  const bool res_pre = F < 0 ? (p.residual != nullptr && !p.res_after) : (F & kEpiResPre) != 0;
  const bool res_post = F < 0 ? (p.residual != nullptr && p.res_after) : (F & kEpiResPost) != 0;
  const bool use_mbits = F < 0 ? p.mask_bits != nullptr : (F & kEpiMaskBits) != 0;
  const bool has_mask = F < 0 ? p.mask != nullptr : (F & kEpiMask) != 0;
  const bool emit_bits = F < 0 ? p.relu_bits != nullptr : (F & kEpiBitsOut) != 0;
  const bool y_fp32 = F < 0 && p.y_fp32;
  const float rs = p.res_scale;
  for (int c0 = 0; c0 < BN; c0 += 16 * NP) {
    uint32_t v[NP][16];
    __syncwarp();
#pragma unroll
    for (int q = 0; q < NP; ++q) tmem_ld16(t_row + c0 + 16 * q, v[q]);
    tmem_ld_wait();
    if (!valid || n0 + c0 >= p.Cout) continue;
#pragma unroll
    for (int q = 0; q < NP; ++q) {
      const int n = n0 + c0 + 16 * q;
      float f[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[q][j]) * alpha;
      if (F >= 0 || (vec_ok && n + 16 <= p.Cout)) {
        if (has_bias) piece_bias(f, p.bias + n, 16);
        if (res_pre) {
          const uint4* rp = reinterpret_cast<const uint4*>(p.residual + rpix * p.res_cstride + n);
          piece_res_fma(f, __ldg(rp), __ldg(rp + 1), rs);
        }
        if (do_relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
          if (emit_bits)
            reinterpret_cast<unsigned short*>(p.relu_bits)[(pix * (p.Cout >> 6) + (n >> 6)) * 4 + ((n >> 4) & 3)] =
                (unsigned short)positive_bits16(f);
        }
        if (use_mbits) {
          apply_bits16(f, __ldg(reinterpret_cast<const unsigned short*>(p.mask_bits) + (pix * (p.Cout >> 6) + (n >> 6)) * 4 + ((n >> 4) & 3)));
        } else if (has_mask) {
          const uint4* mp = reinterpret_cast<const uint4*>(p.mask + pix * p.mask_cstride + n);
          piece_mask_bf16(f, __ldg(mp), __ldg(mp + 1));
        }
        if (res_post) {
          const uint4* rp = reinterpret_cast<const uint4*>(p.residual + rpix * p.res_cstride + n);
          piece_res_fma(f, __ldg(rp), __ldg(rp + 1), rs);
        }
        if (y_fp32) {
          float4* yp = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.y) + pix * p.y_cstride + n);
#pragma unroll
          for (int j = 0; j < 4; ++j) yp[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
        } else {
          uint32_t w[8];
          piece_pack(f, w);
          uint4* yp = reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(p.y) + pix * p.y_cstride + n);
          yp[0] = make_uint4(w[0], w[1], w[2], w[3]);
          yp[1] = make_uint4(w[4], w[5], w[6], w[7]);
        }
      } else {
        // ragged / unaligned channel tail (e.g. Cout = 3): scalar path
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int nn = n + j;
          if (nn < p.Cout) {
            float x = f[j];
            if (p.bias) x += __ldg(p.bias + nn);
            if (res_pre) x = fmaf(__bfloat162float(p.residual[rpix * p.res_cstride + nn]), rs, x);
            if (p.relu) x = fmaxf(x, 0.f);
            if (p.mask) x = __bfloat162float(p.mask[pix * p.mask_cstride + nn]) > 0.f ? x : 0.f;
            if (res_post) x = fmaf(__bfloat162float(p.residual[rpix * p.res_cstride + nn]), rs, x);
            if (p.y_fp32) reinterpret_cast<float*>(p.y)[pix * p.y_cstride + nn] = x;
            else reinterpret_cast<bf16*>(p.y)[pix * p.y_cstride + nn] = __float2bfloat16_rn(x);
          }
        }
      }
    }
  }
}

// Staged-store epilogue.  t_row: TMEM address (lane quadrant of this warp, first column of the accumulator).
// c1..c3: box coordinates (w0, h0, b0) of the tile in the output tensor map; channel coordinate = n0 + chunk * 64.
// stage : this team's first staging tile (1024-byte aligned).  team in {0,1}; row = accumulator row of this thread.
// sbuf != nullptr: the team owns two staging tiles used in turn, so a chunk only waits for the store issued two chunks ago --
// the latency of the previous tensor store is off the critical path and more bytes are in flight; nullptr: one tile.
template <int F>
__device__ __forceinline__ void epilogue_tile_tma(const EpiArgs& p, const CUtensorMap* tmY, uint32_t t_row, int BN, int n0,
                                                  int c1, int c2, int c3, bool valid, long long pix, long long rpix, float alpha,
                                                  uint32_t stage, int team, int row, bool leader, int chunk_stride = 2,
                                                  const EpiAux* aux = nullptr, uint32_t* sbuf = nullptr) {
  constexpr int kTeamThreads = 128;
  constexpr bool sm_apply = F >= 0 && (F & kEpiSmApply) != 0, sm_bwd = F >= 0 && (F & kEpiSmBwd) != 0;
  constexpr float kLog2e = 1.4426950408889634f;
  float sm_a = 0.f, sm_b = 1.f;                    // apply: (row max, 1 / row sum); backward: (delta, -)
  if (sm_apply && valid) {
    const float2* st = reinterpret_cast<const float2*>(p.sm_stats) + pix * p.sm_parts;
    float m = -INFINITY;
    for (int i = 0; i < p.sm_parts; ++i) m = fmaxf(m, __ldcg(&st[i].x));
    float l = 0.f;
    for (int i = 0; i < p.sm_parts; ++i) { const float2 t = __ldcg(&st[i]); l += t.y * fast_ex2((t.x - m) * kLog2e); }
    sm_a = -m * kLog2e; sm_b = 1.f / l;          // exponent offset in base-2 units
  }
  if (sm_bwd && valid) sm_a = __ldg(p.sm_delta + pix);
  const bool has_bias = F < 0 ? p.bias != nullptr : (F & kEpiBias) != 0;
  const bool do_relu = F < 0 ? p.relu != 0 : (F & kEpiRelu) != 0;
  const bool res_pre = F < 0 ? (p.residual != nullptr && !p.res_after) : (F & kEpiResPre) != 0;
  const bool res_post = F < 0 ? (p.residual != nullptr && p.res_after) : (F & kEpiResPost) != 0;
  const bool has_mask = F < 0 ? (p.mask != nullptr || p.mask_bits != nullptr) : (F & kEpiMask) != 0;
  const bool use_mbits = F < 0 ? (has_mask && p.mask_bits != nullptr) : (F & kEpiMaskBits) != 0;
  const bool emit_bits = F < 0 ? (do_relu && p.relu_bits != nullptr) : (F & kEpiBitsOut) != 0;
  // the ReLU is the last arithmetic of the piece (no mask, no post-mask residual): take the bits from the packed output words
  constexpr bool bits_from_packed = F >= 0 && (F & kEpiBitsOut) != 0 && (F & (kEpiMask | kEpiResPost)) == 0;
  const long long nw = p.Cout >> 6;
  const bool full_c = F >= 0 && (F & kEpiFull) != 0;       // no channel-tail tests
  const float rs = p.res_scale;
  const uint32_t sw = (uint32_t)(row & 7);
  // 1: residual tile via TMA, 2: mask tile via TMA (compile-time for F >= 0: the host sets the aux bits iff it passes ``aux``)
  const int aux_kind = F < 0 ? ((aux && (res_pre || res_post || has_mask)) ? aux->kind : 0)
                             : ((F & kEpiAuxRes) ? 1 : ((F & kEpiAuxMask) ? 2 : (sm_bwd ? 3 : 0)));
  const uint32_t asw = aux ? (uint32_t)(aux->arow & 7) : 0u;
  for (int cc = (chunk_stride == 2 ? team : 0); cc * 64 < BN; cc += chunk_stride) {
    const int nbase = n0 + cc * 64;
    if (nbase >= p.Cout) break;
    uint32_t mlo = 0u, mhi = 0u, olo = 0u, ohi = 0u;
    if (use_mbits && valid) {                    // 8 bytes instead of a 128-byte line of the bf16 activation
      const uint2 m = __ldg(reinterpret_cast<const uint2*>(p.mask_bits) + pix * nw + (nbase >> 6));
      mlo = m.x; mhi = m.y;
    }
    const uint32_t stage_cur = stage + (sbuf ? *sbuf * kEpiStageBytes : 0u);
    const uint32_t srow = stage_cur + (uint32_t)row * 128u;
    if (leader) {                                // the store that last used this staging tile has finished reading it
      if (!sbuf) bulk_wait_read0();
      else bulk_wait_read1();
    }
    if (sbuf) *sbuf ^= 1u;
    named_bar_sync(1 + team, kTeamThreads);
    uint32_t arow_addr = 0u, aslot = 0u;
    if (aux_kind) {                              // residual / mask chunk: one TMA box (fetched ahead by the aux producer warp)
      aslot = *aux->cnt % (uint32_t)aux->depth;
      mbar_wait(aux->full0 + 8u * aslot, (*aux->cnt / (uint32_t)aux->depth) & 1u);
      arow_addr = aux->ring + aslot * kEpiStageBytes + (uint32_t)aux->arow * 128u;
      *aux->cnt += 1u;
    }
    // compile-time variants handle two 16-column pieces per iteration: both TMEM loads are in flight before the single wait
    // (the variants use ~77 registers, the general version 102), which hides part of the LDTM latency that two warps per
    // scheduler cannot hide by themselves
    constexpr int NP = F >= 0 ? 2 : 1;
    auto piece = [&](const int s, const uint32_t (&v)[16], const uint32_t mb) -> uint32_t {
        const int n = nbase + s * 16;
        float f[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[j]) * alpha;
        const int nvalid = full_c ? 16 : p.Cout - n;   // channels of this 16-wide piece inside the tensor: >= 16, 8 (Cout % 16 == 8) or <= 0
        const bool in_c = full_c || nvalid > 0;
        // 16-byte unit j (0, 1) of this piece in a bf16 operand: this row of the aux tile when the operand rides the ring
        // (unit u of a 128-byte line lives at u ^ (row & 7)), else a direct load, zeros past the channel tail
        auto unit = [&](const bf16* base, int kind, int j) -> uint4 {
          return (aux_kind == kind) ? ld_shared_v4(arow_addr + (((uint32_t)(2 * s + j) ^ asw) << 4))
                                    : ((full_c || 8 * j < nvalid) ? __ldg(reinterpret_cast<const uint4*>(base) + j)
                                                                  : make_uint4(0u, 0u, 0u, 0u));
        };
        if (sm_apply) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = fast_ex2(fmaf(f[j], kLog2e, sm_a)) * sm_b;
        }
        if (sm_bwd) {                                // dS = P * (dP - delta); P: this row of the aux tile
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const uint4 r = ld_shared_v4(arow_addr + (((uint32_t)(2 * s + j) ^ asw) << 4));
            f[8 * j + 0] = bf16_bits_lo(r.x) * (f[8 * j + 0] - sm_a); f[8 * j + 1] = bf16_bits_hi(r.x) * (f[8 * j + 1] - sm_a);
            f[8 * j + 2] = bf16_bits_lo(r.y) * (f[8 * j + 2] - sm_a); f[8 * j + 3] = bf16_bits_hi(r.y) * (f[8 * j + 3] - sm_a);
            f[8 * j + 4] = bf16_bits_lo(r.z) * (f[8 * j + 4] - sm_a); f[8 * j + 5] = bf16_bits_hi(r.z) * (f[8 * j + 5] - sm_a);
            f[8 * j + 6] = bf16_bits_lo(r.w) * (f[8 * j + 6] - sm_a); f[8 * j + 7] = bf16_bits_hi(r.w) * (f[8 * j + 7] - sm_a);
          }
        }
        if (has_bias && in_c) piece_bias(f, p.bias + n, nvalid);
        if (res_pre && in_c && valid) {
          const bf16* rrow = p.residual + rpix * p.res_cstride + n;
          piece_res_fma(f, unit(rrow, 1, 0), unit(rrow, 1, 1), rs);
        }
        uint32_t ob = 0u;
        if (do_relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
          if (emit_bits && !bits_from_packed) ob = positive_bits16(f);
        }
        if (use_mbits) {
          apply_bits16(f, mb);
        } else if (has_mask && in_c && valid) {
          const bf16* mrow = p.mask + pix * p.mask_cstride + n;
          piece_mask_bf16(f, unit(mrow, 2, 0), unit(mrow, 2, 1));
        }
        if (res_post && in_c && valid) {
          const bf16* rrow = p.residual + rpix * p.res_cstride + n;
          piece_res_fma(f, unit(rrow, 1, 0), unit(rrow, 1, 1), rs);
        }
        // 16 channels = two 16-byte units (2s, 2s+1) of this row's 128-byte line; unit u lives at (u ^ (row & 7))
        uint32_t w[8];
        piece_pack(f, w);
        if (bits_from_packed) ob = positive_bits16_packed(w);
        st_shared_v4(srow + (((uint32_t)(2 * s) ^ sw) << 4), w[0], w[1], w[2], w[3]);
        st_shared_v4(srow + (((uint32_t)(2 * s + 1) ^ sw) << 4), w[4], w[5], w[6], w[7]);
        return ob;
    };
#pragma unroll 1
    for (int s0 = 0; s0 < 4; s0 += NP) {
      uint32_t v[NP][16];
      __syncwarp();
#pragma unroll
      for (int q = 0; q < NP; ++q) tmem_ld16(t_row + cc * 64 + (s0 + q) * 16, v[q]);
      tmem_ld_wait();
#pragma unroll
      for (int q = 0; q < NP; ++q) {
        const int s = s0 + q;
        const uint32_t ob = piece(s, v[q], ((s < 2 ? mlo : mhi) >> (16 * (s & 1))) & 0xFFFFu);
        if (s < 2) olo |= ob << (16 * (s & 1));
        else ohi |= ob << (16 * (s & 1));
      }
    }
    if (emit_bits && valid) reinterpret_cast<uint2*>(p.relu_bits)[pix * nw + (nbase >> 6)] = make_uint2(olo, ohi);
    fence_proxy_async_smem();                    // generic-proxy smem writes -> visible to the TMA (async proxy)
    named_bar_sync(1 + team, kTeamThreads);
    if (leader) {
      tma_store_4d(tmY, stage_cur, nbase, c1, c2, c3);
      bulk_commit();
      if (aux_kind) mbar_arrive(aux->empty0 + 8u * aslot);   // every thread of the team is past its last read of the aux tile (barrier above)
    }
  }
}

}  // namespace sgb
