// Conv-coupling conditioner (layers/coupling.py:26-29) on the 5th-generation tensor cores: tcgen05.mma with fp32-faithful
// two-term operand splitting (kind::f16 with scaled fp16 hi/lo pairs by default, kind::tf32 hi/lo as the alternative),
// accumulators in TMEM, weights streamed by 1-D bulk TMA copies.
//
//   h = W3 * relu( conv_KHxKW_reflect( relu(W1 * x0 + b1) ) + b2 ) + b3          per pixel, per sample
//
// Mapping.  Pixels sit on the MMA M axis (128 rows per instruction), channels on N, input channels (x taps) on K (8 per
// instruction).  A CTA keeps the activations of S whole samples resident in shared memory as K-major SWIZZLE_128B
// operand rows (one 128-byte row = 32 channels of one stored pixel; `P` panels of 32 channels), each value stored twice:
// v (the tensor core truncates it to tf32 = hi) and lo = v - trunc_tf32(v).  The kxk convolution needs no im2col copy:
// a tap (ky,kx) is the same operand seen through a descriptor whose start row is shifted by ky*YS + kx.  Two layouts:
//   plain   : stored row = s*RPS + yp*WP + xp over the reflect-padded image ((H+KH-1) x (W+KW-1)); accumulator row
//             m = stored row of the output pixel; rows whose xp >= W are computed and thrown away;
//   segment : (W % 8 == 0) the image row is cut into segments of 8 output pixels stored with their halo as GS = 8+KW-1
//             rows; stored row = ((yp*S + s)*NSEG + seg)*GS + xs.  An MMA row-group of 8 is one segment and the descriptor's
//             group stride (SBO) is GS*128 bytes, so every accumulator row is a real pixel (no waste on M).
// Operand kinds.  F16 (default): hi = fp16_rn(v), lo' = fp16_rn((v - hi) * 2^11): two 11-bit significands = 22+ bits of v, the
// 2^11 scale keeps lo' a normal fp16 number; a 128-byte row holds 64 channels, K = 16 per instruction, and the accumulator
// columns that collect the two cross products are scaled back by 2^-11 in the epilogue.  Values beyond +-65504 (never seen in
// ActNorm-normalised flows) saturate; CFPP_TC_KIND=tf32 selects the tf32 pair (hi = trunc_tf32(v), lo = v - hi; 32 channels per
// row, K = 8, twice the shared-memory bytes and MMA time) which has fp32 range.
// fp32 accuracy from two-term operands:  A*B ~= A_hi*B_hi + A_hi*B_lo + A_lo*B_hi.  The first two products are ONE instruction
// with the stacked operand [B_hi ; B_lo] (N' = 2N, accumulator columns [0,N) and [N,2N)); the third accumulates into
// [N,2N) as well, so that block holds both cross products (both carry the 2^11 scale of the fp16 kind); the epilogue adds
// the (rescaled) second block to the first.  (tools/umma_probe*.cu measured the descriptor conventions, the
// 2^-21-grade accuracy of the split and the issue rates this layout is built on.)
//
// Roles (448 threads, one persistent CTA per SM): warps 0-11 = epilogue (TMEM -> bias/ReLU/split -> shared, final store
// to HBM; also the x0 -> operand-row transform), warp 12 = MMA issuer (one thread), warp 13 = producer (weight chunks
// through an mbarrier ring + next tile's x0 prefetch).  Per tile: stage 1 (1x1) -> epilogue 1 -> stage 2 (kxk, the
// 94 %) -> epilogue 2 -> stage 3 (1x1) -> epilogue 3.
#include <stdlib.h>
#include <string.h>
#include <type_traits>
#include <cuda_fp16.h>
#include "common.cuh"
#include "umma.cuh"

#ifndef CFPP_TC_WIDE
#define CFPP_TC_WIDE 0   // 1: 32-column epilogue items in the one-CTA-per-SM kernels (spills under the 144-register cap since the packed-math epilogue)
#endif

namespace cfpp {
namespace tc {

struct Plan {
  int B, Cin, Ch, Cout, H, W, KH, KW;
  int kind;                          // 0 = tf32 pair (32 channels / row, K = 8), 1 = scaled fp16 pair (64 channels / row, K = 16)
  int rb;                            // operand row bytes: 128 (SWIZZLE_128B) or, fp16 kind with <= 32 channels, 64 (SWIZZLE_64B)
  int occ;                           // CTAs per SM this plan is sized for (1 or 2)
  int seg, S, NSEG, GS, YS, RPS, WP, HP;
  int R, T1, T2, NG;                 // stored rows per tile, M-tiles of stage 1 / stages 2-3, row groups of stage 2 (segment)
  int P, KS1, N2, N3;                // channel panels, k-steps of stage 1, N of stages 1-2, N of stage 3 (padded to 16)
  int stage_bytes, nstages, ntiles;
  int resident;                      // 1: nstages == chunks per tile, the weight chunks are loaded once per CTA and never recycled
  int pipe;                          // 1: software-pipelined tiles (two operand sets, disjoint accumulator column blocks), see the kernel
  int region_bytes;                  // bytes of one (hi|lo, panel) operand region
  int off_ring, off_stage_x, off_bias, off_tab, off_ls, off_add, off_bar, smem_bytes;   // off_tab: R + T2*128 packed row-decode words; off_ls: per-row log-scale partials; off_add: S x N3 per-sample output bias (b3 + CN(c)) of the fused coupling
  long long x_bstride;
};

// OCC = CTAs resident per SM.  OCC 1: one CTA owns the SM (12 epilogue warps, 512 TMEM columns, ~226 KB).  OCC 2: two CTAs with half
// the shared memory and TMEM columns each (8 epilogue warps): a tile's stages are serial inside a CTA (MMA -> epilogue -> MMA ...),
// so a second resident CTA lets the tensor pipe work on its tile while this one's epilogue warps transform accumulators.
#ifndef CFPP_TC_EPI1
#define CFPP_TC_EPI1 16   // epilogue warps of the one-CTA-per-SM kernels
#endif
__host__ __device__ constexpr int epi_warps(int occ) { return occ == 1 ? CFPP_TC_EPI1 : 8; }   // multiple of 4: a warp reaches TMEM lanes 32*(warp%4) .. +31 only
__host__ __device__ constexpr int cta_threads(int occ) { return (epi_warps(occ) + 2) * 32; }
constexpr int kMaxStages = 12;                 // ring slots; when every weight chunk of a tile fits (<= 12 chunks) the weights stay resident

// byte offset of 16-byte chunk `chunk` of operand row `row`: SWIZZLE_128B (chunk ^= row % 8) or SWIZZLE_64B (chunk ^= (row / 2) % 4)
__host__ __device__ __forceinline__ uint32_t row_off(int row, int chunk, int rb) {
  return rb == 128 ? (uint32_t)row * 128u + (uint32_t)(((chunk ^ row) & 7) << 4) : (uint32_t)row * 64u + (uint32_t)(((chunk ^ (row >> 1)) & 3) << 4);
}
constexpr float kLoScale = 2048.f, kLoInv = 1.f / 2048.f;
// packed fp16 pair {low half = a, high half = b}: round to nearest, saturating to the finite range (one F2FP instruction)
__device__ __forceinline__ uint32_t pack_f16x2_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// (hi, lo') fp16 pair of two values, packed as two half2 words.  hi = v truncated to 11 significant bits (a mask: exactly
// representable in fp16 over its normal range, so the conversion is exact and v - hi needs no conversion back), lo' = rn((v - hi) * 2^11);
// the conversions saturate to the finite fp16 range.  4 instructions per element.
template <bool NONNEG>
__device__ __forceinline__ void f16_split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const float ha = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u), hb = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
  hi = pack_f16x2_sat(ha, hb);
  lo = pack_f16x2_sat((a - ha) * kLoScale, (b - hb) * kLoScale);
}
// Store 8 consecutive channels (col8 = first channel within the panel, multiple of 8) of operand row `row` as (hi, lo) operands.
template <bool F16, bool NONNEG = false>
__device__ __forceinline__ void store_group8(uint8_t* ph, uint8_t* pl, int row, int col8, const float (&v)[8], int rb) {
  if (F16) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) f16_split2<NONNEG>(v[2 * q], v[2 * q + 1], h[q], l[q]);
    const uint32_t off = row_off(row, col8 >> 3, rb);
    *reinterpret_cast<uint4*>(ph + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(pl + off) = make_uint4(l[0], l[1], l[2], l[3]);
  } else {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const uint32_t off = sw128(row, col8 + 4 * q);
      *reinterpret_cast<float4*>(ph + off) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
      *reinterpret_cast<float4*>(pl + off) = make_float4(tf32_lo(v[4 * q]), tf32_lo(v[4 * q + 1]), tf32_lo(v[4 * q + 2]), tf32_lo(v[4 * q + 3]));
    }
  }
}

// TT consecutive M-tiles x KS k-steps of one weight chunk, fully unrolled: per k-step the stacked product (N' = 2N into [0,2N)) and
// the lo-activation product (N into [N,2N)).
template <bool F16, int KS, int TT, int KS0 = 0>
__device__ __forceinline__ void mma_tiles(uint32_t d, uint32_t dcols, uint64_t ah, uint64_t al, uint32_t tile_u, uint64_t bd,
                                          uint32_t id2, uint32_t id1, uint32_t first_acc) {
#pragma unroll
  for (int tt = 0; tt < TT; ++tt) {
    const uint32_t dd = d + tt * dcols, dl = dd + (dcols >> 1);
    const uint64_t a0 = ah + (uint64_t)(tt * tile_u), a1 = al + (uint64_t)(tt * tile_u);
#pragma unroll
    for (int ks = KS0; ks < KS; ++ks) {
      mma_k<F16>(dd, a0 + 2 * ks, bd + 2 * ks, id2, ks ? 1u : first_acc);
      mma_k<F16>(dl, a1 + 2 * ks, bd + 2 * ks, id1, 1);
    }
  }
}
__device__ __forceinline__ int reflect(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

struct Args {
  const float* x; float* h; const uint8_t* wpack; const float* b1; const float* b2; const float* b3; const float* bias1_b;
  // fused affine coupling (coupling.py:50-66), z != NULL: h is not written; x must be the full (B, 2 Cin, H, W) tensor
  float* z; float* ldj; const float* add; const float* logp_c; float logp_scale;
  // training forward (profile-variant kernels only): the post-ReLU activations of stages 1 / 2 as fp32 (B, Ch, H, W) for the backward pass, or NULL
  float* h1_out; float* h2_out;
  long long wrepl_stride; int nrepl;   // experiment: weight stream replicas (CTA uses replica blockIdx % nrepl)
  int dbg;           // debug (profile kernels only): bit 0 = epilogue warps skip their TMEM loads / operand stores, bit 1 = skip the x0 transform
  long long* prof;   // optional (debug): 12 phase-cycle counters of CTA 0's epilogue thread 0, see cfpp_conv_cond_tc_set_profile
};

// Barrier slots (8 bytes each) inside the barrier block.
enum { BAR_FULL = 0, BAR_EMPTY = kMaxStages, BAR_XFULL = 2 * kMaxStages, BAR_XEMPTY, BAR_AREADY, BAR_ACC1, BAR_ACC2, BAR_ACC3, BAR_H1, BAR_H2, BAR_COUNT };

// stored operand row -> (sample, source pixel) of the reflect-padded image
template <bool SEG>
__device__ __forceinline__ void decode_stored(const Plan& p, int r, int& s, int& y, int& x) {
  if (SEG) {
    const int xs = r % p.GS; int q = r / p.GS;
    const int sg = q % p.NSEG; q /= p.NSEG;
    s = q % p.S; const int yp = q / p.S;
    y = reflect(yp - p.KH / 2, p.H); x = reflect(sg * 8 + xs - p.KW / 2, p.W);
  } else {
    s = r / p.RPS; const int rem = r - s * p.RPS;
    const int yp = rem / p.WP, xp = rem - yp * p.WP;
    y = reflect(yp - p.KH / 2, p.H); x = reflect(xp - p.KW / 2, p.W);
  }
}
// accumulator row of stages 2/3 -> output pixel; false for rows that are not a pixel
template <bool SEG>
__device__ __forceinline__ bool decode_out(const Plan& p, int m, int& s, int& y, int& x) {
  if (SEG) {
    int g = m >> 3; const int j = m & 7;
    const int sg = g % p.NSEG; g /= p.NSEG;
    s = g % p.S; y = g / p.S; x = sg * 8 + j;
    return y < p.H;
  } else {
    s = m / p.RPS; const int rem = m - s * p.RPS;
    y = rem / p.WP; x = rem - y * p.WP;
    return s < p.S && y < p.H && x < p.W;
  }
}

// Packed fp32 pairs (Blackwell add / mul / fma .f32x2: two IEEE round-to-nearest operations per issue slot; results identical to the scalar forms)
__device__ __forceinline__ uint64_t pack2(float a, float b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpack2(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) { uint64_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fsub2(uint64_t a, uint64_t b) { uint64_t r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) { uint64_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

// One epilogue item: 32 accumulator columns [c0, c0+32) (16 when only 16 remain) of one row, two column blocks of N each ->
// + bias -> ReLU -> (v, lo) -> operand row `row`.  All four TMEM loads are in flight before the single wait.  All 32 lanes
// must call (tcgen05.ld is warp-collective); `write` only guards the stores.
template <bool F16, bool EMIT = false>
__device__ __forceinline__ void store_split16(const float (&v)[16], const float (&u)[16], const float* __restrict__ bias, uint8_t* ph, uint8_t* pl,
                                              int row, int col, int rb, float* gdst = nullptr, int gstride = 0) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    if (F16) {
      // per pair of channels: (v + b) and the rescaled cross block in packed fp32, ReLU, hi = 11-bit truncation, lo' = (r - hi) * 2^11
      uint32_t h[4], l[4];
      const uint64_t kinv = pack2(kLoInv, kLoInv), ksc = pack2(kLoScale, kLoScale);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = 8 * g + 2 * q;
        const float2 b = *reinterpret_cast<const float2*>(bias + i);
        float r0, r1;
        unpack2(ffma2(pack2(u[i], u[i + 1]), kinv, fadd2(pack2(v[i], v[i + 1]), pack2(b.x, b.y))), r0, r1);
        r0 = fmaxf(r0, 0.f); r1 = fmaxf(r1, 0.f);
        if (EMIT && gdst) { gdst[(size_t)i * gstride] = r0; gdst[(size_t)(i + 1) * gstride] = r1; }      // fp32 activation for the backward pass
        const float h0 = __uint_as_float(__float_as_uint(r0) & 0xFFFFE000u), h1 = __uint_as_float(__float_as_uint(r1) & 0xFFFFE000u);
        float l0, l1;
        unpack2(fmul2(fsub2(pack2(r0, r1), pack2(h0, h1)), ksc), l0, l1);
        h[q] = pack_f16x2_sat(h0, h1);
        l[q] = pack_f16x2_sat(l0, l1);
      }
      const uint32_t off = row_off(row, (col + 8 * g) >> 3, rb);
      *reinterpret_cast<uint4*>(ph + off) = make_uint4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<uint4*>(pl + off) = make_uint4(l[0], l[1], l[2], l[3]);
    } else {
      float o[8];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const float4 b = *reinterpret_cast<const float4*>(bias + 8 * g + 4 * q);
        const int i = 8 * g + 4 * q;
        o[4 * q + 0] = fmaxf(v[i + 0] + u[i + 0] + b.x, 0.f); o[4 * q + 1] = fmaxf(v[i + 1] + u[i + 1] + b.y, 0.f);
        o[4 * q + 2] = fmaxf(v[i + 2] + u[i + 2] + b.z, 0.f); o[4 * q + 3] = fmaxf(v[i + 3] + u[i + 3] + b.w, 0.f);
      }
      if (EMIT && gdst) {
#pragma unroll
        for (int q = 0; q < 8; ++q) gdst[(size_t)(8 * g + q) * gstride] = o[q];
      }
      store_group8<F16, true>(ph, pl, row, col + 8 * g, o, rb);
    }
  }
}
template <bool F16, bool WIDE, bool EMIT = false>
__device__ __forceinline__ void epilogue_to_operand(uint32_t taddr, int N, int c0, const float* __restrict__ bias, uint8_t* a_hi, uint8_t* a_lo,
                                                    int region_bytes, int row, bool write, int rb, float* gdst = nullptr, int gstride = 0) {
  const int cps = F16 ? (rb == 64 ? 5 : 6) : 5;               // log2(channels per operand row)
  float v0[16], u0[16], v1[16], u1[16];
  const bool two = WIDE && c0 + 16 < N;                       // warp-uniform; narrow items (16 columns) halve the live registers
  tmem_ld16(taddr + c0, v0);
  tmem_ld16(taddr + N + c0, u0);
  if (two) { tmem_ld16(taddr + c0 + 16, v1); tmem_ld16(taddr + N + c0 + 16, u1); }
  tmem_ld_wait();
  if (write) {
    const int pn = c0 >> cps, cc = c0 & ((1 << cps) - 1);
    uint8_t* ph = a_hi + pn * region_bytes;
    uint8_t* pl = a_lo + pn * region_bytes;
    store_split16<F16, EMIT>(v0, u0, bias + c0, ph, pl, row, cc, rb, gdst, gstride);
    if (two) store_split16<F16, EMIT>(v1, u1, bias + c0 + 16, ph, pl, row, cc + 16, rb, gdst ? gdst + (size_t)16 * gstride : nullptr, gstride);
  }
}

// stage-2 geometries known at compile time (see stage2_fixed in the kernel); all in descriptor units of 16 bytes
struct GeoL1 { static constexpr int P = 1, T2 = 2, KS = 2, ROW_U1 = 4, YS_U = 20 * 4, REGION_U = 368 * 64 / 16, TILE_U = 10 * 64, STAGE_U = 2 * 32 * 64 / 16, DCOLS = 64,
                                    T1 = 3, KS1 = 1, LIN_U = 8 * 64, DCOLS3 = 32; };
struct GeoL2 { static constexpr int P = 1, T2 = 1, KS = 4, ROW_U1 = 8, YS_U = 20 * 8, REGION_U = 208 * 128 / 16, TILE_U = 10 * 128, STAGE_U = 2 * 64 * 128 / 16, DCOLS = 128,
                                    T1 = 2, KS1 = 1, LIN_U = 8 * 128, DCOLS3 = 64; };
struct GeoL3 { static constexpr int P = 2, T2 = 2, KS = 4, ROW_U1 = 8, YS_U = 6 * 8, REGION_U = 256 * 128 / 16, TILE_U = 8 * 128, STAGE_U = 2 * 128 * 128 / 16, DCOLS = 256,
                                    T1 = 2, KS1 = 2, LIN_U = 8 * 128, DCOLS3 = 128; };

// PIPE (software-pipelined tiles, one CTA per SM).  A tile's stages are a dependent chain  x0 -> MMA 1 -> epilogue 1 -> MMA 2 -> epilogue 2 ->
// MMA 3 -> epilogue 3: run back to back, the epilogue warps idle through every MMA stage and the tensor pipe idles through every epilogue
// (ncu r1: tensor pipe 21 %, issue slots 47 % with two such CTAs per SM).  With PIPE the epilogue warps interleave two tiles,
//     X(i+1)  E2(i)  E1(i+1)  E3(i)        and the issuer     S1(i+1)  S3(i)  S2(i+1),
// so that every MMA stage runs under epilogue work of the other tile: S1(i+1) under E2(i), S3(i) under E1(i+1), S2(i+1) -- the 94 % --
// under E3(i) and X(i+2).  This takes two operand sets in shared memory (tile parity) and three disjoint accumulator column blocks in TMEM
// (stage 1 | stage 2 | stage 3: T1*2*N2 + T2*2*N2 + T2*2*N3 <= 512), and a weight stream in consumption order (W1, W3.., W2..).
template <bool SEG, bool PROF, bool F16, int OCC, bool PIPE>
__global__ void __launch_bounds__(cta_threads(OCC), OCC) conv_cond_tc_kernel(const Plan p, const Args a) {
  constexpr int kEpiWarps = epi_warps(OCC), kEpiGroups = kEpiWarps / 4, kEpiThreads = kEpiWarps * 32;
  constexpr int kMmaWarp = kEpiWarps, kProdWarp = kEpiWarps + 1, kThreads = cta_threads(OCC), kTmemCols = 512 / OCC;
  constexpr int KE = F16 ? 16 : 8;                          // channels per MMA k-step
  const int rb = p.rb, CPR = F16 ? rb >> 1 : 32;            // operand row bytes, channels per operand row (panel)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // pointer arithmetic on the shared array (not an integer round trip) keeps the address space visible to the compiler: LDS / STS, 32-bit addressing
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* a_hi0 = base;                                    // [P][region]; PIPE: a second (hi | lo) set follows for the odd tiles
  uint8_t* a_lo0 = base + (size_t)p.P * p.region_bytes;     // [P][region]
  const uint32_t set_bytes = 2u * (uint32_t)p.P * (uint32_t)p.region_bytes;
  const uint32_t col1 = 0, col2 = PIPE ? (uint32_t)(p.T1 * 2 * p.N2) : 0u, col3 = PIPE ? col2 + (uint32_t)(p.T2 * 2 * p.N2) : 0u;   // accumulator column blocks
  uint8_t* ring = base + p.off_ring;
  float* xstage = reinterpret_cast<float*>(base + p.off_stage_x);
  float* sb1 = reinterpret_cast<float*>(base + p.off_bias);
  float* sb2 = sb1 + p.N2;
  float* sb3 = sb2 + p.N2;
  const uint32_t bars = smem_u32(base + p.off_bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base + p.off_bar + BAR_COUNT * 8);
  auto bar = [&](int i) { return bars + 8u * i; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int HW = p.H * p.W;
  const int xfloats = p.Cin * HW;                           // staged floats per sample

  if (tid == 0) {
    for (int i = 0; i < p.nstages; ++i) { mbar_init(bar(BAR_FULL + i), 1); mbar_init(bar(BAR_EMPTY + i), 1); }
    mbar_init(bar(BAR_XFULL), 1); mbar_init(bar(BAR_XEMPTY), kEpiThreads); mbar_init(bar(BAR_AREADY), kEpiThreads);
    mbar_init(bar(BAR_ACC1), 1); mbar_init(bar(BAR_ACC2), 1); mbar_init(bar(BAR_ACC3), 1);
    mbar_init(bar(BAR_H1), kEpiThreads); mbar_init(bar(BAR_H2), kEpiThreads);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < p.N2; i += kThreads) { sb1[i] = i < p.Ch ? a.b1[i] : 0.f; sb2[i] = i < p.Ch ? a.b2[i] : 0.f; }
  for (int i = tid; i < p.N3; i += kThreads) sb3[i] = i < p.Cout ? a.b3[i] : 0.f;
  // Row-decode tables (the index arithmetic has runtime divisors: done once per CTA, not once per tile).
  //   tab_in[r]  : stored operand row r  -> (s << 24) | (y << 12) | x of the source pixel (reflect / overlap applied)
  //   tab_out[m] : accumulator row m     -> bit 31 = is a pixel, (s << 24) | (y << 12) | x
  uint32_t* tab_in = reinterpret_cast<uint32_t*>(base + p.off_tab);
  uint32_t* tab_out = tab_in + p.R;
  for (int r = tid; r < p.R; r += kThreads) { int s_, y_, x_; decode_stored<SEG>(p, r, s_, y_, x_); tab_in[r] = ((uint32_t)s_ << 24) | ((uint32_t)y_ << 12) | (uint32_t)x_; }
  for (int m = tid; m < p.T2 * 128; m += kThreads) {
    int s_, y_, x_;
    const bool ok = decode_out<SEG>(p, m, s_, y_, x_);
    tab_out[m] = ok ? (0x80000000u | ((uint32_t)s_ << 24) | ((uint32_t)y_ << 12) | (uint32_t)x_) : 0u;
  }
  if (a.z != nullptr) for (int i = tid; i < kEpiGroups * p.T2 * 128; i += kThreads) reinterpret_cast<float*>(base + p.off_ls)[i] = 0.f;
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int nchunks_tile = 1 + p.KH * p.KW * p.P + p.P;     // W1, W2 (tap, panel), W3 (panel)
  const int my_tiles = (p.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == kProdWarp) {
    // ===================== producer: weight chunks through the ring, next tile's x0 into the staging buffer ==========
    if (elect_one()) {
      uint32_t st = 0, rphase = 0;
      auto load_x = [&](int it) {
        const int tile = blockIdx.x + it * gridDim.x;
        const int b0 = tile * p.S, nS = min(p.S, p.B - b0);
        mbar_wait(bar(BAR_XEMPTY), (it & 1) ^ 1);
        mbar_expect_tx(bar(BAR_XFULL), (uint32_t)(nS * xfloats * 4));
        for (int s = 0; s < nS; ++s)
          bulk_g2s(smem_u32(xstage + (size_t)s * xfloats), a.x + (size_t)(b0 + s) * p.x_bstride, (uint32_t)(xfloats * 4), bar(BAR_XFULL));
      };
      auto load_chunk = [&](int c) {
        mbar_wait(bar(BAR_EMPTY + st), rphase ^ 1);
        const uint32_t bytes = (c < nchunks_tile - p.P) ? (uint32_t)(2 * p.N2 * rb) : (uint32_t)(2 * p.N3 * rb);
        mbar_expect_tx(bar(BAR_FULL + st), bytes);
        bulk_g2s(smem_u32(ring + (size_t)st * p.stage_bytes), a.wpack + (size_t)(blockIdx.x % a.nrepl) * a.wrepl_stride + (size_t)c * p.stage_bytes, bytes, bar(BAR_FULL + st));
        if (++st == (uint32_t)p.nstages) { st = 0; rphase ^= 1; }
      };
      if (!PIPE) {
        for (int it = 0; it < my_tiles; ++it) {
          load_x(it);
          if (!(p.resident && it > 0))                             // resident weights: loaded for the first tile only
            for (int c = 0; c < nchunks_tile; ++c) load_chunk(c);
        }
      } else if (my_tiles > 0) {
        const int cW3 = nchunks_tile - p.P;                        // chunks: 0 = W1, [1, cW3) = W2 (tap, panel), [cW3, nchunks) = W3 (panel)
        load_x(0);
        if (p.resident) {
          for (int c = 0; c < nchunks_tile; ++c) load_chunk(c);
          for (int it = 1; it < my_tiles; ++it) load_x(it);
        } else {
          // consumption order of the issuer: S1(0) S2(0) | S1(i+1) S3(i) S2(i+1) ...; the x0 of a tile is requested one iteration early
          if (my_tiles > 1) load_x(1);
          load_chunk(0);
          for (int c = 1; c < cW3; ++c) load_chunk(c);
          for (int it = 0; it < my_tiles; ++it) {
            if (it + 2 < my_tiles) load_x(it + 2);
            if (it + 1 < my_tiles) load_chunk(0);
            for (int c = cW3; c < nchunks_tile; ++c) load_chunk(c);
            if (it + 1 < my_tiles) for (int c = 1; c < cW3; ++c) load_chunk(c);
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer ==================================================================================
    // One thread.  tcgen05.mma issue blocks once ~2 instructions are queued, and this thread's own scalar work runs at
    // dependent-instruction latency, so any work placed BETWEEN weight chunks starves the tensor pipe (measured: every
    // cycle of gap beyond ~100 is lost, tools/umma_probe3.cu).  Hence: loop-invariant descriptors are hoisted, the ring
    // position advances by adds, and the wait for the NEXT chunk sits in the middle of the current chunk's instructions.
    if (elect_one()) {
      const uint32_t idN2 = make_idesc(p.N2, F16), id2N2 = make_idesc(2 * p.N2, F16), idN3 = make_idesc(p.N3, F16), id2N3 = make_idesc(2 * p.N3, F16);
      const uint32_t sbo2 = (uint32_t)(p.GS * rb), sbo1 = (uint32_t)(8 * rb), lin_u = (uint32_t)(8 * rb), row_u1 = (uint32_t)rb >> 4;   // lin_u: 128 rows / 16
      const uint32_t tile_cols2 = 2 * p.N2, tile_cols3 = 2 * p.N3;
      const uint64_t ahi_lin0 = make_desc(smem_u32(a_hi0), sbo1, rb), alo_lin0 = make_desc(smem_u32(a_lo0), sbo1, rb);   // stages 1 / 3: plain 128-row tiles
      const uint64_t ahi_seg0 = make_desc(smem_u32(a_hi0), sbo2, rb), alo_seg0 = make_desc(smem_u32(a_lo0), sbo2, rb);   // stage 2: group stride GS rows
      const uint32_t set_u = set_bytes >> 4;                                                                             // operand set of the odd tiles (PIPE)
      uint64_t ahi_lin = ahi_lin0, alo_lin = alo_lin0, ahi_seg = ahi_seg0, alo_seg = alo_seg0;                           // descriptors of the tile being issued
      uint32_t acc_base = tmem;                                                                                          // accumulator column block of the stage being issued
      const uint64_t bdesc0 = make_desc(smem_u32(ring), sbo1, rb);
      const uint32_t stage_u = (uint32_t)p.stage_bytes >> 4, region_u = (uint32_t)p.region_bytes >> 4;        // descriptor address units (16 B)
      const uint32_t tile_u2 = sbo2, ys_u = (uint32_t)p.YS * row_u1;                                                 // 16 groups * sbo2 / 16; image-row stride
      const int nst = p.nstages, P = p.P, T1 = p.T1, T2 = p.T2, KH = p.KH, KW = p.KW, KS1 = p.KS1;
      const int ks_last = (p.Ch - (P - 1) * CPR) / KE, ks_full = CPR / KE;
      uint32_t st = 0, rphase = 0;                               // ring slot being consumed (persists across tiles)
      const bool prof = PROF && a.prof != nullptr && blockIdx.x == 0;
      long long tp = prof ? clock64() : 0, acc8 = 0, acc9 = 0, acc10 = 0;
      auto tick = [&](int slot) {   // counters live in registers; a global read-modify-write here would distort the timeline
        if (PROF && prof) { const long long now = clock64(); const long long d = now - tp; tp = now; if (slot == 8) acc8 += d; else if (slot == 9) acc9 += d; else acc10 += d; }
      };
      // wait until the chunk AFTER the one in slot `st` has landed (no-op when there is none: end of this CTA's work)
      const bool resident = p.resident != 0;
      bool wskip = false;                                        // resident weights already in place (every tile after the first)
      auto wait_next = [&](bool has_next) {
        if (has_next && !wskip) {
          uint32_t ns = st + 1, nph = rphase;
          if (ns == (uint32_t)nst) { if (resident) return; ns = 0; nph ^= 1; }
          mbar_wait(bar(BAR_FULL) + 8u * ns, nph);
          tc_fence_after();
        }
      };
      // issue the k-steps of the chunk in slot `st` against T M-tiles (concat product N' = 2N, then the lo product, per k-step);
      // the next chunk's barrier is polled before the last M-tile's instructions so its latency hides behind queued MMAs
      auto issue_chunk = [&](uint64_t ah, uint64_t al, uint32_t tile_u, uint32_t dcols, int T, int ksn, uint32_t id2, uint32_t id1,
                             uint32_t first_acc, bool has_next) {
        const uint64_t bd = bdesc0 + st * stage_u;
        uint32_t d = acc_base;
        // Straight-line blocks: the issuing thread's operands live in vector registers and every distinct value costs an R2UR move
        // per use inside a loop body, so k-steps are unrolled at compile time (descriptor + immediate) and M-tiles go two per
        // iteration; the next chunk's barrier is polled before the last block so its latency hides behind queued MMAs.
        if (T == 1) {
          const uint32_t dl = d + (dcols >> 1);
          switch (ksn) {
            case 4:
              mma_k<F16>(d, ah, bd, id2, first_acc);     mma_k<F16>(dl, al, bd, id1, 1);
              mma_k<F16>(d, ah + 2, bd + 2, id2, 1);     mma_k<F16>(dl, al + 2, bd + 2, id1, 1);
              wait_next(has_next);
              mma_k<F16>(d, ah + 4, bd + 4, id2, 1);     mma_k<F16>(dl, al + 4, bd + 4, id1, 1);
              mma_k<F16>(d, ah + 6, bd + 6, id2, 1);     mma_k<F16>(dl, al + 6, bd + 6, id1, 1);
              break;
            case 3: wait_next(has_next); mma_tiles<F16, 3, 1>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
            case 2: wait_next(has_next); mma_tiles<F16, 2, 1>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
            default: wait_next(has_next); mma_tiles<F16, 1, 1>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
          }
        } else {
          auto tiles = [&](int n) {                            // n = 1 or 2 M-tiles at the current position
            if (n == 2) {
              switch (ksn) {
                case 4: mma_tiles<F16, 4, 2>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
                case 3: mma_tiles<F16, 3, 2>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
                case 2: mma_tiles<F16, 2, 2>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
                default: mma_tiles<F16, 1, 2>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
              }
            } else {
              switch (ksn) {
                case 4: mma_tiles<F16, 4, 1>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
                case 3: mma_tiles<F16, 3, 1>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
                case 2: mma_tiles<F16, 2, 1>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
                default: mma_tiles<F16, 1, 1>(d, dcols, ah, al, tile_u, bd, id2, id1, first_acc); break;
              }
            }
            ah += n * tile_u; al += n * tile_u; d += n * dcols;
          };
          int t = 0;
          for (; t + 2 <= T - 1; t += 2) tiles(2);
          for (; t < T - 1; ++t) tiles(1);
          wait_next(has_next);                                 // behind all but the last tile's queued MMAs
          tiles(1);
        }
        if (!resident) tc_commit(bar(BAR_EMPTY) + 8u * st);    // frees the slot when these MMAs have read it
        if (++st == (uint32_t)nst) { st = 0; rphase ^= 1; }
      };

      // the same with the M-tile count and the k-steps per chunk known at compile time (the BASELINE level shapes): one straight-line
      // block per chunk, nothing but the tap's base descriptors changes between chunks
      auto issue_ct = [&](auto Tc, auto KSc, uint64_t ah, uint64_t al, uint32_t tile_u, uint32_t dcols, uint32_t id2, uint32_t id1,
                          uint32_t first_acc, bool has_next) {
        constexpr int T = decltype(Tc)::value, KS = decltype(KSc)::value;
        const uint64_t bd = bdesc0 + st * stage_u;
        if constexpr (T == 1) {
          constexpr int H = (KS + 1) / 2;
          mma_tiles<F16, H, 1>(acc_base, dcols, ah, al, tile_u, bd, id2, id1, first_acc);
          wait_next(has_next);
          if constexpr (H < KS) mma_tiles<F16, KS, 1, H>(acc_base, dcols, ah, al, tile_u, bd, id2, id1, first_acc);
        } else {
          mma_tiles<F16, KS, T - 1>(acc_base, dcols, ah, al, tile_u, bd, id2, id1, first_acc);
          wait_next(has_next);
          mma_tiles<F16, KS, 1>(acc_base + (T - 1) * dcols, dcols, ah + (uint64_t)((T - 1) * tile_u), al + (uint64_t)((T - 1) * tile_u), tile_u, bd, id2, id1, first_acc);
        }
        if (!resident) tc_commit(bar(BAR_EMPTY) + 8u * st);
        if (++st == (uint32_t)nst) { st = 0; rphase ^= 1; }
      };
      auto stage2_ct = [&](auto Tc, auto KSc) {
        uint32_t first_acc = 0, row_u = 0;
        for (int ky = 0; ky < KH; ++ky, row_u += ys_u) {
          uint32_t tap_u = row_u;
          for (int kx = 0; kx < KW; ++kx, tap_u += row_u1) {
            uint32_t pan_u = tap_u;
            for (int pn = 0; pn < P; ++pn, pan_u += region_u) {
              issue_ct(Tc, KSc, ahi_seg + pan_u, alo_seg + pan_u, tile_u2, tile_cols2, id2N2, idN2, first_acc, true);
              first_acc = 1;
            }
          }
        }
      };
      // Stage 2 of a geometry known at compile time (the BASELINE levels): every descriptor is `base + constant`, so the whole stage is one
      // straight-line block of tcgen05.mma with uniform-register adds in between -- no loop counters, no vector-register descriptor
      // arithmetic, no R2UR per chunk.  (Measured: the generic issue paths spend ~270 cycles of dependent scalar work per chunk transition,
      // against ~45 cycles of tensor-pipe time per instruction at N <= 64: tools/umma_probe4.cu.)  The ring protocol is the generic one:
      // the chunk in slot `st` has been waited for by the previous chunk's issue.
      auto stage2_fixed = [&](auto geo, auto res, int it) {
        using G = decltype(geo);
        constexpr int P_ = G::P, T2_ = G::T2;
        constexpr bool RES = decltype(res)::value;               // resident weights: the chunk's slot is its index, a constant too
        const uint64_t ah = ahi_seg0 + ((PIPE && (it & 1)) ? set_u : 0u), al = alo_seg0 + ((PIPE && (it & 1)) ? set_u : 0u);
        if (RES && !wskip) {                                     // first tile of a resident plan: the W2 chunks are still landing
          for (int c = 1; c <= 9 * P_; ++c) mbar_wait(bar(BAR_FULL) + 8u * c, 0);
          tc_fence_after();
        }
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int pn = 0; pn < P_; ++pn) {
              constexpr int KS_ = G::KS;                         // k-steps per chunk (every panel is full at these shapes)
              const uint32_t off = (uint32_t)(ky * G::YS_U + kx * G::ROW_U1 + pn * G::REGION_U);
              const uint64_t bd = RES ? bdesc0 + (uint64_t)((1 + (ky * 3 + kx) * P_ + pn) * G::STAGE_U) : bdesc0 + st * (uint32_t)G::STAGE_U;
#pragma unroll
              for (int tt = 0; tt < T2_; ++tt)
#pragma unroll
                for (int ks = 0; ks < KS_; ++ks) {
                  const uint32_t dd = acc_base + tt * G::DCOLS;
                  mma_k<F16>(dd, ah + (uint64_t)(off + tt * G::TILE_U + 2 * ks), bd + 2 * ks, id2N2, (ky | kx | pn | ks) ? 1u : 0u);
                  mma_k<F16>(dd + G::DCOLS / 2, al + (uint64_t)(off + tt * G::TILE_U + 2 * ks), bd + 2 * ks, idN2, 1u);
                }
              if (!RES) {
                wait_next(true);
                tc_commit(bar(BAR_EMPTY) + 8u * st);
                if (++st == (uint32_t)nst) { st = 0; rphase ^= 1; }
              }
            }
        if (RES) {                                               // the only barrier traffic of a resident stage: the first tile waits for W3's first chunk
          st = (uint32_t)(9 * P_);                               // last W2 chunk: wait_next looks at the slot after it
          wait_next(true);
          st = (uint32_t)(1 + 9 * P_);
        }
      };
      // stages 1 and 3 of the same geometries (1x1 convolutions over plain 128-row tiles)
      auto stage1_fixed = [&](auto geo, auto res, int it) {
        using G = decltype(geo);
        constexpr bool RES = decltype(res)::value;
        const uint64_t ah = ahi_lin0 + ((PIPE && (it & 1)) ? set_u : 0u), al = alo_lin0 + ((PIPE && (it & 1)) ? set_u : 0u);
        const uint64_t bd = RES ? bdesc0 : bdesc0 + st * (uint32_t)G::STAGE_U;
#pragma unroll
        for (int tt = 0; tt < G::T1; ++tt)
#pragma unroll
          for (int ks = 0; ks < G::KS1; ++ks) {
            const uint32_t dd = acc_base + tt * G::DCOLS;
            mma_k<F16>(dd, ah + (uint64_t)(tt * G::LIN_U + 2 * ks), bd + 2 * ks, id2N2, ks ? 1u : 0u);
            mma_k<F16>(dd + G::DCOLS / 2, al + (uint64_t)(tt * G::LIN_U + 2 * ks), bd + 2 * ks, idN2, 1u);
          }
        if (!RES) {
          wait_next(true);
          tc_commit(bar(BAR_EMPTY) + 8u * st);
          if (++st == (uint32_t)nst) { st = 0; rphase ^= 1; }
        } else st = 1;                                           // (stage2_fixed waits for the W2 chunks itself on the first tile)
      };
      auto stage3_fixed = [&](auto geo, auto res, int it, bool last_tile) {
        using G = decltype(geo);
        constexpr bool RES = decltype(res)::value;
        const uint64_t ah = ahi_lin0 + ((PIPE && (it & 1)) ? set_u : 0u), al = alo_lin0 + ((PIPE && (it & 1)) ? set_u : 0u);
#pragma unroll
        for (int pn = 0; pn < G::P; ++pn) {
          const uint64_t bd = RES ? bdesc0 + (uint64_t)((1 + 9 * G::P + pn) * G::STAGE_U) : bdesc0 + st * (uint32_t)G::STAGE_U;
#pragma unroll
          for (int tt = 0; tt < G::T2; ++tt)
#pragma unroll
            for (int ks = 0; ks < G::KS; ++ks) {
              const uint32_t dd = acc_base + tt * G::DCOLS3;
              mma_k<F16>(dd, ah + (uint64_t)(pn * G::REGION_U + tt * G::LIN_U + 2 * ks), bd + 2 * ks, id2N3, (pn | ks) ? 1u : 0u);
              mma_k<F16>(dd + G::DCOLS3 / 2, al + (uint64_t)(pn * G::REGION_U + tt * G::LIN_U + 2 * ks), bd + 2 * ks, idN3, 1u);
            }
          if (!RES) {
            wait_next(!(last_tile && pn == G::P - 1));
            tc_commit(bar(BAR_EMPTY) + 8u * st);
            if (++st == (uint32_t)nst) { st = 0; rphase ^= 1; }
          }
        }
        if (RES) st = 0;                                         // resident: the ring holds exactly one tile's chunks
      };
      using I1 = std::integral_constant<int, 1>; using I2 = std::integral_constant<int, 2>; using I4 = std::integral_constant<int, 4>;
      const int s2class = (ks_last != ks_full) ? 0 : (T2 == 1 && ks_full == 4) ? 1 : (T2 == 2 && ks_full == 4) ? 2 : (T2 == 2 && ks_full == 2) ? 3
                          : (T2 == 4 && ks_full == 2) ? 4 : (T2 == 4 && ks_full == 4) ? 5 : 0;

      // compile-time geometries (descriptor units of 16 bytes): the three conv-coupling levels of BASELINE configs[1] at the plans make_plan picks
      //   L1: Ch 32, 16x16, segments (S 1, NSEG 2, GS 10), 64-byte rows;  L2: Ch 64, 8x8, segments (S 2, GS 10), 128-byte rows;
      //   L3: Ch 128, 4x4, plain layout (WP 6), two channel panels, 128-byte rows
      const int s2fixed = (!F16 || KH != 3 || KW != 3 || ks_last != ks_full) ? 0
          : (SEG && rb == 64 && P == 1 && T2 == 2 && ks_full == 2 && ys_u == GeoL1::YS_U && region_u == GeoL1::REGION_U && tile_u2 == GeoL1::TILE_U && stage_u == GeoL1::STAGE_U && tile_cols2 == GeoL1::DCOLS && T1 == GeoL1::T1 && KS1 == GeoL1::KS1 && tile_cols3 == GeoL1::DCOLS3) ? 1
          : (SEG && rb == 128 && P == 1 && T2 == 1 && ks_full == 4 && ys_u == GeoL2::YS_U && region_u == GeoL2::REGION_U && stage_u == GeoL2::STAGE_U && tile_cols2 == GeoL2::DCOLS && T1 == GeoL2::T1 && KS1 == GeoL2::KS1 && tile_cols3 == GeoL2::DCOLS3) ? 2
          : (!SEG && rb == 128 && P == 2 && T2 == 2 && ks_full == 4 && ys_u == GeoL3::YS_U && region_u == GeoL3::REGION_U && tile_u2 == GeoL3::TILE_U && stage_u == GeoL3::STAGE_U && tile_cols2 == GeoL3::DCOLS && T1 == GeoL3::T1 && KS1 == GeoL3::KS1 && tile_cols3 == GeoL3::DCOLS3) ? 3 : 0;
      const int cW3 = nchunks_tile - P;                          // first W3 chunk
      auto use_tile = [&](int it) {                              // operand set of tile `it`
        const uint32_t o = (PIPE && (it & 1)) ? set_u : 0u;
        ahi_lin = ahi_lin0 + o; alo_lin = alo_lin0 + o; ahi_seg = ahi_seg0 + o; alo_seg = alo_seg0 + o;
      };
      // ---- stage 1: H1 = W1 x0 over every stored row ----
      auto stage1 = [&](int it) {
        use_tile(it); acc_base = tmem + col1;
        if (PIPE && resident) st = 0;                            // resident weights sit at their chunk index
        mbar_wait(bar(BAR_AREADY), it & 1);
        tc_fence_after();
        tick(10);
        if (s2fixed == 1) { if (resident) stage1_fixed(GeoL1{}, std::true_type{}, it); else stage1_fixed(GeoL1{}, std::false_type{}, it); }
        else if (s2fixed == 2) stage1_fixed(GeoL2{}, std::false_type{}, it);
        else if (s2fixed == 3) stage1_fixed(GeoL3{}, std::false_type{}, it);
        else issue_chunk(ahi_lin, alo_lin, lin_u, tile_cols2, T1, KS1, id2N2, idN2, 0, true);
        tc_commit(bar(BAR_ACC1));
        tick(9);
      };
      // ---- stage 2: KH x KW taps as shifted operand views ----
      auto stage2 = [&](int it) {
        use_tile(it); acc_base = tmem + col2;
        if (PIPE && resident) st = 1;
        mbar_wait(bar(BAR_H1), it & 1);
        tc_fence_after();
        tick(10);
        uint32_t first_acc = 0;
        uint32_t row_u = 0;                                      // ky * YS rows, in descriptor units
        if (s2fixed == 1) { if (resident) stage2_fixed(GeoL1{}, std::true_type{}, it); else stage2_fixed(GeoL1{}, std::false_type{}, it); }
        else if (s2fixed == 2) stage2_fixed(GeoL2{}, std::false_type{}, it);
        else if (s2fixed == 3) stage2_fixed(GeoL3{}, std::false_type{}, it);
        else if (s2class == 1) stage2_ct(I1{}, I4{});
        else if (s2class == 2) stage2_ct(I2{}, I4{});
        else if (s2class == 3) stage2_ct(I2{}, I2{});
        else if (s2class == 4) stage2_ct(std::integral_constant<int, 4>{}, I2{});
        else if (s2class == 5) stage2_ct(std::integral_constant<int, 4>{}, I4{});
        else
        for (int ky = 0; ky < KH; ++ky, row_u += ys_u) {
          uint32_t tap_u = row_u;                                // + kx rows (8 units each)
          for (int kx = 0; kx < KW; ++kx, tap_u += row_u1) {
            uint32_t pan_u = tap_u;
            for (int pn = 0; pn < P; ++pn, pan_u += region_u) {
              issue_chunk(ahi_seg + pan_u, alo_seg + pan_u, tile_u2, tile_cols2, T2, pn == P - 1 ? ks_last : ks_full, id2N2, idN2, first_acc, true);
              first_acc = 1;
            }
          }
        }
        tc_commit(bar(BAR_ACC2));
        tick(9);
      };
      // ---- stage 3: h = W3 H2 ----
      auto stage3 = [&](int it) {
        const bool last_tile = it == my_tiles - 1;
        use_tile(it); acc_base = tmem + col3;
        if (PIPE && resident) st = (uint32_t)cW3;
        mbar_wait(bar(BAR_H2), it & 1);
        tc_fence_after();
        tick(10);
        uint32_t pan_u = 0;
        if (s2fixed == 1) { if (resident) stage3_fixed(GeoL1{}, std::true_type{}, it, last_tile); else stage3_fixed(GeoL1{}, std::false_type{}, it, last_tile); }
        else if (s2fixed == 2) stage3_fixed(GeoL2{}, std::false_type{}, it, last_tile);
        else if (s2fixed == 3) stage3_fixed(GeoL3{}, std::false_type{}, it, last_tile);
        else
        for (int pn = 0; pn < P; ++pn, pan_u += region_u)
          issue_chunk(ahi_lin + pan_u, alo_lin + pan_u, lin_u, tile_cols3, T2, pn == P - 1 ? ks_last : ks_full, id2N3, idN3, pn > 0,
                      !(last_tile && pn == P - 1));
        tc_commit(bar(BAR_ACC3));
        tick(9);
      };
      if (!PIPE) {
        if (my_tiles > 0) { mbar_wait(bar(BAR_FULL), 0); tc_fence_after(); }   // first chunk of the first tile; every later chunk is pre-waited
        for (int it = 0; it < my_tiles; ++it) {
          wskip = resident && it > 0;
          stage1(it); stage2(it); stage3(it);
        }
      } else if (my_tiles > 0) {
        if (resident) {                                          // every chunk is loaded once, up front: wait for all of them here, never again
          for (int c = 0; c < nchunks_tile; ++c) mbar_wait(bar(BAR_FULL) + 8u * c, 0);
          tc_fence_after();
          wskip = true;
        } else { mbar_wait(bar(BAR_FULL), 0); tc_fence_after(); }
        stage1(0); stage2(0);
        for (int it = 0; it < my_tiles; ++it) {
          if (it + 1 < my_tiles) stage1(it + 1);
          stage3(it);
          if (it + 1 < my_tiles) stage2(it + 1);
        }
      }
      if (PROF && prof) { a.prof[8] = acc8; a.prof[9] = acc9; a.prof[10] = acc10; }
    }
  } else {
    // ===================== epilogue warps: quadrant = warp % 4 (TMEM lanes 32*quadrant .. +31), group = warp / 4 ========
    // An epilogue "item" is (M-tile, 16 accumulator columns); the kEpiGroups warps of a quadrant take items round-robin.
    const int quad = warp & 3, grp = warp >> 2;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const int row_in_tile = quad * 32 + lane;
    const int ng1 = p.KS1 * KE / 8;                           // groups of 8 channels of x0 per stored row (K zero-padded to whole k-steps)
    constexpr bool kWide = CFPP_TC_WIDE && OCC == 1;                          // epilogue item width of stages 1-2: 32 columns, 16 under the two-CTA register budget
    constexpr int kIW = kWide ? 32 : 16;
    const int nc2 = (p.N2 + kIW - 1) / kIW, nc3 = p.N3 >> 4;  // items per M-tile (stage 3 items are 16 columns)
    const bool prof = PROF && a.prof != nullptr && blockIdx.x == 0 && tid == 0;
    long long tp = 0, pacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    auto tick = [&](int slot) { if (PROF && prof) { const long long now = clock64(); pacc[slot] += now - tp; tp = now; } };
    auto stepX = [&](int it) {
      const uint32_t ph = it & 1;
      const int tile = blockIdx.x + it * gridDim.x;
      const int b0 = tile * p.S, nS = min(p.S, p.B - b0);
      uint8_t* a_hi = a_hi0 + ((PIPE && (it & 1)) ? set_bytes : 0u);   // operand set of this tile
      uint8_t* a_lo = a_lo0 + ((PIPE && (it & 1)) ? set_bytes : 0u);
      (void)ph; (void)b0; (void)nS; (void)a_hi; (void)a_lo;
      // ---- x0 staging -> operand rows (reflect halo / segment overlap applied here) ----
      if (PROF && prof) tp = clock64();
      mbar_wait(bar(BAR_XFULL), ph);
      tick(0);
      if (a.z != nullptr && tid == 0) {                        // fused coupling: z[:, :C/2] = x0, straight from the staged copy (contiguous per sample)
        for (int s = 0; s < nS; ++s)
          bulk_s2g(a.z + (size_t)(b0 + s) * p.Cout * HW, smem_u32(xstage + (size_t)s * xfloats), (uint32_t)(xfloats * 4));
        bulk_commit();
      }
      if (!(PROF && (a.dbg & 2)))
      for (int r = tid; r < p.R; r += kEpiThreads) {
        const uint32_t w = tab_in[r];
        const int s = w >> 24, y = (w >> 12) & 0xFFF, x = w & 0xFFF;
        const float* src = xstage + (size_t)s * xfloats + y * p.W + x;
        const bool live = s < nS;
        for (int j = 0; j < ng1; ++j) {
          float o[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) { const int c = 8 * j + q; o[q] = (c < p.Cin && live) ? src[c * HW] : 0.f; }
          store_group8<F16>(a_hi, a_lo, r, 8 * j, o, rb);
        }
      }
      if (a.z != nullptr && a.add != nullptr) {                // fused coupling: b3 + CN(c) of this tile's samples (read by epilogue 3, ordered by the barrier chain)
        float* sadd = reinterpret_cast<float*>(base + p.off_add) + ((PIPE && (it & 1)) ? p.S * p.N3 : 0);
        for (int i = tid; i < nS * p.N3; i += kEpiThreads) {
          const int s_ = i / p.N3, c_ = i - s_ * p.N3;
          sadd[i] = c_ < p.Cout ? sb3[c_] + __ldg(a.add + (size_t)(b0 + s_) * p.Cout + c_) : 0.f;
        }
      }
      fence_async_smem();
      if (a.z != nullptr && tid == 0) bulk_wait_read();        // the staging buffer may be refilled once the bulk store has read it
      mbar_arrive(bar(BAR_XEMPTY));
      mbar_arrive(bar(BAR_AREADY));
      tick(1);
    };
    auto stepE1 = [&](int it) {
      const uint32_t ph = it & 1;
      const int tile = blockIdx.x + it * gridDim.x;
      const int b0 = tile * p.S, nS = min(p.S, p.B - b0);
      uint8_t* a_hi = a_hi0 + ((PIPE && (it & 1)) ? set_bytes : 0u);   // operand set of this tile
      uint8_t* a_lo = a_lo0 + ((PIPE && (it & 1)) ? set_bytes : 0u);
      (void)ph; (void)b0; (void)nS; (void)a_hi; (void)a_lo;
      // ---- epilogue 1: H1 = relu(acc + b1) for every stored row ----
      mbar_wait(bar(BAR_ACC1), ph);
      tc_fence_after();
      tick(2);
      if (!(PROF && (a.dbg & 1)))
      for (int item = grp, t = 0, ci = grp; item < p.T1 * nc2; item += kEpiGroups, ci += kEpiGroups) {
        while (ci >= nc2) { ci -= nc2; ++t; }                  // item -> (M-tile t, column item ci) without a division
        const int c0 = ci * kIW;
        const int r = t * 128 + row_in_tile;
        float* g1 = nullptr;                                     // training forward: this stored row's source pixel (halo rows rewrite their mirror pixel's value)
        if (PROF && a.h1_out != nullptr && r < p.R) {
          const uint32_t w = tab_in[r];
          const int s = w >> 24;
          if (s < nS) g1 = a.h1_out + ((size_t)(b0 + s) * p.Ch + c0) * HW + ((w >> 12) & 0xFFF) * p.W + (w & 0xFFF);
        }
        if (a.bias1_b == nullptr)                                // two call sites: the shared-memory bias keeps LDS addressing
          epilogue_to_operand<F16, kWide, PROF>(tmem + col1 + lane_base + t * 2 * p.N2, p.N2, c0, sb1, a_hi, a_lo, p.region_bytes, r, r < p.R, rb, g1, HW);
        else
          epilogue_to_operand<F16, kWide, PROF>(tmem + col1 + lane_base + t * 2 * p.N2, p.N2, c0,
                                                a.bias1_b + (size_t)min(b0 + (r < p.R ? (int)(tab_in[r] >> 24) : 0), p.B - 1) * p.Ch, a_hi, a_lo, p.region_bytes, r, r < p.R, rb, g1, HW);
      }
      fence_async_smem();
      tc_fence_before();
      mbar_arrive(bar(BAR_H1));
      tick(3);
    };
    auto stepE2 = [&](int it) {
      const uint32_t ph = it & 1;
      const int tile = blockIdx.x + it * gridDim.x;
      const int b0 = tile * p.S, nS = min(p.S, p.B - b0);
      uint8_t* a_hi = a_hi0 + ((PIPE && (it & 1)) ? set_bytes : 0u);   // operand set of this tile
      uint8_t* a_lo = a_lo0 + ((PIPE && (it & 1)) ? set_bytes : 0u);
      (void)ph; (void)b0; (void)nS; (void)a_hi; (void)a_lo;
      // ---- epilogue 2: H2 = relu(acc + b2) at the accumulator's own row index ----
      mbar_wait(bar(BAR_ACC2), ph);
      tc_fence_after();
      tick(4);
      if (!(PROF && (a.dbg & 1)))
      for (int item = grp, t = 0, ci = grp; item < p.T2 * nc2; item += kEpiGroups, ci += kEpiGroups) {
        while (ci >= nc2) { ci -= nc2; ++t; }
        const int c0 = ci * kIW;
        const int m = t * 128 + row_in_tile;
        float* g2 = nullptr;
        if (PROF && a.h2_out != nullptr) {
          const uint32_t w = tab_out[m];
          const int s = (w >> 24) & 0x7F;
          if ((w >> 31) != 0 && s < nS) g2 = a.h2_out + ((size_t)(b0 + s) * p.Ch + c0) * HW + ((w >> 12) & 0xFFF) * p.W + (w & 0xFFF);
        }
        epilogue_to_operand<F16, kWide, PROF>(tmem + col2 + lane_base + t * 2 * p.N2, p.N2, c0, sb2, a_hi, a_lo, p.region_bytes, m, (tab_out[m] >> 31) != 0, rb, g2, HW);
      }
      fence_async_smem();
      tc_fence_before();
      mbar_arrive(bar(BAR_H2));
      tick(5);
    };
    auto stepE3 = [&](int it) {
      const uint32_t ph = it & 1;
      const int tile = blockIdx.x + it * gridDim.x;
      const int b0 = tile * p.S, nS = min(p.S, p.B - b0);
      uint8_t* a_hi = a_hi0 + ((PIPE && (it & 1)) ? set_bytes : 0u);   // operand set of this tile
      uint8_t* a_lo = a_lo0 + ((PIPE && (it & 1)) ? set_bytes : 0u);
      (void)ph; (void)b0; (void)nS; (void)a_hi; (void)a_lo;
      // ---- epilogue 3: h = acc + b3 -> HBM (NCHW) ----
      // fused coupling: the x1 values of an item are fetched one item ahead, the first item's before the wait for the stage-3 MMAs, so the
      // HBM latency of these loads hides behind the tensor pipe instead of sitting between the accumulator load and the transform
      const int half = p.Cout >> 1, nck = half >> 3;             // items of 8 (t, r) channel pairs; half % 8 == 0 (host)
      float x1c[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      auto fetch_x1 = [&](int t, int ci, float (&dst)[8]) {
        const uint32_t w = tab_out[t * 128 + row_in_tile];
        const int s = (w >> 24) & 0x7F;
        if ((w >> 31) != 0 && s < nS) {
          const float* xs1 = a.x + (size_t)(b0 + s) * p.x_bstride + (size_t)(half + (ci << 3)) * HW + ((w >> 12) & 0xFFF) * p.W + (w & 0xFFF);
#pragma unroll
          for (int i = 0; i < 8; ++i) dst[i] = __ldg(xs1 + (size_t)i * HW);
        }
      };
      if (a.z != nullptr && grp < p.T2 * nck) { int t = 0, ci = grp; while (ci >= nck) { ci -= nck; ++t; } fetch_x1(t, ci, x1c); }
      mbar_wait(bar(BAR_ACC3), ph);
      tc_fence_after();
      tick(6);
      if (a.z != nullptr) {
        // ---- fused affine coupling: (t | r) = acc + b3 (+ CN(c)); z0 = x0, z1 = x1 * exp(2 tanh(r / 2)) + t; ldj = sum log-scale ----
        float* lsp = reinterpret_cast<float*>(base + p.off_ls) + grp * (p.T2 * 128);
        for (int item = grp, t = 0, ci = grp; item < p.T2 * nck; item += kEpiGroups, ci += kEpiGroups) {
          while (ci >= nck) { ci -= nck; ++t; }
          const int k0 = ci << 3;
          const int m = t * 128 + row_in_tile;
          const uint32_t w = tab_out[m];
          const int s = (w >> 24) & 0x7F, y = (w >> 12) & 0xFFF, x = w & 0xFFF;
          const bool valid = (w >> 31) != 0 && s < nS;
          const size_t bb = (size_t)(b0 + (valid ? s : 0));
          const int pix = y * p.W + x;
          const uint32_t taddr = tmem + col3 + lane_base + t * 2 * p.N3;
          float vt[8], ut[8], vr[8], ur[8];
          tmem_ld8(taddr + k0, vt); tmem_ld8(taddr + p.N3 + k0, ut);
          tmem_ld8(taddr + half + k0, vr); tmem_ld8(taddr + p.N3 + half + k0, ur);
          float x1v[8], x1n[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int i = 0; i < 8; ++i) x1v[i] = x1c[i];
          if (item + kEpiGroups < p.T2 * nck) {                  // the next item's x1 goes in flight under this item's transform
            int t2 = t, c2 = ci + kEpiGroups; while (c2 >= nck) { c2 -= nck; ++t2; }
            fetch_x1(t2, c2, x1n);
          }
          tmem_ld_wait();
          if (valid) {
            float* zd = a.z + (bb * p.Cout + k0) * HW + pix;
            const float* ob = a.add ? reinterpret_cast<const float*>(base + p.off_add) + ((PIPE && (it & 1)) ? p.S * p.N3 : 0) + s * p.N3 : sb3;   // output bias: b3 (+ CN(c) of the sample)
            float lsum = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float tt = (F16 ? fmaf(ut[i], kLoInv, vt[i]) : vt[i] + ut[i]) + ob[k0 + i];
              const float rr = (F16 ? fmaf(ur[i], kLoInv, vr[i]) : vr[i] + ur[i]) + ob[half + k0 + i];
              // log_s = 2 tanh(r/2) = 2 (1 - e^-r) / (1 + e^-r) with the SFU exponential (relative error ~2^-21; tanh saturates in fp32 beyond
              // |r| = 18, the clamp keeps e^-r finite): ~12 instructions instead of ~60 for tanhf + expf on the epilogue warps' critical path
              const float e = __expf(-fminf(fmaxf(rr, -30.f), 30.f));
              const float ls = 2.0f * __fdividef(1.0f - e, 1.0f + e);
              zd[(size_t)(half + i) * HW] = fmaf(x1v[i], __expf(ls), tt);
              lsum += ls;
            }
            lsp[m] += lsum;
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) x1c[i] = x1n[i];
        }
        tc_fence_before();
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        {   // per-sample sum: one warp per sample, lanes stride over the accumulator rows in a fixed order, then a shuffle tree -- deterministic
          const float* l0 = reinterpret_cast<const float*>(base + p.off_ls);
          const int nrows = p.T2 * 128;
          for (int smp = warp; smp < nS; smp += kEpiWarps) {
            float acc = 0.f;
            for (int m = lane; m < nrows; m += 32) {
              const uint32_t w = tab_out[m];
              if ((w >> 31) != 0 && (int)((w >> 24) & 0x7F) == smp)
                for (int g2 = 0; g2 < kEpiGroups; ++g2) acc += l0[g2 * nrows + m];
            }
            acc = warp_sum(acc);
            if (lane == 0) a.ldj[b0 + smp] = acc + (a.logp_c ? a.logp_scale * a.logp_c[b0 + smp] : 0.f);
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        for (int i = tid; i < kEpiGroups * p.T2 * 128; i += kEpiThreads) reinterpret_cast<float*>(base + p.off_ls)[i] = 0.f;
      } else if (!(PROF && (a.dbg & 1)))
      for (int item = grp, t = 0, ci = grp; item < p.T2 * nc3; item += kEpiGroups, ci += kEpiGroups) {
        while (ci >= nc3) { ci -= nc3; ++t; }
        const int c0 = ci << 4;
        const int m = t * 128 + row_in_tile;
        const uint32_t w = tab_out[m];
        const int s = (w >> 24) & 0x7F, y = (w >> 12) & 0xFFF, x = w & 0xFFF;
        const bool valid = (w >> 31) != 0 && s < nS;
        float* dst = a.h + ((size_t)(b0 + (valid ? s : 0)) * p.Cout) * HW + y * p.W + x;
        const uint32_t taddr = tmem + col3 + lane_base + t * 2 * p.N3;
        float v[16], u[16];
        tmem_ld16(taddr + c0, v);
        tmem_ld16(taddr + p.N3 + c0, u);
        tmem_ld_wait();
        if (valid) {
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (c0 + i < p.Cout) dst[(size_t)(c0 + i) * HW] = (F16 ? fmaf(u[i], kLoInv, v[i]) : v[i] + u[i]) + sb3[c0 + i];
        }
      }
      tc_fence_before();
      tick(7);
    };
    if (!PIPE) {
      for (int it = 0; it < my_tiles; ++it) { stepX(it); stepE1(it); stepE2(it); stepE3(it); }
    } else if (my_tiles > 0) {
      // two tiles interleaved: the MMA stage an epilogue step waits for was issued two steps earlier (see the kernel's header comment)
      stepX(0); stepE1(0);
      for (int it = 0; it < my_tiles; ++it) {
        if (it + 1 < my_tiles) stepX(it + 1);
        stepE2(it);
        if (it + 1 < my_tiles) stepE1(it + 1);
        stepE3(it);
      }
    }
    if (PROF && prof) {
#pragma unroll
      for (int i = 0; i < 8; ++i) a.prof[i] = pacc[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
}

// One-time weight repack: torch-layout conv weights -> the chunk stream the producer copies verbatim into the ring.
// chunk c (stride stage_bytes): [hi image: N rows x 128 B, K-major SW128][lo image], row n / column k of the image =
//   c == 0           : W1[n][k]                                   (N = N2, k < Cin)
//   1 + tap*P + pn   : W2[n][pn*32 + k][ky][kx]                   (N = N2)
//   1 + taps*P + pn  : W3[n][pn*32 + k]                           (N = N3, rows >= Cout zero)
__global__ void pack_tc_kernel(const float* __restrict__ w1, const float* __restrict__ w2, const float* __restrict__ w3, uint8_t* __restrict__ out,
                               int Cin, int Ch, int Cout, int KH, int KW, int P, int N2, int N3, int stage_bytes, int w1_stride, int f16, int rb) {
  const int taps = KH * KW;
  const int CPR = f16 ? rb >> 1 : 32;
  const int nchunks = 1 + taps * P + P;
  const int c = blockIdx.x;
  if (c >= nchunks) return;
  const int N = c < 1 + taps * P ? N2 : N3;
  uint8_t* img = out + (size_t)c * stage_bytes;
  for (int i = threadIdx.x; i < N * CPR; i += blockDim.x) {
    const int n = i / CPR, k = i % CPR;
    float v = 0.f;
    if (c == 0) { if (n < Ch && k < Cin) v = w1[(size_t)n * w1_stride + k]; }
    else if (c < 1 + taps * P) {
      const int tap = (c - 1) / P, pn = (c - 1) % P, ci = pn * CPR + k;
      if (n < Ch && ci < Ch) v = w2[((size_t)n * Ch + ci) * taps + tap];
    } else {
      const int pn = c - 1 - taps * P, ci = pn * CPR + k;
      if (n < Cout && ci < Ch) v = w3[(size_t)n * Ch + ci];
    }
    if (f16) {
      const uint32_t off = row_off(n, k >> 3, rb) + ((k & 7) << 1);
      const float vc = fminf(fmaxf(v, -65504.f), 65504.f);
      const __half hi = __float2half_rn(vc);
      *reinterpret_cast<__half*>(img + off) = hi;
      *reinterpret_cast<__half*>(img + (size_t)N * rb + off) = __float2half_rn((vc - __half2float(hi)) * kLoScale);
    } else {
      const uint32_t off = sw128(n, k);
      *reinterpret_cast<float*>(img + off) = v;
      *reinterpret_cast<float*>(img + (size_t)N * 128 + off) = tf32_lo(v);
    }
  }
}

// ---- host-side geometry ------------------------------------------------------------------------------------------------
static int env_int(const char* name, int dflt) { const char* v = getenv(name); return v && *v ? atoi(v) : dflt; }

// operand kind of this process: 1 = scaled fp16 pairs (default), 0 = tf32 pairs (CFPP_TC_KIND=tf32)
static int tc_kind() {
  static int k = -1;
  if (k < 0) { const char* v = getenv("CFPP_TC_KIND"); k = (v && strcmp(v, "tf32") == 0) ? 0 : 1; }
  return k;
}

// operand row bytes: the fp16 kind stores <= 32 channels in 64-byte rows (SWIZZLE_64B) -- half the shared memory of a padded 128-byte row
static int row_bytes(int kind, int Cin, int Ch) { return (kind == 1 && Ch <= 32 && Cin <= 32 && env_int("CFPP_TC_RB64", 1)) ? 64 : 128; }

static bool make_plan_occ(Plan& p, double& waste_out, int occ, int pipe, int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, long long x_bstride, int sms) {
  const int max_s = env_int("CFPP_TC_MAXS", 32);
  const int kind = tc_kind(), rb = row_bytes(kind, Cin, Ch), CPR = kind ? rb >> 1 : 32, KE = kind ? 16 : 8;
  if (!((KH == 1 || KH == 3) && (KW == 1 || KW == 3))) return false;
  if ((KH == 3 && H < 2) || (KW == 3 && W < 2)) return false;
  if (Ch % 16 != 0 || Ch < 16 || Ch > 128 || Cin < 1 || Cin > CPR || Cout < 1 || Cout > 128) return false;
  if ((Cin * H * W) % 4 != 0 || x_bstride % 4 != 0) return false;      // 16-byte bulk copies of x0
  p = Plan{};
  p.B = B; p.Cin = Cin; p.Ch = Ch; p.Cout = Cout; p.H = H; p.W = W; p.KH = KH; p.KW = KW; p.x_bstride = x_bstride;
  p.kind = kind; p.rb = rb; p.occ = occ; p.pipe = pipe;
  sms *= occ;                                                            // resident CTA slots
  const int tmem_cols = 512 / occ;
  p.P = (Ch + CPR - 1) / CPR; p.KS1 = (Cin + KE - 1) / KE; p.N2 = Ch; p.N3 = (Cout + 15) / 16 * 16;
  p.HP = H + KH - 1; p.WP = W + KW - 1;
  p.stage_bytes = 2 * p.N2 * rb;
  const int HW = H * W;
  // dynamic shared memory per CTA: 227 KB alone; two co-resident CTAs share the SM's 228 KB less 1 KB reserved per CTA; minus alignment slack
  const int kSmemMax = (occ == 1 ? 227 * 1024 : (228 * 1024) / 2 - 1024) - 1024;
  const int bias_bytes = (2 * p.N2 + p.N3) * 4, bar_bytes = BAR_COUNT * 8 + 16;
  double best_cost = 1e30; Plan best{}; bool found = false;
  for (int seg = 0; seg <= 1; ++seg) {
    if (seg && (W % 8 != 0)) continue;
    for (int S = 1; S <= max_s && S <= B; ++S) {
      Plan q = p; q.seg = seg; q.S = S;
      if (seg) {
        q.NSEG = W / 8; q.GS = 8 + KW - 1; q.YS = S * q.NSEG * q.GS;
        q.R = q.HP * S * q.NSEG * q.GS; q.NG = H * S * q.NSEG; q.T2 = (q.NG + 15) / 16;
      } else {
        q.NSEG = 1; q.GS = 8; q.YS = q.WP; q.RPS = q.HP * q.WP;
        q.R = S * q.RPS;
        const int mmax = (S - 1) * q.RPS + (H - 1) * q.WP + W;          // accumulator rows that can be pixels
        q.T2 = (mmax + 127) / 128; q.NG = q.T2 * 16;
      }
      q.T1 = (q.R + 127) / 128;
      if (q.T1 * 2 * q.N2 > tmem_cols || q.T2 * 2 * q.N2 > tmem_cols || q.T2 * 2 * q.N3 > tmem_cols) break;
      if (pipe && q.T1 * 2 * q.N2 + q.T2 * 2 * q.N2 + q.T2 * 2 * q.N3 > tmem_cols) break;   // three disjoint accumulator column blocks
      q.region_bytes = ((q.R + 15) / 16 * 16) * rb;          // multiple of 1024 bytes: every region starts on a swizzle-atom boundary
      // operand rows the MMAs may touch (garbage rows included) must stay inside this CTA's shared memory
      const int set_bytes = 2 * q.P * q.region_bytes;           // one (hi | lo) operand set; PIPE keeps two (tile parity)
      q.off_ring = (pipe ? 2 : 1) * set_bytes;
      const int xbytes = (S * Cin * HW * 4 + 127) / 128 * 128;
      const int tab_bytes = (q.R + q.T2 * 128) * 4;
      const int ls_bytes = epi_warps(occ) / 4 * q.T2 * 128 * 4;          // per (epilogue group, accumulator row) log-scale partials of the fused coupling
      const int add_bytes = (pipe ? 2 : 1) * S * q.N3 * 4;                 // PIPE: one per tile parity (stepX of tile i+1 runs before epilogue 3 of tile i)
      const int fixed = q.off_ring + xbytes + bias_bytes + tab_bytes + ls_bytes + add_bytes + bar_bytes + 256;
      int nst = (kSmemMax - fixed) / q.stage_bytes;
      if (nst < 2) break;
      const int nchunks = 1 + KH * KW * q.P + q.P;
      q.resident = (nchunks <= kMaxStages && nst >= nchunks && env_int("CFPP_TC_RESIDENT", 1)) ? 1 : 0;
      if (q.resident) nst = nchunks;
      if (nst > kMaxStages) nst = kMaxStages;
      q.nstages = nst;
      const int reach1 = q.T1 * 128 * rb;                                                     // stage 1 / 3 tiles
      const int reach2 = ((q.T2 * 16 - 1) * q.GS + (KH - 1) * q.YS + (KW - 1) + 8) * rb;       // last group of the last tap
      const int reach = (reach1 > reach2 ? reach1 : reach2) + (2 * q.P - 1) * q.region_bytes + (pipe ? set_bytes : 0);
      if (reach > q.off_ring + nst * q.stage_bytes) continue;
      q.off_stage_x = q.off_ring + nst * q.stage_bytes;
      q.off_bias = q.off_stage_x + xbytes;
      q.off_tab = (q.off_bias + bias_bytes + 15) / 16 * 16;
      q.off_ls = (q.off_tab + tab_bytes + 15) / 16 * 16;
      q.off_add = (q.off_ls + ls_bytes + 15) / 16 * 16;
      q.off_bar = (q.off_add + add_bytes + 15) / 16 * 16;
      q.smem_bytes = q.off_bar + bar_bytes + 1024;
      q.ntiles = (B + S - 1) / S;
      // cost: MMA row-slots per real pixel, plus a penalty when the batch no longer fills the SMs evenly
      const double waste = (double)(q.T2 * 128) / (double)(S * HW);
      const int waves = (q.ntiles + sms - 1) / sms;
      const double imbalance = (double)(waves * sms) / (double)q.ntiles;
      // (a grid that leaves SMs idle pays for them too: at B = 256 the 4x4 level ran 37 two-M-tile CTAs on 148 SMs; 86 one-M-tile CTAs take half the time)
      const double cost = waste * imbalance * (1.0 + 0.02 / S);
      if (cost < best_cost - 1e-9) { best_cost = cost; best = q; found = true; waste_out = waste; }
    }
  }
  if (found) p = best;
  return found;
}

// CFPP_TC_OCC = 1 / 2 forces the residency; default: two CTAs per SM when such a plan exists and wastes at most 30 % more MMA rows.
// CFPP_TC_PIPE = 0 turns the software-pipelined form off; default: used (one CTA per SM) whenever the shape has such a plan (fp16 kind)
// -- since the straight-line issue paths it is ahead of two resident CTAs at the 16x16 and 8x8 levels (0.217 / 0.144 ms against 0.240 / 0.147)
// and it wastes at most 30 % more MMA rows than the best unpipelined plan.
static bool make_plan(Plan& p, int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, long long x_bstride, int sms) {
  const int force = env_int("CFPP_TC_OCC", 0);
  Plan p1, p2, pp; double w1 = 0, w2 = 0, wp = 0;
  const bool ok1 = force != 2 && make_plan_occ(p1, w1, 1, 0, B, Cin, Ch, Cout, H, W, KH, KW, x_bstride, sms);
  const bool ok2 = force != 1 && make_plan_occ(p2, w2, 2, 0, B, Cin, Ch, Cout, H, W, KH, KW, x_bstride, sms);
  const bool okp = force != 2 && tc_kind() == 1 && env_int("CFPP_TC_PIPE", 1) && make_plan_occ(pp, wp, 1, 1, B, Cin, Ch, Cout, H, W, KH, KW, x_bstride, sms);
  if (okp) {
    const double wbest = ok1 && ok2 ? (w1 < w2 ? w1 : w2) : ok1 ? w1 : ok2 ? w2 : wp;
    if (wp <= 1.3 * wbest) { p = pp; return true; }
  }
  if (ok2 && (!ok1 || w2 <= 1.3 * w1)) { p = p2; return true; }
  if (ok1) { p = p1; return true; }
  return false;
}

static Plan g_last_plan;
static long long* g_prof = nullptr;

}  // namespace tc
}  // namespace cfpp
using namespace cfpp;

static bool tc_channels_ok(int Cin, int Ch, int Cout, int KH, int KW) {
  return Ch % 16 == 0 && Ch >= 16 && Ch <= 128 && Cin >= 1 && Cin <= (tc::tc_kind() ? 64 : 32) && Cout >= 1 && Cout <= 128 && (KH == 1 || KH == 3) && (KW == 1 || KW == 3);
}

extern "C" int64_t cfpp_conv_cond_tc_pack_bytes(int Cin, int Ch, int Cout, int KH, int KW) {
  if (!tc_channels_ok(Cin, Ch, Cout, KH, KW)) return -1;
  const int rb = tc::row_bytes(tc::tc_kind(), Cin, Ch), CPR = tc::tc_kind() ? rb >> 1 : 32, P = (Ch + CPR - 1) / CPR;
  return (int64_t)(1 + KH * KW * P + P) * (2 * Ch * rb);
}

extern "C" int cfpp_conv_cond_tc_pack(const float* w1, int w1_stride, const float* w2, const float* w3, void* out,
                                      int Cin, int Ch, int Cout, int KH, int KW, void* stream) {
  CFPP_REQUIRE(cfpp_conv_cond_tc_pack_bytes(Cin, Ch, Cout, KH, KW) > 0, "conv_cond_tc_pack: unsupported channel counts / kernel size");
  const int rb = tc::row_bytes(tc::tc_kind(), Cin, Ch), CPR = tc::tc_kind() ? rb >> 1 : 32, P = (Ch + CPR - 1) / CPR, N2 = Ch, N3 = (Cout + 15) / 16 * 16;
  const int nchunks = 1 + KH * KW * P + P;
  tc::pack_tc_kernel<<<nchunks, 256, 0, (cudaStream_t)stream>>>(w1, w2, w3, (uint8_t*)out, Cin, Ch, Cout, KH, KW, P, N2, N3, 2 * N2 * rb, w1_stride, tc::tc_kind(), rb);
  return check_launch("conv_cond_tc_pack");
}

extern "C" int cfpp_conv_cond_tc_supported(int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, int64_t x_bstride) {
  tc::Plan p;
  return B > 0 && tc::make_plan(p, B, Cin, Ch, Cout, H, W, KH, KW, x_bstride, num_sms()) ? 1 : 0;
}

static int conv_cond_tc_launch(const float* x, int64_t x_bstride, float* h, const void* wpack, const float* b1, const float* bias1_b,
                               const float* b2, const float* b3, float* z, float* ldj, const float* add, const float* logp_c, float logp_scale,
                               int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, void* stream, float* h1_out = nullptr, float* h2_out = nullptr) {
  if (B <= 0) return CFPP_OK;
  tc::Plan p;
  if (!tc::make_plan(p, B, Cin, Ch, Cout, H, W, KH, KW, x_bstride, num_sms())) {
    set_error("conv_cond_tc: shape (Cin %d, Ch %d, Cout %d, %dx%d, k %dx%d) has no tensor-core plan", Cin, Ch, Cout, H, W, KH, KW);
    return CFPP_ERR_UNSUPPORTED;
  }
  CFPP_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(wpack) & 15) == 0, "conv_cond_tc: x / wpack must be 16-byte aligned");
  tc::g_last_plan = p;
  const int P_ = p.P;
  const long long pack_bytes = (long long)(1 + KH * KW * P_ + P_) * (2 * Ch * p.rb);
  tc::Args a{x, h, (const uint8_t*)wpack, b1, b2, b3, bias1_b, z, ldj, add, logp_c, logp_scale, h1_out, h2_out, pack_bytes, tc::env_int("CFPP_TC_REPL", 1), tc::env_int("CFPP_TC_DBG", 0), tc::g_prof};
  const int slots = num_sms() * p.occ;
  const int grid = p.ntiles < slots ? p.ntiles : slots;
  cudaStream_t st = (cudaStream_t)stream;
  using KernelFn = void (*)(const tc::Plan, const tc::Args);
  static const KernelFn kernels[20] = {
      tc::conv_cond_tc_kernel<false, false, false, 1, false>, tc::conv_cond_tc_kernel<false, false, true, 1, false>,
      tc::conv_cond_tc_kernel<false, true, false, 1, false>,  tc::conv_cond_tc_kernel<false, true, true, 1, false>,
      tc::conv_cond_tc_kernel<true, false, false, 1, false>,  tc::conv_cond_tc_kernel<true, false, true, 1, false>,
      tc::conv_cond_tc_kernel<true, true, false, 1, false>,   tc::conv_cond_tc_kernel<true, true, true, 1, false>,
      tc::conv_cond_tc_kernel<false, false, false, 2, false>, tc::conv_cond_tc_kernel<false, false, true, 2, false>,
      tc::conv_cond_tc_kernel<false, true, false, 2, false>,  tc::conv_cond_tc_kernel<false, true, true, 2, false>,
      tc::conv_cond_tc_kernel<true, false, false, 2, false>,  tc::conv_cond_tc_kernel<true, false, true, 2, false>,
      tc::conv_cond_tc_kernel<true, true, false, 2, false>,   tc::conv_cond_tc_kernel<true, true, true, 2, false>,
      // software-pipelined tiles: fp16 kind, one CTA per SM; index 16 + (seg ? 2 : 0) + (profile ? 1 : 0)
      tc::conv_cond_tc_kernel<false, false, true, 1, true>,   tc::conv_cond_tc_kernel<false, true, true, 1, true>,
      tc::conv_cond_tc_kernel<true, false, true, 1, true>,    tc::conv_cond_tc_kernel<true, true, true, 1, true>};
  static DeviceOnce attr_set;
  if (attr_set.first()) {
    for (int i = 0; i < 20; ++i) {
      cudaFuncSetAttribute(kernels[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (i < 8 || i >= 16) ? 227 * 1024 : (228 * 1024) / 2 - 1024);
      cudaFuncSetAttribute(kernels[i], cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
  }
  const bool aux = a.prof != nullptr || h1_out != nullptr || h2_out != nullptr;   // the profile-variant kernels also carry the training outputs
  const int ki = p.pipe ? 16 + (p.seg ? 2 : 0) + (aux ? 1 : 0)
                        : (p.occ == 2 ? 8 : 0) | (p.seg ? 4 : 0) | (aux ? 2 : 0) | (p.kind ? 1 : 0);
  kernels[ki]<<<grid, tc::cta_threads(p.occ), p.smem_bytes, st>>>(p, a);
  return check_launch("conv_cond_tc_fwd");
}

extern "C" int cfpp_conv_cond_tc_fwd(const float* x, int64_t x_bstride, float* h, const void* wpack,
                                     const float* b1, const float* bias1_b, const float* b2, const float* b3,
                                     int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, void* stream) {
  return conv_cond_tc_launch(x, x_bstride, h, wpack, b1, bias1_b, b2, b3, nullptr, nullptr, nullptr, nullptr, 0.f, B, Cin, Ch, Cout, H, W, KH, KW, stream);
}

/* Training forward of the conditioner: h as above plus the post-ReLU activations a1 = relu(W1 x0 + b1), a2 = relu(W2 * a1 + b2) as fp32
 * (B, Ch, H, W), which the backward pass needs (ReLU masks, weight gradients). */
extern "C" int cfpp_conv_cond_tc_train_fwd(const float* x, int64_t x_bstride, float* h, float* a1, float* a2, const void* wpack,
                                           const float* b1, const float* bias1_b, const float* b2, const float* b3,
                                           int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, void* stream) {
  CFPP_REQUIRE(h && a1 && a2, "conv_cond_tc_train: null output");
  return conv_cond_tc_launch(x, x_bstride, h, wpack, b1, bias1_b, b2, b3, nullptr, nullptr, nullptr, nullptr, 0.f, B, Cin, Ch, Cout, H, W, KH, KW, stream, a1, a2);
}

extern "C" int cfpp_conv_cond_tc_coupling_supported(int B, int C, int Ch, int H, int W, int KH, int KW) {
  tc::Plan p;
  return B > 0 && C % 16 == 0 && tc::make_plan(p, B, C / 2, Ch, C, H, W, KH, KW, (long long)C * H * W, num_sms()) ? 1 : 0;
}

extern "C" int cfpp_conv_cond_tc_coupling_fwd(const float* x, float* z, float* ldj, const void* wpack, const float* b1, const float* bias1_b,
                                              const float* b2, const float* b3, const float* add, const float* logp_c, float logp_scale,
                                              int B, int C, int Ch, int H, int W, int KH, int KW, void* stream) {
  CFPP_REQUIRE(C % 16 == 0, "conv_cond_tc_coupling: C=%d must be a multiple of 16 (8 (t, r) channel pairs per epilogue item)", C);
  CFPP_REQUIRE(z && ldj, "conv_cond_tc_coupling: null output");
  return conv_cond_tc_launch(x, (int64_t)C * H * W, nullptr, wpack, b1, bias1_b, b2, b3, z, ldj, add, logp_c, logp_scale, B, C / 2, Ch, C, H, W, KH, KW, stream);
}

/* operand kind of this process: 1 = scaled fp16 pairs (default), 0 = tf32 pairs (environment CFPP_TC_KIND=tf32) */
extern "C" int cfpp_conv_cond_tc_kind(void) { return tc::tc_kind(); }

/* geometry of the last launch, for tests / bench reporting: {seg, S, R, T1, T2, nstages, smem_bytes, ntiles, CTAs per SM, row bytes} */
extern "C" void cfpp_conv_cond_tc_last_plan(int* out8) {   /* 11 values, see cfpp.h */
  const tc::Plan& p = tc::g_last_plan;
  out8[8] = p.occ; out8[9] = p.rb; out8[10] = p.pipe;
  out8[0] = p.seg; out8[1] = p.S; out8[2] = p.R; out8[3] = p.T1; out8[4] = p.T2; out8[5] = p.nstages; out8[6] = p.smem_bytes; out8[7] = p.ntiles;
}

/* debug: device array of 12 int64 cycle counters accumulated by CTA 0 over its tiles (NULL = off):
 * {wait x0, x0 transform, wait stage-1 MMAs, epilogue 1, wait stage-2 MMAs, epilogue 2, wait stage-3 MMAs, epilogue 3,
 *  MMA thread: wait weight chunk, issue, wait operands, spare} */
extern "C" void cfpp_conv_cond_tc_set_profile(void* counters8) { tc::g_prof = (long long*)counters8; }
