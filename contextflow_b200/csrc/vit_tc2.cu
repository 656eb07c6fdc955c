// SimpleViT conditioner of TransCoupling on the tensor cores, general form: token widths T <= 192 (up to three 64-channel operand
// panels), any number of tokens per sample up to 128 (the ATM stack: T in {36, 72, 144, 152}, 9 / 18 / 36 / 38 tokens).
//
// A CTA owns 128 token rows (whole samples); every linear layer is a set of 128 x 64 x 64 tcgen05.mma groups on fp16 hi / scaled-lo
// operand pairs (fp32 faithful), weights stream through a bulk-TMA ring.  A GEMM with K = T has P = ceil(T / 64) operand panels and
// N = T output chunks: the MMA issuer walks (output chunk, K panel), accumulating the panels of a chunk into one 128-column TMEM block
// (main | scaled cross products); one 16 KB weight chunk per (output chunk, K panel).
//
// Four threads per token row (the layout of vit_tc4 in vit_tc.cu): 16 compute warps share the tile, warp w serves TMEM lane quadrant
// w % 4 and column group g = w / 4, i.e. columns 16 g .. +15 of EVERY 64-wide chunk.  (With one thread per row a scheduler has one compute
// warp and nothing to switch to while a TMEM load or the MMA round trip is outstanding.)  The residual stream is P x 16 registers per
// thread (no row buffer in shared memory: the ring gets the space); row-wide sums cross the four column groups through shared memory under
// a per-quadrant named barrier.  The attention runs on the tensor cores as well: S = q k^T over the whole tile (128 x 128, only a sample's
// own block is used), softmax in registers (32 key columns per thread), O = P v with v^T staged as a B operand; q / k / v and the
// probabilities use the operand panels, which are free between the q,k,v GEMM and the next LayerNorm.  LayerNorm / bias rows of the
// current layer are staged in shared memory once per layer.
#include "vit_tc_helpers.cuh"

namespace cfpp {
namespace vt2 {
using namespace vtx;

constexpr int kRows = 128, kPanels = 3;
constexpr int kMaxStages = 8;                       // ring slots: as many 16 KB weight chunks as the shared memory left by the tile allows
constexpr int kChunkBytes = 2 * kW * 128;           // [hi image 64 rows x 128 B][lo image]
constexpr int kPanelBytes = 2 * kRows * 128;        // hi rows + lo rows of one 64-channel operand panel

struct Args {
  const float* x; int64_t x_bstride; float* h; cfpp_vit_desc d; const uint8_t* wpack; int B, S, ntiles, NPT, P, PD, nstages;
};

enum { BAR_FULL = 0, BAR_EMPTY = kMaxStages, BAR_AREADY = 2 * kMaxStages, BAR_ACC, BAR_COUNT };

constexpr int kCG = 4, kCW = kW / kCG;
constexpr int kThreads5 = (4 * kCG + 2) * 32;

__device__ __forceinline__ uint64_t pack2(float a, float b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpack2(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) { uint64_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fsub2(uint64_t a, uint64_t b) { uint64_t r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) { uint64_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ uint64_t splat2(float a) { return pack2(a, a); }

__device__ __forceinline__ void compute_sync5() { asm volatile("bar.sync 1, 512;" ::: "memory"); }                 // the 512 compute threads
__device__ __forceinline__ void quad_sync5(int quad) { asm volatile("bar.sync %0, 128;" ::"r"(2 + quad) : "memory"); }   // the four warps of a lane quadrant

// sum of `v` over the four column-group threads of row r; `red` = this call's [kCG][kRows] table (callers alternate two tables)
__device__ __forceinline__ float row_sum5(float v, float* red, int r, int g, int quad) {
  red[g * kRows + r] = v;
  quad_sync5(quad);
  return (red[r] + red[kRows + r]) + (red[2 * kRows + r] + red[3 * kRows + r]);
}
// (hi, lo') fp16 pairs of two values in packed arithmetic
__device__ __forceinline__ void f16_split2p(float a, float b, uint32_t& hi, uint32_t& lo) {
  const float ha = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u), hb = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
  float la, lb;
  unpack2(fmul2(fsub2(pack2(a, b), pack2(ha, hb)), splat2(kLoScale)), la, lb);
  hi = pack_f16x2_sat(ha, hb);
  lo = pack_f16x2_sat(la, lb);
}
// the thread's 16 channels of operand row `row` of one panel (two 16-byte pieces of the hi / lo images)
__device__ __forceinline__ void store_operand16(uint8_t* a_hi, uint8_t* a_lo, int row, int g, const float (&v)[kCW]) {
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) f16_split2p(v[8 * c + 2 * q], v[8 * c + 2 * q + 1], h[q], l[q]);
    const uint32_t off = (uint32_t)row * 128u + (uint32_t)((((2 * g + c) ^ row) & 7) << 4);
    *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}
// the thread's 16 columns of its accumulator row of one output chunk: main block + 2^-11 * cross block
__device__ __forceinline__ void load_acc16(uint32_t taddr, int g, float (&o)[kCW]) {
  float v[16], u[16];
  tmem_ld16(taddr + kCW * g, v);
  tmem_ld16(taddr + kW + kCW * g, u);
  tmem_ld_wait();
  const uint64_t k2 = splat2(kLoInv);
#pragma unroll
  for (int i = 0; i < kCW; i += 2) unpack2(ffma2(pack2(u[i], u[i + 1]), k2, pack2(v[i], v[i + 1])), o[i], o[i + 1]);
}
// GELU (erf form) of a pair: erf_as with the polynomial in packed arithmetic
__device__ __forceinline__ void gelu2(float u0, float u1, float& o0, float& o1) {
  const uint64_t u = pack2(u0, u1);
  float t0, t1;
  unpack2(fmul2(u, splat2(0.70710678118654752440f)), t0, t1);
  const float a0 = fabsf(t0), a1 = fabsf(t1);
  const uint64_t ax = pack2(a0, a1);
  float d0, d1;
  unpack2(ffma2(splat2(0.3275911f), ax, splat2(1.0f)), d0, d1);
  const uint64_t t = pack2(__fdividef(1.0f, d0), __fdividef(1.0f, d1));
  uint64_t p = ffma2(t, splat2(1.061405429f), splat2(-1.453152027f));
  p = ffma2(t, p, splat2(1.421413741f));
  p = ffma2(t, p, splat2(-0.284496736f));
  p = ffma2(t, p, splat2(0.254829592f));
  p = fmul2(t, p);
  float e0, e1;
  unpack2(fmul2(ax, ax), e0, e1);
  float r0, r1;
  unpack2(fsub2(splat2(1.0f), fmul2(p, pack2(__expf(-e0), __expf(-e1)))), r0, r1);
  r0 = copysignf(r0, t0); r1 = copysignf(r1, t1);
  const uint64_t hu = fmul2(u, splat2(0.5f));
  unpack2(ffma2(hu, pack2(r0, r1), hu), o0, o1);
}

// maximum of `v` over the four column-group threads of row r (same table protocol as row_sum5)
__device__ __forceinline__ float row_max5(float v, float* red, int r, int g, int quad) {
  red[g * kRows + r] = v;
  quad_sync5(quad);
  return fmaxf(fmaxf(red[r], red[kRows + r]), fmaxf(red[2 * kRows + r], red[3 * kRows + r]));
}
// v^T as the B operand of O = P V (N = 64 value channels, K = 128 keys): key panel kp = r / 64 is a 16 KB block laid out like a weight chunk,
// [hi image: 64 channel rows x 128 B (64 keys)][lo image]; the thread writes its 16 channels of key r (one fp16 per row, SWIZZLE_128B)
__device__ __forceinline__ void store_vt16(uint8_t* vt, int r, int g, const float (&v)[kCW]) {
  const int rk = r & 63;
  uint8_t* hi = vt + (r >> 6) * kChunkBytes;
  uint8_t* lo = hi + kW * 128;
#pragma unroll
  for (int i = 0; i < kCW; i += 2) {
    uint32_t h2, l2;
    f16_split2p(v[i], v[i + 1], h2, l2);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int c = kCW * g + i + e;
      const uint32_t off = (uint32_t)c * 128u + (uint32_t)((((rk >> 3) ^ c) & 7) << 4) + (uint32_t)((rk & 7) << 1);
      *reinterpret_cast<unsigned short*>(hi + off) = (unsigned short)(e ? (h2 >> 16) : (h2 & 0xFFFFu));
      *reinterpret_cast<unsigned short*>(lo + off) = (unsigned short)(e ? (l2 >> 16) : (l2 & 0xFFFFu));
    }
  }
}
// the thread's 32 key columns 32 g .. +31 of probability row `row` as A-operand pieces: key panel g / 2, 16-byte pieces 4 (g % 2) .. +3
__device__ __forceinline__ void store_p32(uint8_t* ops, int row, int g, const float (&pv)[32]) {
  uint8_t* a_hi = ops + (g >> 1) * kPanelBytes;
  uint8_t* a_lo = a_hi + kRows * 128;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) f16_split2p(pv[8 * c + 2 * q], pv[8 * c + 2 * q + 1], h[q], l[q]);
    const uint32_t off = (uint32_t)row * 128u + (uint32_t)((((4 * (g & 1) + c) ^ row) & 7) << 4);
    *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

enum { G_LN0W = 0, G_LN0B, G_PEB, G_LN1W, G_LN1B, G_LNFW, G_LNFB, G_ROWS };

template <int P>
__global__ void __launch_bounds__(kThreads5, 1) vit_tc5_kernel(const Args a) {
  extern __shared__ __align__(1024) uint8_t vt5_smem_raw[];
  uint8_t* base = vt5_smem_raw + ((1024u - (smem_u32(vt5_smem_raw) & 1023u)) & 1023u);   // pointer arithmetic on the shared array keeps the address space (LDS / STS, not generic LD / ST)
  constexpr int PW = P * kW;
  uint8_t* ops = base;                                        // kPanels x [hi 128 rows x 128 B][lo]
  uint8_t* ring = ops + kPanels * kPanelBytes;                // nstages x kChunkBytes
  const int kStages = a.nstages;
  float* red2 = reinterpret_cast<float*>(ring + kStages * kChunkBytes);    // [2][kCG][128] row-reduction partials
  float* lprm = red2 + 2 * kCG * kRows;                       // [6][PW]: lna_w lna_b lnf_w lnf_b b1 b2 of the current layer, zero padded
  float* gprm = lprm + 6 * PW;                                // [G_ROWS][PW]: ln0 w/b (patch_dim wide), pe_b, ln1 w/b, final norm w/b
  int* foff_in = reinterpret_cast<int*>(gprm + G_ROWS * PW);  // [PW] feature part of the patchify offset; -1 beyond patch_dim
  int* foff_out = foff_in + PW;                               // [PW] the same for the output h; -1 beyond T
  const uint32_t bars = smem_u32(foff_out + PW);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(foff_out + PW) + 2 * BAR_COUNT;
  auto bar = [&](int i) { return bars + 8u * i; };
  const cfpp_vit_desc& d = a.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int T = d.T, ntok = d.n_tok, depth = d.depth, PD = a.PD;
  constexpr int kMmaWarp = 4 * kCG, kProdWarp = 4 * kCG + 1;

  if (tid == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(bar(BAR_FULL + i), 1); mbar_init(bar(BAR_EMPTY + i), 1); }
    mbar_init(bar(BAR_AREADY), kRows * kCG); mbar_init(bar(BAR_ACC), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int idx = tid; idx < G_ROWS * PW; idx += kThreads5) {
    const int row = idx / PW, i = idx - row * PW;
    const float* src = row == G_LN0W ? d.ln0_w : row == G_LN0B ? d.ln0_b : row == G_PEB ? d.pe_b : row == G_LN1W ? d.ln1_w : row == G_LN1B ? d.ln1_b
                     : row == G_LNFW ? d.lnf_w : d.lnf_b;
    const int n = row <= G_LN0B ? d.patch_dim : T;
    gprm[idx] = i < n ? __ldg(src + i) : 0.f;
  }
  {   // 'b c (h p1) (w p2) -> b (h w) (p1 p2 c)' and its inverse: offset = token part + feature part; the feature parts as tables
    const int HW_ = d.H * d.W, Cout_ = T / (d.p1 * d.p2);
    for (int f = tid; f < PW; f += kThreads5) {
      int oi = -1, oo = -1;
      if (f < d.patch_dim) { const int c = f % d.Cin, pp = f / d.Cin, ii = pp / d.p2, j = pp - ii * d.p2; oi = c * HW_ + ii * d.W + j; }
      if (f < T) { const int c = f % Cout_, pp = f / Cout_, ii = pp / d.p2, j = pp - ii * d.p2; oo = c * HW_ + ii * d.W + j; }
      foff_in[f] = oi; foff_out[f] = oo;
    }
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int chunks_per_tile = P * PD + depth * (3 * P + P + 2 * P * P);
  const int my_tiles = (a.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == kProdWarp) {
    if (elect_one()) {
      uint32_t st = 0, ph = 0;
      for (int it = 0; it < my_tiles; ++it)
        for (int c = 0; c < chunks_per_tile; ++c) {
          mbar_wait(bar(BAR_EMPTY + st), ph ^ 1);
          mbar_expect_tx(bar(BAR_FULL + st), kChunkBytes);
          bulk_g2s(smem_u32(ring + (size_t)st * kChunkBytes), a.wpack + (size_t)c * kChunkBytes, kChunkBytes, bar(BAR_FULL + st));
          if (++st == (uint32_t)kStages) { st = 0; ph ^= 1; }
        }
    }
  } else if (warp == kMmaWarp) {
    if (elect_one()) {
      const uint32_t id128 = make_idesc(2 * kW), id64 = make_idesc(kW);
      const uint64_t a0 = make_desc(smem_u32(ops)), b0 = make_desc(smem_u32(ring));
      uint32_t st = 0, ph = 0, na = 0;
      auto gemm = [&](int NC, int PK) {                          // NC output chunks x PK operand panels
        mbar_wait(bar(BAR_AREADY), na & 1); ++na;
        tc_fence_after();
        for (int n = 0; n < NC; ++n)
          for (int p = 0; p < PK; ++p) {
            mbar_wait(bar(BAR_FULL + st), ph);
            tc_fence_after();
            const uint64_t bd = b0 + (uint64_t)(st * (kChunkBytes >> 4));
            const uint64_t ah = a0 + (uint64_t)(p * (kPanelBytes >> 4)), al = ah + (uint64_t)((kRows * 128) >> 4);
            const uint32_t dd = tmem + n * 2 * kW;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              mma_f16(dd, ah + 2 * ks, bd + 2 * ks, id128, (p | ks) ? 1u : 0u);
              mma_f16(dd + kW, al + 2 * ks, bd + 2 * ks, id64, 1u);
            }
            tc_commit(bar(BAR_EMPTY + st));
            if (++st == (uint32_t)kStages) { st = 0; ph ^= 1; }
          }
        tc_commit(bar(BAR_ACC));
      };
      for (int it = 0; it < my_tiles; ++it) {
        gemm(P, PD);
        for (int l = 0; l < depth; ++l) {
          gemm(3, P);
          {
            const uint64_t ah = a0, al = a0 + (uint64_t)((kRows * 128) >> 4), bk = a0 + (uint64_t)(kPanelBytes >> 4);
            // S = q k^T: A = q rows (panel 0), B = k rows (panel 1: 128 hi rows | 128 lo rows); main block columns 0-127, cross block 128-255
            mbar_wait(bar(BAR_AREADY), na & 1); ++na;
            tc_fence_after();
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              mma_f16(tmem, ah + 2 * ks, bk + 2 * ks, make_idesc(4 * kW), ks ? 1u : 0u);
              mma_f16(tmem + 2 * kW, al + 2 * ks, bk + 2 * ks, id128, 1u);
            }
            tc_commit(bar(BAR_ACC));
            // O = P v: A = probability rows (key panels 0-1 = operand panels 0-1), B = v^T (panel 2: one chunk-shaped block per key panel); columns 384-511
            mbar_wait(bar(BAR_AREADY), na & 1); ++na;
            tc_fence_after();
#pragma unroll
            for (int kp = 0; kp < 2; ++kp) {
              const uint64_t ph_ = a0 + (uint64_t)(kp * (kPanelBytes >> 4)), pl_ = ph_ + (uint64_t)((kRows * 128) >> 4);
              const uint64_t bv = a0 + (uint64_t)(2 * (kPanelBytes >> 4) + kp * (kChunkBytes >> 4));
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                mma_f16(tmem + 6 * kW, ph_ + 2 * ks, bv + 2 * ks, id128, (kp | ks) ? 1u : 0u);
                mma_f16(tmem + 7 * kW, pl_ + 2 * ks, bv + 2 * ks, id64, 1u);
              }
            }
            tc_commit(bar(BAR_ACC));
          }
          gemm(P, 1); gemm(P, P); gemm(P, P);
        }
      }
    }
  } else {
    // ===================== compute threads: (row, column group) =====================
    const int quad = warp & 3, g = warp >> 2;
    const int r = quad * 32 + lane, c0 = kCW * g;
    const int HW = d.H * d.W, tw = d.W / d.p2, Cout = T / (d.p1 * d.p2);
    const int64_t lstride = 4 * (int64_t)T + (int64_t)T * 192 + 64 * (int64_t)a.NPT + 2 * (int64_t)T * a.NPT + 2 * (int64_t)a.NPT;
    const uint32_t trow = tmem + ((uint32_t)(quad * 32) << 16);
    uint32_t nacc = 0;
    int flip = 0;
    auto a_ready = [&]() { fence_async_smem(); mbar_arrive(bar(BAR_AREADY)); };
    auto acc_wait = [&]() { mbar_wait(bar(BAR_ACC), nacc & 1); ++nacc; tc_fence_after(); };
    auto op_hi = [&](int p) { return ops + p * kPanelBytes; };
    auto op_lo = [&](int p) { return ops + p * kPanelBytes + kRows * 128; };
    // LayerNorm statistics over the first n entries of the row (entries beyond n are zero: they add (PW - n) mean^2 to the centred sum)
    auto ln_stats5 = [&](const float (&x)[P][kCW], int n, float& mean, float& rstd) {
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int c = 0; c < P; ++c)
#pragma unroll
        for (int i = 0; i < kCW; i += 2) { s0 += x[c][i]; s1 += x[c][i + 1]; }
      mean = row_sum5(s0 + s1, red2 + (flip & 1) * kCG * kRows, r, g, quad) / (float)n; ++flip;
      float v0 = 0.f, v1 = 0.f;
#pragma unroll
      for (int c = 0; c < P; ++c)
#pragma unroll
        for (int i = 0; i < kCW; i += 2) { const float d0 = x[c][i] - mean, d1 = x[c][i + 1] - mean; v0 = fmaf(d0, d0, v0); v1 = fmaf(d1, d1, v1); }
      const float ss = row_sum5(v0 + v1, red2 + (flip & 1) * kCG * kRows, r, g, quad); ++flip;
      const float var = fmaxf(ss - (float)(PW - n) * mean * mean, 0.f) / (float)n;
      rstd = rsqrtf(var + 1e-5f);
    };
    // one chunk of the normalised row: out = (x - mean) rstd w + b (w, b rows zero beyond the live width: so is out)
    auto ln_chunk = [&](const float (&x)[kCW], float (&out)[kCW], float mean, float rstd, const float* w, const float* b) {
      const uint64_t m2 = splat2(mean), r2 = splat2(rstd);
#pragma unroll
      for (int i = 0; i < kCW; i += 4) {
        const float4 w4 = *reinterpret_cast<const float4*>(w + i), b4 = *reinterpret_cast<const float4*>(b + i);
        unpack2(ffma2(fmul2(fsub2(pack2(x[i], x[i + 1]), m2), r2), pack2(w4.x, w4.y), pack2(b4.x, b4.y)), out[i], out[i + 1]);
        unpack2(ffma2(fmul2(fsub2(pack2(x[i + 2], x[i + 3]), m2), r2), pack2(w4.z, w4.w), pack2(b4.z, b4.w)), out[i + 2], out[i + 3]);
      }
    };
    // LayerNorm(n) of the row -> operand panels 0 .. np-1
    auto ln_to_operands = [&](const float (&x)[P][kCW], int n, int np, const float* w, const float* b) {
      float mean, rstd;
      ln_stats5(x, n, mean, rstd);
#pragma unroll
      for (int c = 0; c < P; ++c)
        if (c < np) {
          float y[kCW];
          ln_chunk(x[c], y, mean, rstd, w + kW * c + c0, b + kW * c + c0);
          store_operand16(op_hi(c), op_lo(c), r, g, y);
        }
    };
    for (int it = 0; it < my_tiles; ++it) {
      const int tile = blockIdx.x + it * gridDim.x;
      const int b0 = tile * a.S;
      const int s = r / ntok, tok = r - s * ntok;
      const bool live = r < a.S * ntok && b0 + s < a.B;
      const int th = tok / tw, tww = tok - th * tw;
      const int tokoff = th * d.p1 * d.W + tww * d.p2;
      float x[P][kCW];                                           // invariant: entries beyond the live width are zero
      // ---- patchify, LayerNorm(patch_dim) -> operands, Linear, + bias, LayerNorm(T), + positional embedding ----
      {
        const float* xs = a.x + (int64_t)(b0 + s) * a.x_bstride + tokoff;
#pragma unroll
        for (int c = 0; c < P; ++c)
#pragma unroll
          for (int i = 0; i < kCW; ++i) { const int o = foff_in[kW * c + c0 + i]; x[c][i] = (live && o >= 0) ? __ldg(xs + o) : 0.f; }
      }
      ln_to_operands(x, d.patch_dim, PD, gprm + G_LN0W * PW, gprm + G_LN0B * PW);
      a_ready();
      acc_wait();
#pragma unroll
      for (int c = 0; c < P; ++c) {
        load_acc16(trow + c * 2 * kW, g, x[c]);
        const float* pb = gprm + G_PEB * PW + kW * c + c0;
#pragma unroll
        for (int i = 0; i < kCW; ++i) x[c][i] += pb[i];
      }
      tc_fence_before();
      {
        float mean, rstd;
        ln_stats5(x, T, mean, rstd);
#pragma unroll
        for (int c = 0; c < P; ++c) {
          ln_chunk(x[c], x[c], mean, rstd, gprm + G_LN1W * PW + kW * c + c0, gprm + G_LN1B * PW + kW * c + c0);
#pragma unroll
          for (int i = 0; i < kCW; ++i) { const int col = kW * c + c0 + i; if (col < T) x[c][i] += __ldg(d.pos + tok * T + col); }
        }
      }

      for (int l = 0; l < depth; ++l) {
        // ---- this layer's LayerNorm / bias rows -> shared memory ----
        compute_sync5();                                             // everyone is done with the previous layer's rows
        {
          const float* Lp = d.layers + l * lstride;
          const float* lnf = Lp + 2 * T + (int64_t)T * 192 + 64 * (int64_t)a.NPT;
          const float* b1 = lnf + 2 * T + (int64_t)T * a.NPT;
          const float* b2 = b1 + a.NPT + (int64_t)T * a.NPT;
          for (int idx = g * kRows + r; idx < 6 * PW; idx += kRows * kCG) {
            const int k = idx / PW, i = idx - k * PW;
            const float* src = k == 0 ? Lp : k == 1 ? Lp + T : k == 2 ? lnf : k == 3 ? lnf + T : k == 4 ? b1 : b2;
            lprm[idx] = i < T ? __ldg(src + i) : 0.f;
          }
        }
        compute_sync5();
        // ---- attention: x += Wo softmax(q k^T / 8) v ----
        ln_to_operands(x, T, P, lprm, lprm + PW);
        a_ready();
        acc_wait();
        float o[kCW];
        const int r0 = r - tok;
        {
          float t16[kCW];
          load_acc16(trow + 2 * kW, g, t16);                      // k -> B-operand rows (panel 1)
          store_operand16(op_hi(1), op_lo(1), r, g, t16);
          load_acc16(trow + 4 * kW, g, t16);                      // v -> v^T (panel 2)
          store_vt16(ops + 2 * kPanelBytes, r, g, t16);
          load_acc16(trow, g, t16);                               // q -> A-operand rows (panel 0)
          store_operand16(op_hi(0), op_lo(0), r, g, t16);
        }
        tc_fence_before();
        a_ready();
        acc_wait();                                               // S = q k^T
        float pv[32];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float v[16], u[16];
          tmem_ld16(trow + 32 * g + 16 * h, v);
          tmem_ld16(trow + 2 * kW + 32 * g + 16 * h, u);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) pv[16 * h + i] = fmaf(u[i], kLoInv, v[i]) * 0.125f;   // dim_head ** -0.5
        }
        tc_fence_before();
        const int jlo = r0 - 32 * g, jhi = jlo + ntok;            // this thread's key columns i with jlo <= i < jhi belong to the row's sample
        float mx = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i) { if (!(live && i >= jlo && i < jhi)) pv[i] = -INFINITY; mx = fmaxf(mx, pv[i]); }
        mx = row_max5(mx, red2 + (flip & 1) * kCG * kRows, r, g, quad); ++flip;
        if (!live) mx = 0.f;
        float den = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) { pv[i] = __expf(pv[i] - mx); den += pv[i]; }
        den = row_sum5(den, red2 + (flip & 1) * kCG * kRows, r, g, quad); ++flip;
        const float inv = live ? 1.0f / den : 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) pv[i] *= inv;
        store_p32(ops, r, g, pv);
        a_ready();
        acc_wait();                                               // O = P v
        load_acc16(trow + 6 * kW, g, o);
        tc_fence_before();
        store_operand16(op_hi(0), op_lo(0), r, g, o);
        a_ready();
        acc_wait();                                                  // (all compute threads have arrived: nobody still reads k / v)
#pragma unroll
        for (int c = 0; c < P; ++c) {
          float y[kCW];
          load_acc16(trow + c * 2 * kW, g, y);
#pragma unroll
          for (int i = 0; i < kCW; i += 2) unpack2(fadd2(pack2(x[c][i], x[c][i + 1]), pack2(y[i], y[i + 1])), x[c][i], x[c][i + 1]);
        }
        tc_fence_before();
        // ---- MLP: x += W2 gelu(W1 LN(x) + b1) + b2 ----
        ln_to_operands(x, T, P, lprm + 2 * PW, lprm + 3 * PW);
        a_ready();
        acc_wait();
#pragma unroll
        for (int c = 0; c < P; ++c) {
          float y[kCW];
          load_acc16(trow + c * 2 * kW, g, y);
          const float* pb1 = lprm + 4 * PW + kW * c + c0;
#pragma unroll
          for (int i = 0; i < kCW; i += 2) gelu2(y[i] + pb1[i], y[i + 1] + pb1[i + 1], y[i], y[i + 1]);
          store_operand16(op_hi(c), op_lo(c), r, g, y);              // hidden chunk c = operand panel c of the second MLP layer
        }
        tc_fence_before();
        a_ready();
        acc_wait();
#pragma unroll
        for (int c = 0; c < P; ++c) {
          float y[kCW];
          load_acc16(trow + c * 2 * kW, g, y);
          const float* pb2 = lprm + 5 * PW + kW * c + c0;
#pragma unroll
          for (int i = 0; i < kCW; i += 2)
            unpack2(fadd2(pack2(x[c][i], x[c][i + 1]), fadd2(pack2(y[i], y[i + 1]), pack2(pb2[i], pb2[i + 1]))), x[c][i], x[c][i + 1]);
        }
        tc_fence_before();
      }
      // ---- final LayerNorm, un-patchify 'b (h w) (p1 p2 c) -> b c (h p1) (w p2)' ----
      {
        float mean, rstd;
        ln_stats5(x, T, mean, rstd);
        float* hs = a.h + (int64_t)(b0 + s) * Cout * HW + tokoff;
#pragma unroll
        for (int c = 0; c < P; ++c) {
          float y[kCW];
          ln_chunk(x[c], y, mean, rstd, gprm + G_LNFW * PW + kW * c + c0, gprm + G_LNFB * PW + kW * c + c0);
          if (live) {
#pragma unroll
            for (int i = 0; i < kCW; ++i) { const int o = foff_out[kW * c + c0 + i]; if (o >= 0) hs[o] = y[i]; }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}

static size_t fixed_bytes5(int P) {
  const size_t PW = (size_t)P * kW;
  return 1024 + (size_t)kPanels * kPanelBytes + (size_t)2 * kCG * kRows * 4 + (6 + G_ROWS) * PW * 4 + 2 * PW * 4 + BAR_COUNT * 8 + 64;
}
static int stages_for5(int P) {
  const long long left = 227LL * 1024 - (long long)fixed_bytes5(P);
  long long n = left / kChunkBytes;
  return (int)(n > kMaxStages ? kMaxStages : n);
}

}  // namespace vt2
}  // namespace cfpp
using namespace cfpp;

extern "C" int cfpp_vit_tc2_supported(int T, int patch_dim, int n_tok, int Cextra) {
  if (!(T >= 4 && T % 4 == 0 && T <= 192 && patch_dim >= 1 && patch_dim <= T && Cextra == 0 && n_tok >= 1 && n_tok <= vt2::kRows)) return 0;
  return vt2::stages_for5((T + 63) / 64) >= 2 ? 1 : 0;
}

/* chunks of the weight stream: embed (P x PD), then per layer qkv (3 x P), out (P x 1), mlp1 (P x P), mlp2 (P x P); P = ceil(T/64) */
extern "C" int64_t cfpp_vit_tc2_chunks(int T, int patch_dim, int depth) {
  const int P = (T + 63) / 64, PD = (patch_dim + 63) / 64;
  return (int64_t)P * PD + (int64_t)depth * (3 * P + P + 2 * P * P);
}

extern "C" int cfpp_vit_tc2_fwd(const float* x, int64_t x_bstride, float* h, const cfpp_vit_desc* desc, const void* wpack, int B, void* stream) {
  CFPP_REQUIRE(desc && wpack, "vit_tc2: null descriptor / weights");
  const cfpp_vit_desc& d = *desc;
  CFPP_REQUIRE(cfpp_vit_tc2_supported(d.T, d.patch_dim, d.n_tok, 0), "vit_tc2: T=%d patch_dim=%d n_tok=%d has no tensor-core plan", d.T, d.patch_dim, d.n_tok);
  CFPP_REQUIRE(d.n_tok == (d.H / d.p1) * (d.W / d.p2) && d.patch_dim == d.Cin * d.p1 * d.p2 && d.T % (d.p1 * d.p2) == 0, "vit_tc2: inconsistent descriptor");
  CFPP_REQUIRE((reinterpret_cast<uintptr_t>(wpack) & 15) == 0, "vit_tc2: wpack must be 16-byte aligned");
  if (B <= 0) return CFPP_OK;
  vt2::Args a{x, x_bstride, h, d, (const uint8_t*)wpack, B, vt2::kRows / d.n_tok, 0, (d.T + 15) / 16 * 16, (d.T + 63) / 64, (d.patch_dim + 63) / 64, 0};
  a.ntiles = (B + a.S - 1) / a.S;
  a.nstages = vt2::stages_for5(a.P);
  const size_t smem = vt2::fixed_bytes5(a.P) + (size_t)a.nstages * vt2::kChunkBytes;
  const int grid = a.ntiles < num_sms() ? a.ntiles : num_sms();
#define CFPP_VT5(P_) do { static DeviceHighWater attr;           /* per device: one process may drive several GPUs */ \
    if (attr.raise((long long)smem)) cudaFuncSetAttribute(vt2::vit_tc5_kernel<P_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    vt2::vit_tc5_kernel<P_><<<grid, vt2::kThreads5, smem, (cudaStream_t)stream>>>(a); } while (0)
  if (a.P == 1) CFPP_VT5(1); else if (a.P == 2) CFPP_VT5(2); else CFPP_VT5(3);
#undef CFPP_VT5
  return check_launch("vit_cond_tc_fwd");
}
