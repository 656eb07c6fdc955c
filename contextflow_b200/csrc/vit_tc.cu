// SimpleViT conditioner of TransCoupling (layers/simple_vit.py:91-127; heads = 1, dim_head = 64, dim = mlp_dim = T) on the
// 5th-generation tensor cores, for token widths T <= 64 (the SMAP stack: T = 52, 4 tokens per sample).
//
// Mapping.  A CTA owns 128 token rows (128 / n_tok whole samples) = one MMA M-tile; compute thread r (4 warps) IS token row r for the
// whole network: its residual stream x[T] lives in registers, LayerNorm / GELU / softmax are loops over the thread's own registers
// (no shuffles, no shared-memory round trips), and after a GEMM the thread reads exactly its own accumulator row from TMEM
// (tcgen05.ld 32x32b: lane = row).  Every linear layer (patch embedding, q, k, v, out-projection, the two MLP layers) is a 128 x 64 x 64
// tcgen05.mma group: the thread writes its activation row as one 128-byte K-major operand row (64 channels, fp16 hi / scaled-lo pair,
// SWIZZLE_128B -- the operand arithmetic of conv_cond_tc.cu: 22+ significand bits, three products, two instructions per k-step through
// the stacked [B_hi; B_lo'] weight image); weights stream through a bulk-TMA mbarrier ring, one 16 KB chunk per 64 x 64 matrix.
// Attention (n_tok <= 32 keys, all inside the thread's own warp) runs on the CUDA cores from k / v rows staged in shared memory.
// Roles: warps 0-3 compute (thread = row), warp 4 = MMA issuer, warp 5 = weight producer.
#include <stdlib.h>
#include <cuda_fp16.h>
#include "common.cuh"

namespace cfpp {
namespace vt {

constexpr int kRows = 128, kW = 64;                 // rows per CTA tile; padded feature width (one operand panel)
constexpr int kThreads = 192, kStages = 4;
constexpr int kChunkBytes = 2 * kW * 128;           // [hi image 64 rows x 128 B][lo image]
constexpr int kKVStride = 68;                       // floats per staged k / v row (16-byte aligned, rows of a warp in distinct bank groups)
constexpr float kLoScale = 2048.f, kLoInv = 1.f / 2048.f;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory"); }
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok)
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {       // K-major SWIZZLE_128B, 8-row group stride 1024 bytes
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__host__ __device__ constexpr uint32_t make_idesc(int n) {           // kind::f16: fp16 operands, fp32 accumulate, K-major A and B, M = 128
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
                 "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(taddr) : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
  return pred != 0;
}
// packed fp16 pair {lo half = a, hi half = b}, round to nearest, saturating to the finite range (one F2FP instruction)
__device__ __forceinline__ uint32_t pack_f16x2_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// (hi, lo') fp16 pair of two values: hi = v truncated to 11 significant bits (exact in fp16 over its normal range), lo' = rn((v - hi) * 2^11);
// 4 instructions per element
__device__ __forceinline__ void f16_split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const float ha = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u), hb = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
  hi = pack_f16x2_sat(ha, hb);
  lo = pack_f16x2_sat((a - ha) * kLoScale, (b - hb) * kLoScale);
}
// the thread's activation row (64 channels, zero beyond the live width) -> operand row `row` of the hi / lo regions
__device__ __forceinline__ void store_operand_row(uint8_t* a_hi, uint8_t* a_lo, int row, const float (&v)[kW]) {
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) f16_split2(v[8 * c + 2 * q], v[8 * c + 2 * q + 1], h[q], l[q]);
    const uint32_t off = (uint32_t)row * 128u + (uint32_t)(((c ^ row) & 7) << 4);
    *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}
// the thread's accumulator row of one 64-wide GEMM output: main block [c0, c0+64) + 2^-11 * cross block [c0+64, c0+128)
__device__ __forceinline__ void load_acc_row(uint32_t taddr, float (&o)[kW]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float v[16], u[16];
    tmem_ld16(taddr + 16 * q, v);
    tmem_ld16(taddr + kW + 16 * q, u);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) o[16 * q + i] = fmaf(u[i], kLoInv, v[i]);
  }
}
// LayerNorm (eps 1e-5) over the first T entries of the thread's row.  The row is zero beyond T (invariant of every caller), so the sums
// run over all 64 registers without predicates: the padding adds nothing to the mean and (64 - T) mean^2 to the centred sum of squares,
// which is subtracted.  w / b: shared-memory rows of 64 floats, zero beyond T (the output keeps the invariant).  Four partial sums for ILP.
__device__ __forceinline__ void layer_norm_row(const float (&x)[kW], float (&out)[kW], int T, const float* w, const float* b) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
  for (int i = 0; i < kW; i += 4) { s0 += x[i]; s1 += x[i + 1]; s2 += x[i + 2]; s3 += x[i + 3]; }
  const float mean = ((s0 + s1) + (s2 + s3)) / (float)T;
  float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
#pragma unroll
  for (int i = 0; i < kW; i += 4) {
    const float d0 = x[i] - mean, d1 = x[i + 1] - mean, d2 = x[i + 2] - mean, d3 = x[i + 3] - mean;
    v0 = fmaf(d0, d0, v0); v1 = fmaf(d1, d1, v1); v2 = fmaf(d2, d2, v2); v3 = fmaf(d3, d3, v3);
  }
  const float var = fmaxf(((v0 + v1) + (v2 + v3)) - (float)(kW - T) * mean * mean, 0.f) / (float)T;
  const float rstd = 1.0f / sqrtf(var + 1e-5f);
#pragma unroll
  for (int i = 0; i < kW; i += 4) {
    const float4 w4 = *reinterpret_cast<const float4*>(w + i), b4 = *reinterpret_cast<const float4*>(b + i);
    out[i] = fmaf((x[i] - mean) * rstd, w4.x, b4.x); out[i + 1] = fmaf((x[i + 1] - mean) * rstd, w4.y, b4.y);
    out[i + 2] = fmaf((x[i + 2] - mean) * rstd, w4.z, b4.z); out[i + 3] = fmaf((x[i + 3] - mean) * rstd, w4.w, b4.w);
  }
}
// erf by Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7) with the SFU exponential / reciprocal: ~14 instructions instead of ~40 for erff
__device__ __forceinline__ float erf_as(float x) {
  const float ax = fabsf(x);
  const float t = __fdividef(1.0f, fmaf(0.3275911f, ax, 1.0f));
  const float poly = t * fmaf(t, fmaf(t, fmaf(t, fmaf(t, 1.061405429f, -1.453152027f), 1.421413741f), -0.284496736f), 0.254829592f);
  const float r = 1.0f - poly * __expf(-ax * ax);
  return copysignf(r, x);
}

struct Args {
  const float* x; int64_t x_bstride; float* h; cfpp_vit_desc d; const uint8_t* wpack; int B, S, ntiles, NPT;
};

enum { BAR_FULL = 0, BAR_EMPTY = kStages, BAR_AREADY = 2 * kStages, BAR_ACC, BAR_COUNT };

__global__ void __launch_bounds__(kThreads, 1) vit_tc_kernel(const Args a) {
  extern __shared__ __align__(1024) uint8_t vt_smem_raw[];
  uint8_t* base = vt_smem_raw + ((1024u - (smem_u32(vt_smem_raw) & 1023u)) & 1023u);   // (pointer arithmetic on the shared array keeps the address space)
  uint8_t* a_hi = base;                                       // 128 rows x 128 B
  uint8_t* a_lo = base + kRows * 128;
  uint8_t* ring = base + 2 * kRows * 128;                     // kStages x kChunkBytes
  float* Ks = reinterpret_cast<float*>(ring + kStages * kChunkBytes);   // [128][kKVStride]
  float* Vs = Ks + kRows * kKVStride;
  float* prm = Vs + kRows * kKVStride;                         // parameter rows of 64 floats, zero padded (see fill below)
  const int prm_rows = 7 + a.d.n_tok + 6 * a.d.depth;
  const uint32_t bars = smem_u32(prm + prm_rows * kW);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(prm + prm_rows * kW) + 2 * BAR_COUNT;
  auto bar = [&](int i) { return bars + 8u * i; };
  const cfpp_vit_desc& d = a.d;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int T = d.T, ntok = d.n_tok, depth = d.depth;

  if (tid == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(bar(BAR_FULL + i), 1); mbar_init(bar(BAR_EMPTY + i), 1); }
    mbar_init(bar(BAR_AREADY), kRows); mbar_init(bar(BAR_ACC), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {   // LayerNorm weights / biases, Linear biases and the positional table: rows of 64 floats in shared memory, zero beyond the live width
    //   0 ln0_w  1 ln0_b  2 pe_b  3 ln1_w  4 ln1_b  5 lnf_w  6 lnf_b | 7.. pos[tok] | per layer: lna_w lna_b lnf_w lnf_b b1 b2
    const int64_t lstride = 4 * (int64_t)T + (int64_t)T * 192 + 64 * (int64_t)a.NPT + 2 * (int64_t)T * a.NPT + 2 * (int64_t)a.NPT;
    for (int idx = tid; idx < prm_rows * kW; idx += kThreads) {
      const int row = idx / kW, i = idx - row * kW;
      const float* src = nullptr; int n = T;
      if (row == 0) { src = d.ln0_w; n = d.patch_dim; } else if (row == 1) { src = d.ln0_b; n = d.patch_dim; }
      else if (row == 2) src = d.pe_b; else if (row == 3) src = d.ln1_w; else if (row == 4) src = d.ln1_b;
      else if (row == 5) src = d.lnf_w; else if (row == 6) src = d.lnf_b;
      else if (row < 7 + ntok) src = d.pos + (row - 7) * T;
      else {
        const int l = (row - 7 - ntok) / 6, k = (row - 7 - ntok) % 6;
        const float* Lp = d.layers + l * lstride;
        const float* lnf = Lp + 2 * T + (int64_t)T * 192 + 64 * (int64_t)a.NPT;
        const float* b1 = lnf + 2 * T + (int64_t)T * a.NPT;
        src = k == 0 ? Lp : k == 1 ? Lp + T : k == 2 ? lnf : k == 3 ? lnf + T : k == 4 ? b1 : b1 + a.NPT + (int64_t)T * a.NPT;
      }
      prm[idx] = i < n ? __ldg(src + i) : 0.f;
    }
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int chunks_per_tile = 1 + 6 * depth;                  // patch embedding; per layer q, k, v, out, mlp1, mlp2
  const int my_tiles = (a.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == 5) {
    // ===================== producer: the tile's weight chunks, in consumption order, through the ring =====================
    if (elect_one()) {
      uint32_t st = 0, ph = 0;
      for (int it = 0; it < my_tiles; ++it)
        for (int c = 0; c < chunks_per_tile; ++c) {
          mbar_wait(bar(BAR_EMPTY + st), ph ^ 1);
          mbar_expect_tx(bar(BAR_FULL + st), kChunkBytes);
          bulk_g2s(smem_u32(ring + (size_t)st * kChunkBytes), a.wpack + (size_t)c * kChunkBytes, kChunkBytes, bar(BAR_FULL + st));
          if (++st == kStages) { st = 0; ph ^= 1; }
        }
    }
  } else if (warp == 4) {
    // ===================== MMA issuer: one thread; a GEMM group = 1 or 3 chunks against the resident operand tile =====================
    if (elect_one()) {
      const uint32_t id128 = make_idesc(2 * kW), id64 = make_idesc(kW);
      const uint64_t ah = make_desc(smem_u32(a_hi)), al = make_desc(smem_u32(a_lo)), b0 = make_desc(smem_u32(ring));
      uint32_t st = 0, ph = 0, na = 0;                         // ring slot / phase; A-ready count
      auto group = [&](int nchunks) {
        mbar_wait(bar(BAR_AREADY), na & 1); ++na;
        tc_fence_after();
        for (int c = 0; c < nchunks; ++c) {
          mbar_wait(bar(BAR_FULL + st), ph);
          tc_fence_after();
          const uint64_t bd = b0 + (uint64_t)(st * (kChunkBytes >> 4));
          const uint32_t dd = tmem + c * 2 * kW;               // stacked product -> [dd, dd+128); cross product of the lo activations -> [dd+64, dd+128)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            mma_f16(dd, ah + 2 * ks, bd + 2 * ks, id128, ks ? 1u : 0u);
            mma_f16(dd + kW, al + 2 * ks, bd + 2 * ks, id64, 1u);
          }
          tc_commit(bar(BAR_EMPTY + st));
          if (++st == kStages) { st = 0; ph ^= 1; }
        }
        tc_commit(bar(BAR_ACC));
      };
      for (int it = 0; it < my_tiles; ++it) {
        group(1);                                               // patch embedding
        for (int l = 0; l < depth; ++l) { group(3); group(1); group(1); group(1); }
      }
    }
  } else {
    // ===================== compute threads: thread = token row =====================
    const int r = tid;
    const int HW = d.H * d.W, tw = d.W / d.p2, Cout = T / (d.p1 * d.p2);
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);    // this warp's TMEM lane quadrant
    uint32_t nacc = 0;                                           // ACC barrier uses so far (phase parity)
    auto a_ready = [&]() { fence_async_smem(); mbar_arrive(bar(BAR_AREADY)); };
    auto acc_wait = [&]() { mbar_wait(bar(BAR_ACC), nacc & 1); ++nacc; tc_fence_after(); };
    auto prow = [&](int row) { return prm + row * kW; };
    for (int it = 0; it < my_tiles; ++it) {
      const int tile = blockIdx.x + it * gridDim.x;
      const int b0 = tile * a.S;
      const int s = r / ntok, tok = r - s * ntok;
      const bool live = r < a.S * ntok && b0 + s < a.B;
      const int th = tok / tw, tww = tok - th * tw;
      float x[kW], y[kW];                                        // invariant: entries beyond the live width are zero
      // ---- patchify 'b c (h p1) (w p2) -> b (h w) (p1 p2 c)', LayerNorm(patch_dim), Linear, LayerNorm(T), + positional embedding ----
#pragma unroll
      for (int f = 0; f < kW; ++f) {
        float v = 0.f;
        if (live && f < d.patch_dim) {
          const int c = f % d.Cin, pp = f / d.Cin, i = pp / d.p2, j = pp - i * d.p2;
          v = __ldg(a.x + (int64_t)(b0 + s) * a.x_bstride + (int64_t)c * HW + (th * d.p1 + i) * d.W + (tww * d.p2 + j));
        }
        x[f] = v;
      }
      layer_norm_row(x, y, d.patch_dim, prow(0), prow(1));
      store_operand_row(a_hi, a_lo, r, y);
      a_ready();
      acc_wait();
      load_acc_row(trow, x);
      tc_fence_before();
      {
        const float* pb = prow(2);
#pragma unroll
        for (int i = 0; i < kW; ++i) x[i] += pb[i];
      }
      layer_norm_row(x, x, T, prow(3), prow(4));
      {
        const float* pp = prow(7 + tok);
#pragma unroll
        for (int i = 0; i < kW; ++i) x[i] += pp[i];
      }

      for (int l = 0; l < depth; ++l) {
        const float* lp = prow(7 + ntok + 6 * l);                  // lna_w lna_b lnf_w lnf_b b1 b2
        // ---- attention: x += Wo softmax(q k^T / 8) v ----
        layer_norm_row(x, y, T, lp, lp + kW);
        store_operand_row(a_hi, a_lo, r, y);
        a_ready();
        acc_wait();
        {
          float kv[kW];
          load_acc_row(trow + 2 * kW, kv);                        // k
#pragma unroll
          for (int q = 0; q < 16; ++q) *reinterpret_cast<float4*>(Ks + r * kKVStride + 4 * q) = make_float4(kv[4 * q], kv[4 * q + 1], kv[4 * q + 2], kv[4 * q + 3]);
          load_acc_row(trow + 4 * kW, kv);                        // v
#pragma unroll
          for (int q = 0; q < 16; ++q) *reinterpret_cast<float4*>(Vs + r * kKVStride + 4 * q) = make_float4(kv[4 * q], kv[4 * q + 1], kv[4 * q + 2], kv[4 * q + 3]);
        }
        load_acc_row(trow, y);                                    // q (row r) stays in registers
        tc_fence_before();
        __syncwarp();                                             // the keys / values of a sample are rows of this warp (n_tok divides 32)
        {
          float o[kW];
#pragma unroll
          for (int i = 0; i < kW; ++i) o[i] = 0.f;
          float mx = -INFINITY, den = 0.f;
          const int r0 = r - tok;
          for (int j = 0; j < ntok; ++j) {
            const float* kr = Ks + (r0 + j) * kKVStride;
            float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const float4 k4 = *reinterpret_cast<const float4*>(kr + 4 * q);
              d0 = fmaf(y[4 * q], k4.x, d0); d1 = fmaf(y[4 * q + 1], k4.y, d1); d2 = fmaf(y[4 * q + 2], k4.z, d2); d3 = fmaf(y[4 * q + 3], k4.w, d3);
            }
            const float dot = ((d0 + d1) + (d2 + d3)) * 0.125f;    // dim_head ** -0.5
            if (dot > mx) {                                             // a new running maximum: rescale what was accumulated
              const float corr = __expf(mx - dot);
              den *= corr;
#pragma unroll
              for (int i = 0; i < kW; ++i) o[i] *= corr;
              mx = dot;
            }
            const float pj = __expf(dot - mx);
            den += pj;
            const float* vr = Vs + (r0 + j) * kKVStride;
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const float4 v4 = *reinterpret_cast<const float4*>(vr + 4 * q);
              o[4 * q] = fmaf(pj, v4.x, o[4 * q]); o[4 * q + 1] = fmaf(pj, v4.y, o[4 * q + 1]);
              o[4 * q + 2] = fmaf(pj, v4.z, o[4 * q + 2]); o[4 * q + 3] = fmaf(pj, v4.w, o[4 * q + 3]);
            }
          }
          const float inv = 1.0f / den;
#pragma unroll
          for (int i = 0; i < kW; ++i) o[i] *= inv;
          __syncwarp();                                           // every lane has finished reading k / v before the next layer overwrites them
          store_operand_row(a_hi, a_lo, r, o);
        }
        a_ready();
        acc_wait();
        load_acc_row(trow, y);
        tc_fence_before();
#pragma unroll
        for (int i = 0; i < kW; ++i) x[i] += y[i];
        // ---- MLP: x += W2 gelu(W1 LN(x) + b1) + b2 ----
        layer_norm_row(x, y, T, lp + 2 * kW, lp + 3 * kW);
        store_operand_row(a_hi, a_lo, r, y);
        a_ready();
        acc_wait();
        load_acc_row(trow, y);
        tc_fence_before();
        {
          const float* pb1 = lp + 4 * kW;
#pragma unroll
          for (int i = 0; i < kW; ++i) { const float u = y[i] + pb1[i]; y[i] = 0.5f * u * (1.0f + erf_as(u * 0.70710678118654752440f)); }
        }
        store_operand_row(a_hi, a_lo, r, y);
        a_ready();
        acc_wait();
        load_acc_row(trow, y);
        tc_fence_before();
        {
          const float* pb2 = lp + 5 * kW;
#pragma unroll
          for (int i = 0; i < kW; ++i) x[i] += y[i] + pb2[i];
        }
      }
      layer_norm_row(x, x, T, prow(5), prow(6));
      // ---- un-patchify 'b (h w) (p1 p2 c) -> b c (h p1) (w p2)', c = T / (p1 p2) ----
      if (live) {
#pragma unroll
        for (int f = 0; f < kW; ++f) {
          if (f < T) {
            const int c = f % Cout, pp = f / Cout, i = pp / d.p2, j = pp - i * d.p2;
            a.h[((int64_t)(b0 + s) * Cout + c) * HW + (th * d.p1 + i) * d.W + (tww * d.p2 + j)] = x[f];
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}



// Packed fp32 pairs (Blackwell add / mul / fma .f32x2: two IEEE round-to-nearest operations per issue slot, results identical to scalar code)
__device__ __forceinline__ uint64_t pack2(float a, float b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpack2(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) { uint64_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fsub2(uint64_t a, uint64_t b) { uint64_t r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) { uint64_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ uint64_t splat2(float a) { return pack2(a, a); }
// GELU (erf form) of a pair: the Abramowitz & Stegun erf of erf_as above with the polynomial in packed arithmetic
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

// ---------------------------------------------------------------------------------------------------------------------------------------
// Four threads per token row.  The kernel above keeps a whole 64-wide row in ONE thread: 4 compute warps per SM, one per scheduler, every
// LayerNorm / GELU / operand split a 64-step serial instruction stream with nothing to switch to while a TMEM load, a shared-memory store
// or the MMA round trip is outstanding (ncu r1u: issue slots 19 %, tensor pipe 4 %).  Here 16 compute warps share the tile: warp w serves
// TMEM lane quadrant w % 4 (rows 32 (w % 4) .. +31, the hardware's warp -> lane rule) and column group g = w / 4 (columns 16 g .. +15): the
// row state per thread shrinks to 16 registers, each scheduler holds 4 compute warps, and row-wide quantities cross the four column groups
// through shared memory with a named barrier per quadrant:
//   * LayerNorm: two reductions (sum, centred sum of squares), partials in a double-buffered [4][128] table, combined in a fixed order;
//   * attention: q, k, v rows are staged in shared memory; thread (row, g) computes the FULL 64-wide dot products for the keys j = g, g + 4, ..
//     and publishes the scores; after the quadrant barrier every thread forms the softmax (n_tok <= 32 exponentials, redundantly) and its
//     own 16 columns of sum_j p_j v_j.
// Everything else (operand rows, weight ring, the single MMA issuer, fp16 hi / scaled-lo arithmetic) is the kernel above.
constexpr int kCG = 4, kCW = kW / kCG;              // column groups per row, columns per thread
constexpr int kThreads4 = (4 * kCG + 2) * 32;       // 16 compute warps + MMA issuer + weight producer
constexpr int kStages4 = 3;
constexpr int kSStride = 33;                        // floats per row of the score table (n_tok <= 32)

__device__ __forceinline__ void quad_sync(int quad) { asm volatile("bar.sync %0, %1;" ::"r"(1 + quad), "n"(kCG * 32) : "memory"); }

// sum of `v` over the four column-group threads of a row; `red` = this call's [kCG][kRows] table (callers alternate two tables)
__device__ __forceinline__ float row_sum4(float v, float* red, int r, int g, int quad) {
  red[g * kRows + r] = v;
  quad_sync(quad);
  return (red[r] + red[kRows + r]) + (red[2 * kRows + r] + red[3 * kRows + r]);
}

// LayerNorm over the first T entries of a row spread over four threads (16 columns each, zero beyond T): same padding algebra as above
__device__ __forceinline__ void layer_norm4(const float (&x)[kCW], float (&out)[kCW], int T, const float* w, const float* b, float* red2, int& flip,
                                            int r, int g, int quad) {
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int i = 0; i < kCW; i += 2) { s0 += x[i]; s1 += x[i + 1]; }
  const float mean = row_sum4(s0 + s1, red2 + (flip & 1) * kCG * kRows, r, g, quad) / (float)T; ++flip;
  float v0 = 0.f, v1 = 0.f;
#pragma unroll
  for (int i = 0; i < kCW; i += 2) { const float d0 = x[i] - mean, d1 = x[i + 1] - mean; v0 = fmaf(d0, d0, v0); v1 = fmaf(d1, d1, v1); }
  const float ss = row_sum4(v0 + v1, red2 + (flip & 1) * kCG * kRows, r, g, quad); ++flip;
  const float var = fmaxf(ss - (float)(kW - T) * mean * mean, 0.f) / (float)T;
  const float rstd = rsqrtf(var + 1e-5f);
  const uint64_t m2 = splat2(mean), r2 = splat2(rstd);
#pragma unroll
  for (int i = 0; i < kCW; i += 4) {
    const float4 w4 = *reinterpret_cast<const float4*>(w + i), b4 = *reinterpret_cast<const float4*>(b + i);
    unpack2(ffma2(fmul2(fsub2(pack2(x[i], x[i + 1]), m2), r2), pack2(w4.x, w4.y), pack2(b4.x, b4.y)), out[i], out[i + 1]);
    unpack2(ffma2(fmul2(fsub2(pack2(x[i + 2], x[i + 3]), m2), r2), pack2(w4.z, w4.w), pack2(b4.z, b4.w)), out[i + 2], out[i + 3]);
  }
}
// (hi, lo') fp16 pairs of two values in packed arithmetic: 3 instructions per element
__device__ __forceinline__ void f16_split2p(float a, float b, uint32_t& hi, uint32_t& lo) {
  const float ha = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u), hb = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
  float la, lb;
  unpack2(fmul2(fsub2(pack2(a, b), pack2(ha, hb)), splat2(kLoScale)), la, lb);
  hi = pack_f16x2_sat(ha, hb);
  lo = pack_f16x2_sat(la, lb);
}
// the thread's 16 channels of operand row `row` (two 16-byte chunks of the hi / lo regions)
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
// the thread's 16 columns of its accumulator row: main block + 2^-11 * cross block
__device__ __forceinline__ void load_acc16(uint32_t taddr, int g, float (&o)[kCW]) {
  float v[16], u[16];
  tmem_ld16(taddr + kCW * g, v);
  tmem_ld16(taddr + kW + kCW * g, u);
  tmem_ld_wait();
  const uint64_t k2 = splat2(kLoInv);
#pragma unroll
  for (int i = 0; i < kCW; i += 2) unpack2(ffma2(pack2(u[i], u[i + 1]), k2, pack2(v[i], v[i + 1])), o[i], o[i + 1]);
}

enum { B4_FULL = 0, B4_EMPTY = kStages4, B4_AREADY = 2 * kStages4, B4_ACC, B4_COUNT };

__global__ void __launch_bounds__(kThreads4, 1) vit_tc4_kernel(const Args a) {
  extern __shared__ __align__(1024) uint8_t vt_smem_raw[];
  uint8_t* base = vt_smem_raw + ((1024u - (smem_u32(vt_smem_raw) & 1023u)) & 1023u);
  uint8_t* a_hi = base;                                       // 128 rows x 128 B
  uint8_t* a_lo = base + kRows * 128;
  uint8_t* ring = base + 2 * kRows * 128;                     // kStages4 x kChunkBytes
  float* Ks = reinterpret_cast<float*>(ring + kStages4 * kChunkBytes);   // [128][kKVStride]
  float* Vs = Ks + kRows * kKVStride;
  float* Qs = Vs + kRows * kKVStride;
  float* Sc = Qs + kRows * kKVStride;                         // [128][kSStride] attention scores
  float* red2 = Sc + kRows * kSStride;                        // [2][kCG][128] row-reduction partials
  float* prm = red2 + 2 * kCG * kRows;                        // parameter rows of 64 floats, zero padded
  const int prm_rows = 7 + a.d.n_tok + 6 * a.d.depth;
  int* idx_in = reinterpret_cast<int*>(prm + prm_rows * kW);  // [n_tok][64] element offset of (token, feature) inside a sample of x; -1 beyond patch_dim
  int* idx_out = idx_in + a.d.n_tok * kW;                     // [n_tok][64] the same for the output h; -1 beyond T
  const uint32_t bars = smem_u32(idx_out + a.d.n_tok * kW);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(idx_out + a.d.n_tok * kW) + 2 * B4_COUNT;
  auto bar = [&](int i) { return bars + 8u * i; };
  const cfpp_vit_desc& d = a.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int T = d.T, ntok = d.n_tok, depth = d.depth;
  constexpr int kMmaWarp = 4 * kCG, kProdWarp = 4 * kCG + 1;

  if (tid == 0) {
    for (int i = 0; i < kStages4; ++i) { mbar_init(bar(B4_FULL + i), 1); mbar_init(bar(B4_EMPTY + i), 1); }
    mbar_init(bar(B4_AREADY), kRows * kCG); mbar_init(bar(B4_ACC), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {   // parameter rows, as in the kernel above
    const int64_t lstride = 4 * (int64_t)T + (int64_t)T * 192 + 64 * (int64_t)a.NPT + 2 * (int64_t)T * a.NPT + 2 * (int64_t)a.NPT;
    for (int idx = tid; idx < prm_rows * kW; idx += kThreads4) {
      const int row = idx / kW, i = idx - row * kW;
      const float* src = nullptr; int n = T;
      if (row == 0) { src = d.ln0_w; n = d.patch_dim; } else if (row == 1) { src = d.ln0_b; n = d.patch_dim; }
      else if (row == 2) src = d.pe_b; else if (row == 3) src = d.ln1_w; else if (row == 4) src = d.ln1_b;
      else if (row == 5) src = d.lnf_w; else if (row == 6) src = d.lnf_b;
      else if (row < 7 + ntok) src = d.pos + (row - 7) * T;
      else {
        const int l = (row - 7 - ntok) / 6, k = (row - 7 - ntok) % 6;
        const float* Lp = d.layers + l * lstride;
        const float* lnf = Lp + 2 * T + (int64_t)T * 192 + 64 * (int64_t)a.NPT;
        const float* b1 = lnf + 2 * T + (int64_t)T * a.NPT;
        src = k == 0 ? Lp : k == 1 ? Lp + T : k == 2 ? lnf : k == 3 ? lnf + T : k == 4 ? b1 : b1 + a.NPT + (int64_t)T * a.NPT;
      }
      prm[idx] = i < n ? __ldg(src + i) : 0.f;
    }
  }
  {   // 'b c (h p1) (w p2) -> b (h w) (p1 p2 c)' and its inverse as offset tables: the runtime divisions are paid once per CTA, not per tile
    const int HW_ = d.H * d.W, tw_ = d.W / d.p2, Cout_ = T / (d.p1 * d.p2);
    for (int idx = tid; idx < ntok * kW; idx += kThreads4) {
      const int tok = idx / kW, f = idx - tok * kW;
      const int th = tok / tw_, tww = tok - th * tw_;
      int oi = -1, oo = -1;
      if (f < d.patch_dim) { const int c = f % d.Cin, pp = f / d.Cin, ii = pp / d.p2, j = pp - ii * d.p2; oi = c * HW_ + (th * d.p1 + ii) * d.W + (tww * d.p2 + j); }
      if (f < T) { const int c = f % Cout_, pp = f / Cout_, ii = pp / d.p2, j = pp - ii * d.p2; oo = c * HW_ + (th * d.p1 + ii) * d.W + (tww * d.p2 + j); }
      idx_in[idx] = oi; idx_out[idx] = oo;
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

  const int chunks_per_tile = 1 + 6 * depth;
  const int my_tiles = (a.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == kProdWarp) {
    if (elect_one()) {
      uint32_t st = 0, ph = 0;
      for (int it = 0; it < my_tiles; ++it)
        for (int c = 0; c < chunks_per_tile; ++c) {
          mbar_wait(bar(B4_EMPTY + st), ph ^ 1);
          mbar_expect_tx(bar(B4_FULL + st), kChunkBytes);
          bulk_g2s(smem_u32(ring + (size_t)st * kChunkBytes), a.wpack + (size_t)c * kChunkBytes, kChunkBytes, bar(B4_FULL + st));
          if (++st == kStages4) { st = 0; ph ^= 1; }
        }
    }
  } else if (warp == kMmaWarp) {
    if (elect_one()) {
      const uint32_t id128 = make_idesc(2 * kW), id64 = make_idesc(kW);
      const uint64_t ah = make_desc(smem_u32(a_hi)), al = make_desc(smem_u32(a_lo)), b0 = make_desc(smem_u32(ring));
      uint32_t st = 0, ph = 0, na = 0;
      auto group = [&](int nchunks) {
        mbar_wait(bar(B4_AREADY), na & 1); ++na;
        tc_fence_after();
        for (int c = 0; c < nchunks; ++c) {
          mbar_wait(bar(B4_FULL + st), ph);
          tc_fence_after();
          const uint64_t bd = b0 + (uint64_t)(st * (kChunkBytes >> 4));
          const uint32_t dd = tmem + c * 2 * kW;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            mma_f16(dd, ah + 2 * ks, bd + 2 * ks, id128, ks ? 1u : 0u);
            mma_f16(dd + kW, al + 2 * ks, bd + 2 * ks, id64, 1u);
          }
          tc_commit(bar(B4_EMPTY + st));
          if (++st == kStages4) { st = 0; ph ^= 1; }
        }
        tc_commit(bar(B4_ACC));
      };
      for (int it = 0; it < my_tiles; ++it) {
        group(1);
        for (int l = 0; l < depth; ++l) { group(3); group(1); group(1); group(1); }
      }
    }
  } else {
    // ===================== compute threads: (row, column group) =====================
    const int quad = warp & 3, g = warp >> 2;
    const int r = quad * 32 + lane, c0 = kCW * g;
    const int HW = d.H * d.W, Cout = T / (d.p1 * d.p2);
    const uint32_t trow = tmem + ((uint32_t)(quad * 32) << 16);
    uint32_t nacc = 0;
    int flip = 0;
    auto a_ready = [&]() { fence_async_smem(); mbar_arrive(bar(B4_AREADY)); };
    auto acc_wait = [&]() { mbar_wait(bar(B4_ACC), nacc & 1); ++nacc; tc_fence_after(); };
    auto prow = [&](int row) { return prm + row * kW + c0; };
    for (int it = 0; it < my_tiles; ++it) {
      const int tile = blockIdx.x + it * gridDim.x;
      const int b0 = tile * a.S;
      const int s = r / ntok, tok = r - s * ntok;
      const bool live = r < a.S * ntok && b0 + s < a.B;
      float x[kCW], y[kCW];                                      // invariant: entries beyond the live width are zero
      {
        const float* xs = a.x + (int64_t)(b0 + s) * a.x_bstride;
        const int* oi = idx_in + tok * kW + c0;
#pragma unroll
        for (int i = 0; i < kCW; ++i) { const int o = oi[i]; x[i] = (live && o >= 0) ? __ldg(xs + o) : 0.f; }
      }
      layer_norm4(x, y, d.patch_dim, prow(0), prow(1), red2, flip, r, g, quad);
      store_operand16(a_hi, a_lo, r, g, y);
      a_ready();
      acc_wait();
      load_acc16(trow, g, x);
      tc_fence_before();
      {
        const float* pb = prow(2);
#pragma unroll
        for (int i = 0; i < kCW; ++i) x[i] += pb[i];
      }
      layer_norm4(x, x, T, prow(3), prow(4), red2, flip, r, g, quad);
      {
        const float* pp = prow(7 + tok);
#pragma unroll
        for (int i = 0; i < kCW; ++i) x[i] += pp[i];
      }

      for (int l = 0; l < depth; ++l) {
        const int lrow = 7 + ntok + 6 * l;                         // lna_w lna_b lnf_w lnf_b b1 b2
        // ---- attention: x += Wo softmax(q k^T / 8) v ----
        layer_norm4(x, y, T, prow(lrow), prow(lrow + 1), red2, flip, r, g, quad);
        store_operand16(a_hi, a_lo, r, g, y);
        a_ready();
        acc_wait();
        {
          float t16[kCW];
          load_acc16(trow + 2 * kW, g, t16);                       // k
#pragma unroll
          for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(Ks + r * kKVStride + c0 + 4 * q) = make_float4(t16[4 * q], t16[4 * q + 1], t16[4 * q + 2], t16[4 * q + 3]);
          load_acc16(trow + 4 * kW, g, t16);                       // v
#pragma unroll
          for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(Vs + r * kKVStride + c0 + 4 * q) = make_float4(t16[4 * q], t16[4 * q + 1], t16[4 * q + 2], t16[4 * q + 3]);
          load_acc16(trow, g, t16);                                // q
#pragma unroll
          for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(Qs + r * kKVStride + c0 + 4 * q) = make_float4(t16[4 * q], t16[4 * q + 1], t16[4 * q + 2], t16[4 * q + 3]);
        }
        tc_fence_before();
        quad_sync(quad);                                           // the keys / values of a sample are rows of this quadrant (n_tok divides 32)
        const int r0 = r - tok;
        for (int j = g; j < ntok; j += kCG) {                      // full-width scores of the keys this column group owns
          const float* qr = Qs + r * kKVStride;
          const float* kr = Ks + (r0 + j) * kKVStride;
          float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const float4 q4 = *reinterpret_cast<const float4*>(qr + 4 * q), k4 = *reinterpret_cast<const float4*>(kr + 4 * q);
            d0 = fmaf(q4.x, k4.x, d0); d1 = fmaf(q4.y, k4.y, d1); d2 = fmaf(q4.z, k4.z, d2); d3 = fmaf(q4.w, k4.w, d3);
          }
          Sc[r * kSStride + j] = ((d0 + d1) + (d2 + d3)) * 0.125f;   // dim_head ** -0.5
        }
        quad_sync(quad);
        {
          float o[kCW];
#pragma unroll
          for (int i = 0; i < kCW; ++i) o[i] = 0.f;
          float mx = -INFINITY;
          for (int j = 0; j < ntok; ++j) mx = fmaxf(mx, Sc[r * kSStride + j]);
          float den = 0.f;
          for (int j = 0; j < ntok; ++j) {
            const float pj = __expf(Sc[r * kSStride + j] - mx);
            den += pj;
            const float* vr = Vs + (r0 + j) * kKVStride + c0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 v4 = *reinterpret_cast<const float4*>(vr + 4 * q);
              o[4 * q] = fmaf(pj, v4.x, o[4 * q]); o[4 * q + 1] = fmaf(pj, v4.y, o[4 * q + 1]);
              o[4 * q + 2] = fmaf(pj, v4.z, o[4 * q + 2]); o[4 * q + 3] = fmaf(pj, v4.w, o[4 * q + 3]);
            }
          }
          const float inv = 1.0f / den;
#pragma unroll
          for (int i = 0; i < kCW; ++i) o[i] *= inv;
          store_operand16(a_hi, a_lo, r, g, o);
        }
        a_ready();                                                 // (the MMA group starts only when every thread is past its k / v / score reads)
        acc_wait();
        load_acc16(trow, g, y);
        tc_fence_before();
#pragma unroll
        for (int i = 0; i < kCW; i += 2) unpack2(fadd2(pack2(x[i], x[i + 1]), pack2(y[i], y[i + 1])), x[i], x[i + 1]);
        // ---- MLP: x += W2 gelu(W1 LN(x) + b1) + b2 ----
        layer_norm4(x, y, T, prow(lrow + 2), prow(lrow + 3), red2, flip, r, g, quad);
        store_operand16(a_hi, a_lo, r, g, y);
        a_ready();
        acc_wait();
        load_acc16(trow, g, y);
        tc_fence_before();
        {
          const float* pb1 = prow(lrow + 4);
#pragma unroll
          for (int i = 0; i < kCW; i += 2) gelu2(y[i] + pb1[i], y[i + 1] + pb1[i + 1], y[i], y[i + 1]);
        }
        store_operand16(a_hi, a_lo, r, g, y);
        a_ready();
        acc_wait();
        load_acc16(trow, g, y);
        tc_fence_before();
        {
          const float* pb2 = prow(lrow + 5);
#pragma unroll
          for (int i = 0; i < kCW; i += 2) unpack2(fadd2(pack2(x[i], x[i + 1]), fadd2(pack2(y[i], y[i + 1]), pack2(pb2[i], pb2[i + 1]))), x[i], x[i + 1]);
        }
      }
      layer_norm4(x, x, T, prow(5), prow(6), red2, flip, r, g, quad);
      if (live) {
        float* hs = a.h + (int64_t)(b0 + s) * Cout * HW;
        const int* oo = idx_out + tok * kW + c0;
#pragma unroll
        for (int i = 0; i < kCW; ++i) { const int o = oo[i]; if (o >= 0) hs[o] = x[i]; }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}

static size_t smem_bytes4(int n_tok, int depth) {
  return 1024 + 2 * kRows * 128 + (size_t)kStages4 * kChunkBytes + 3 * (size_t)kRows * kKVStride * 4 + (size_t)kRows * kSStride * 4 +
         (size_t)2 * kCG * kRows * 4 + (size_t)(7 + n_tok + 6 * depth) * kW * 4 + (size_t)2 * n_tok * kW * 4 + B4_COUNT * 8 + 64;
}

// One 64 x 64 weight matrix -> one chunk: [hi image][lo image], rows = output features (zero beyond n_rows), 64 input channels per
// 128-byte row (zero beyond k_cols), SWIZZLE_128B.  w is row-major (out, in) with leading dimension ld (nn.Linear.weight).
__global__ void pack_chunk_kernel(const float* __restrict__ w, int ld, int n_rows, int k_cols, uint8_t* __restrict__ out) {
  for (int i = threadIdx.x; i < kW * kW; i += blockDim.x) {
    const int n = i / kW, k = i % kW;
    const float v = (n < n_rows && k < k_cols) ? w[(size_t)n * ld + k] : 0.f;
    const float vc = fminf(fmaxf(v, -65504.f), 65504.f);
    const __half hi = __float2half_rn(vc);
    const uint32_t off = (uint32_t)n * 128u + (uint32_t)((((k >> 3) ^ n) & 7) << 4) + (uint32_t)((k & 7) << 1);
    *reinterpret_cast<__half*>(out + off) = hi;
    *reinterpret_cast<__half*>(out + kW * 128 + off) = __float2half_rn((vc - __half2float(hi)) * kLoScale);
  }
}

static size_t smem_bytes(int n_tok, int depth) {
  return 1024 + 2 * kRows * 128 + (size_t)kStages * kChunkBytes + 2 * (size_t)kRows * kKVStride * 4 + (size_t)(7 + n_tok + 6 * depth) * kW * 4 +
         BAR_COUNT * 8 + 64;
}

}  // namespace vt
}  // namespace cfpp
using namespace cfpp;

extern "C" int cfpp_vit_tc_supported(int T, int patch_dim, int n_tok, int Cextra) {
  return (T >= 4 && T <= vt::kW && patch_dim >= 1 && patch_dim <= vt::kW && Cextra == 0 && n_tok >= 1 && n_tok <= 32 && 32 % n_tok == 0) ? 1 : 0;
}

extern "C" int64_t cfpp_vit_tc_pack_bytes(int depth) { return (int64_t)(1 + 6 * depth) * vt::kChunkBytes; }

extern "C" int cfpp_vit_tc_pack_chunk(const float* w, int ld, int n_rows, int k_cols, void* out_chunk, void* stream) {
  CFPP_REQUIRE(w && out_chunk && n_rows >= 1 && n_rows <= vt::kW && k_cols >= 1 && k_cols <= vt::kW && ld >= k_cols, "vit_tc_pack_chunk: %d x %d (ld %d)", n_rows, k_cols, ld);
  vt::pack_chunk_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(w, ld, n_rows, k_cols, (uint8_t*)out_chunk);
  return check_launch("vit_tc_pack_chunk");
}

extern "C" int cfpp_vit_tc_fwd(const float* x, int64_t x_bstride, float* h, const cfpp_vit_desc* desc, const void* wpack, int B, void* stream) {
  CFPP_REQUIRE(desc && wpack, "vit_tc: null descriptor / weights");
  const cfpp_vit_desc& d = *desc;
  CFPP_REQUIRE(cfpp_vit_tc_supported(d.T, d.patch_dim, d.n_tok, 0), "vit_tc: T=%d patch_dim=%d n_tok=%d has no tensor-core plan", d.T, d.patch_dim, d.n_tok);
  CFPP_REQUIRE(d.n_tok == (d.H / d.p1) * (d.W / d.p2) && d.patch_dim == d.Cin * d.p1 * d.p2 && d.T % (d.p1 * d.p2) == 0, "vit_tc: inconsistent descriptor");
  CFPP_REQUIRE((reinterpret_cast<uintptr_t>(wpack) & 15) == 0, "vit_tc: wpack must be 16-byte aligned");
  if (B <= 0) return CFPP_OK;
  vt::Args a{x, x_bstride, h, d, (const uint8_t*)wpack, B, vt::kRows / d.n_tok, 0, (d.T + 15) / 16 * 16};
  a.ntiles = (B + a.S - 1) / a.S;
  const int grid = a.ntiles < num_sms() ? a.ntiles : num_sms();
  const size_t smem4 = vt::smem_bytes4(d.n_tok, d.depth);
  if (smem4 <= 227 * 1024) {
    static DeviceHighWater attr4;                               // per device: one process may drive several GPUs
    if (attr4.raise((long long)smem4)) cudaFuncSetAttribute(vt::vit_tc4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4);
    vt::vit_tc4_kernel<<<grid, vt::kThreads4, smem4, (cudaStream_t)stream>>>(a);
    return check_launch("vit_cond_tc_fwd");
  }
  // one thread per token row needs less shared memory: it takes the shapes whose four-threads-per-row tile does not fit
  const size_t smem = vt::smem_bytes(d.n_tok, d.depth);
  CFPP_REQUIRE(smem <= 227 * 1024, "vit_tc: depth %d does not fit the shared-memory parameter table", d.depth);
  static DeviceHighWater attr;
  if (attr.raise((long long)smem)) cudaFuncSetAttribute(vt::vit_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  vt::vit_tc_kernel<<<grid, vt::kThreads, smem, (cudaStream_t)stream>>>(a);
  return check_launch("vit_cond_tc_fwd");
}
