// Gaussian-mixture log-prob (gmm_tile.cu) as a tensor-core contraction: tcgen05.mma, kind::tf32 with fp32-faithful hi/lo operands.
//
//   comp[b, mk] = -sum_e a (x - m)^2  =  sum_e x^2 (-a)  +  sum_e x (2 a m)  -  sum_e a m^2,        m = mu[mk,e] + c[vm, mk, d(e)]
//
// The first two sums are one GEMM per tile of 128 samples that share a context tuple (gmm_tile.cu's bucketing): samples on M, the
// padded components (N = MK rounded up to 16) on N, K = 2E ([x^2 | x] against [-a ; 2am]).  The last sum depends on the parameters
// and the tuple only; the CTA accumulates it in double while it builds the B operand and subtracts it in the epilogue.
//
// Operands.  Raw latents and a = 1/(2 sigma^2) need fp32 range (sigma = 1e-3 gives a = 5e5, beyond fp16), so both sides are tf32
// pairs, as conv_cond_tc.cu's tf32 kind: hi = v (the tensor core truncates it to tf32), lo = v - trunc_tf32(v), and
//   A*B ~= A_hi*B_hi + A_hi*B_lo + A_lo*B_hi  =  one MMA of A_hi against the stacked [B_hi ; B_lo] (N' = 2N, accumulator columns [0,2N))
//                                                + one MMA of A_lo against B_hi into columns [N,2N);
// the epilogue adds the two column blocks.
//
// Mapping.  A CTA (128 threads, thread t = tile row t = TMEM lane t) owns one tile x one slice of e.  Per chunk of 32 elements it
// writes x^2 and x of its 128 rows (hi, lo: four 16 KB SWIZZLE_128B K-major regions) and -a and 2am of the tile's tuple (two
// stacked [hi ; lo] regions of 2N rows), one thread issues 16 MMAs, and the next chunk's x and parameters are loaded into registers
// while they run.  The shared memory holds one chunk (106 KB at N = 80), so two CTAs share an SM and one converts while the
// other's MMAs run.  The slice's partial sums go to the same [nsplit][slots][MKP] buffer as gmm_tile.cu's tile_kernel, and its
// finish_kernel combines them in a fixed order (no atomics: bit-identical from run to run).
//
// Accuracy guard.  The expansion trades (x-m)^2 for a difference of sums, each as large as S = sum_e a m^2 when x ~ m.  With tf32
// pairs every product carries a relative error of about 2^-22 (the dropped A_lo*B_lo term and the truncation of the lo operands),
// and the fp32 accumulation adds about as much, so the absolute error of comp is below eps * (|comp| + 4 S) with eps = 2^-20: the
// x^2 a and a m^2 sums are each ~S and the cross sum ~2S.  The |comp| part is relative and far inside rtol; the 4 eps S part must
// stay below a tenth of the log-prob tolerance, atol + rtol |out| (atol 1e-3, rtol 1e-4), where |out| >= -(max_k LB[m,k] + log K)
// because comp <= 0 (used only when no logp term is added).  A slice of len elements is held to len / E of that; a slice that
// exceeds it is flagged, and gmm_tile.cu's exact tile_kernel recomputes that slice in place of this kernel's partial sums.
#include "common.cuh"
#include "umma.cuh"
#include "gmm_tc.cuh"

namespace cfpp {
namespace gtc {
using namespace tc;

constexpr int EC = 32;                  // event elements per chunk (one 128-byte operand row)
constexpr int kThreads = 128;
constexpr int kARegion = TS * 128;      // bytes of one A region (x^2 hi, x^2 lo, x hi, x lo)
constexpr float kEps = 1.f / 1048576.f; // 2^-20, see the header
constexpr float kGuardFrac = 0.1f, kAtol = 1e-3f, kRtol = 1e-4f;


__host__ __device__ constexpr int tmem_cols(int N) { return 2 * N <= 32 ? 32 : (2 * N <= 64 ? 64 : (2 * N <= 128 ? 128 : 256)); }
__host__ __device__ constexpr int smem_bytes(int N) { return 1024 + 4 * kARegion + 2 * (2 * N * 128) + TS * 4 + 128 * 4 + 64; }

// NJ = N / 16: thread t builds the B rows of components t/8 + 16 j (j < NJ), elements 4 (t%8) .. +3 of the chunk.
template <int NJ>
__global__ void __launch_bounds__(kThreads, 1) gmm_tc_kernel(const Args a) {
  constexpr int N = 16 * NJ;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ax2h = base;                      // A regions
  uint8_t* ax2l = base + kARegion;
  uint8_t* axh = base + 2 * kARegion;
  uint8_t* axl = base + 3 * kARegion;
  uint8_t* bna = base + 4 * kARegion;        // [-a hi ; -a lo]   2N rows
  uint8_t* bam = bna + 2 * N * 128;          // [2am hi ; 2am lo] 2N rows
  int* bidx = reinterpret_cast<int*>(bam + 2 * N * 128);
  float* cst = reinterpret_cast<float*>(bidx + TS);
  uint64_t* bar_p = reinterpret_cast<uint64_t*>(cst + 128);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_p + 1);
  int* flag = reinterpret_cast<int*>(tmem_slot + 1);

  const int tile = blockIdx.x, split = blockIdx.y;
  if (a.n_tiles && tile >= *a.n_tiles) return;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar = smem_u32(bar_p);
  for (int i = tid; i < TS; i += kThreads) {
    const int slot = tile * TS + i;
    bidx[i] = a.perm ? a.perm[slot] : (slot < a.B ? slot : -1);
  }
  if (tid == 0) {
    *flag = 0;
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  constexpr int kCols = tmem_cols(N);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int key = a.tile_vs ? a.tile_vs[tile] : 0;
  const int vs = a.scale_in_low ? key % a.key_div : key, vm = a.scale_in_low ? key / a.key_div : key;
  const float2* PTv = a.PT + (int64_t)vs * a.EP * a.MKP;
  const float* mrow = a.mtab ? a.mtab + (int64_t)vm * a.mwidth + a.moff : nullptr;
  const int e_begin = split * a.esplit, e_end = min(a.E, e_begin + a.esplit);
  const int nch = (e_end - e_begin + EC - 1) / EC;
  const int q = tid & 7, r0 = tid >> 3;      // A items: rows r0 + 16 i, quad q; B items: components r0 + 16 j, quad q

  float4 xr[8];
  float2 pr[NJ][4];
  float cr[NJ][4];
  double cs[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) cs[j] = 0.0;

  auto load = [&](int c) {
    const int e = e_begin + c * EC + 4 * q;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int b = bidx[r0 + 16 * i];
      xr[i] = (b >= 0 && e < e_end) ? __ldg(reinterpret_cast<const float4*>(a.x + (int64_t)b * a.x_bstride + e)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int mk = r0 + 16 * j;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const bool ok = mk < a.MK && e + u < e_end;
        pr[j][u] = ok ? __ldg(PTv + (int64_t)(e + u) * a.MKP + mk) : make_float2(0.f, 0.f);
        cr[j][u] = (ok && mrow) ? __ldg(mrow + mk * a.D + (e + u) / a.HW) : 0.f;
      }
    }
  };
  auto store4 = [&](uint8_t* hi, uint8_t* lo, int row, float4 v) {
    const uint32_t off = sw128(row, 4 * q);
    *reinterpret_cast<float4*>(hi + off) = v;
    *reinterpret_cast<float4*>(lo + off) = make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w));
  };

  const uint64_t dx2h = make_desc(smem_u32(ax2h), 1024), dx2l = make_desc(smem_u32(ax2l), 1024);
  const uint64_t dxh = make_desc(smem_u32(axh), 1024), dxl = make_desc(smem_u32(axl), 1024);
  const uint64_t dna = make_desc(smem_u32(bna), 1024), dam = make_desc(smem_u32(bam), 1024);
  constexpr uint32_t id2 = make_idesc(2 * N, false), id1 = make_idesc(N, false);

  if (nch > 0) load(0);
  for (int c = 0; c < nch; ++c) {
    if (c > 0) mbar_wait(bar, (c - 1) & 1);                      // the previous chunk's MMAs have read the operands
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 v = xr[i];
      store4(ax2h, ax2l, r0 + 16 * i, make_float4(v.x * v.x, v.y * v.y, v.z * v.z, v.w * v.w));
      store4(axh, axl, r0 + 16 * i, v);
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      float na[4], am[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float m = pr[j][u].x + cr[j][u], av = pr[j][u].y;
        na[u] = -av;
        am[u] = 2.f * av * m;
        cs[j] = fma((double)av * (double)m, (double)m, cs[j]);
      }
      const int mk = r0 + 16 * j;
      const uint32_t off = sw128(mk, 4 * q), offl = sw128(N + mk, 4 * q);
      *reinterpret_cast<float4*>(bna + off) = make_float4(na[0], na[1], na[2], na[3]);
      *reinterpret_cast<float4*>(bna + offl) = make_float4(tf32_lo(na[0]), tf32_lo(na[1]), tf32_lo(na[2]), tf32_lo(na[3]));
      *reinterpret_cast<float4*>(bam + off) = make_float4(am[0], am[1], am[2], am[3]);
      *reinterpret_cast<float4*>(bam + offl) = make_float4(tf32_lo(am[0]), tf32_lo(am[1]), tf32_lo(am[2]), tf32_lo(am[3]));
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < EC / 8; ++ks) {
          mma_k<false>(tmem, dx2h + 2 * ks, dna + 2 * ks, id2, (c | ks) ? 1u : 0u);
          mma_k<false>(tmem + N, dx2l + 2 * ks, dna + 2 * ks, id1, 1u);
          mma_k<false>(tmem, dxh + 2 * ks, dam + 2 * ks, id2, 1u);
          mma_k<false>(tmem + N, dxl + 2 * ks, dam + 2 * ks, id1, 1u);
        }
        tc_commit(bar);
      }
      __syncwarp();
    }
    if (c + 1 < nch) load(c + 1);                                 // overlaps the MMAs just issued
  }

  // the slice's constant term and accuracy guard, per component (8 threads share one)
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    double s = cs[j];
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    const int mk = r0 + 16 * j;
    if (q == 0) {
      cst[mk] = (float)s;
      if (mk < a.MK) {
        const int m = mk / a.K;
        float lbmax = -INFINITY;
        for (int k = 0; k < a.K; ++k) lbmax = fmaxf(lbmax, a.LB[vs * a.MKP + m * a.K + k]);
        const float low = a.has_logp ? 0.f : fmaxf(0.f, -(lbmax + logf((float)a.K)));
        const float allow = kGuardFrac * (kAtol + kRtol * low) * (float)(e_end - e_begin) / (float)a.E;
        if (!(4.f * kEps * (float)s <= allow)) *flag = 1;        // also catches a non-finite sum
      }
    }
  }
  if (nch > 0) mbar_wait(bar, (nch - 1) & 1);
  tc_fence_after();
  __syncthreads();
  if (tid == 0) a.flags[(int64_t)split * a.tiles + tile] = *flag;

  // epilogue: row tid of the accumulator -> partial sums of sample bidx[tid]
  const int b = bidx[tid];
  const uint32_t taddr = tmem + ((uint32_t)(32 * warp) << 16);
  float* dst = a.part + ((int64_t)split * a.slots + (int64_t)tile * TS + tid) * a.MKP;
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    float v[16], u[16];
    tmem_ld16(taddr + 16 * j, v);
    tmem_ld16(taddr + N + 16 * j, u);
    tmem_ld_wait();
    if (b >= 0 && nch > 0) {
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        const int mk = 16 * j + i;
        if (mk < a.MKP)
          *reinterpret_cast<float4*>(dst + mk) = make_float4(v[i] + u[i] - cst[mk], v[i + 1] + u[i + 1] - cst[mk + 1],
                                                             v[i + 2] + u[i + 2] - cst[mk + 2], v[i + 3] + u[i + 3] - cst[mk + 3]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kCols) : "memory");
}

int n_of(int MK) { return (MK + 15) & ~15; }

// Slices of e per tile: the estimated CTA-rounds times the chunks per slice (plus ~2 chunks of fixed cost per CTA), minimised.
int splits_for(int B, int n_keys, int E, int MK) {
  const int nch = (E + EC - 1) / EC;
  const int64_t est_tiles = ((int64_t)B + TS - 1) / TS + (n_keys > 1 ? n_keys / 2 : 0);
  const int occ = smem_bytes(n_of(MK)) * 2 <= 227 * 1024 ? 2 : 1;
  const int64_t slots = (int64_t)num_sms() * occ;
  int best = 1; double best_cost = 1e300;
  for (int ns = 1; ns <= nch; ++ns) {
    const int per = (nch + ns - 1) / ns, eff = (nch + per - 1) / per;
    if (eff != ns) continue;
    const double cost = (double)((est_tiles * ns + slots - 1) / slots) * (per + 2);
    if (cost < best_cost) { best_cost = cost; best = ns; }
  }
  return best;
}

int launch(const Args& a, cudaStream_t st) {
  const int N = a.N;
  const size_t smem = (size_t)smem_bytes(N);
  dim3 grid((unsigned)a.tiles, (unsigned)a.nsplit);
#define CFPP_GTC_LAUNCH(NJV)                                                                                          \
  case NJV: {                                                                                                          \
    static DeviceOnce attr;                                                                                            \
    if (attr.first()) cudaFuncSetAttribute(gmm_tc_kernel<NJV>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(16 * NJV)); \
    gmm_tc_kernel<NJV><<<grid, kThreads, smem, st>>>(a);                                                               \
  } break
  switch (N / 16) {
    CFPP_GTC_LAUNCH(1); CFPP_GTC_LAUNCH(2); CFPP_GTC_LAUNCH(3); CFPP_GTC_LAUNCH(4);
    CFPP_GTC_LAUNCH(5); CFPP_GTC_LAUNCH(6); CFPP_GTC_LAUNCH(7); CFPP_GTC_LAUNCH(8);
    default: set_error("gmm_tc: N=%d", N); return CFPP_ERR_ARG;
  }
#undef CFPP_GTC_LAUNCH
  return check_launch("gmm_tile_tc");
}

}  // namespace gtc
}  // namespace cfpp
