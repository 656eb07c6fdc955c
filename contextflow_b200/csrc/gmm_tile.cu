// Gaussian-mixture log-prob (layers/distributions/gaussian.py:142-161) as a register-tiled contraction.
//
//   comp[b, mk] = sum_e  -a[mk,e] * (x[b,e] - mu[mk,e] - c[b,mk,d(e)])^2          a = 1 / (2 sigma^2)
//   out[b, m]   = logsumexp_k( comp[b, m*K+k] + LB[mk] ) (+ logp term),           LB = logmix - sum_e log sigma - E/2 log 2pi
//
// It has the shape of a GEMM (samples x components, reduced over the event elements e) with a 3-4 instruction inner
// product instead of one FMA, and it is FP32-issue bound, not HBM bound (cfg2: 8 KB of x per sample against 327 680 Gaussian
// evaluations).  The earlier kernel kept 8 samples per CTA and re-read every component's parameters from L2 for each group of
// 8 samples (1.3 MB per CTA): L2-bandwidth bound at ~9 % of the FP32 peak.  Here a CTA owns a tile of 64 samples x all M*K
// components x one slice of e; a thread owns 8 samples x TM components in registers; x and the interleaved (mu, a) parameter
// table stream through shared memory in chunks of 32 elements (cp.async double buffer), so a parameter is read from L2 once
// per 64 samples.  The slices of e give the grid enough CTAs to balance 148 SMs; their partial sums are combined in a fixed
// order by the finishing kernel (deterministic).
//
// Context (embedding-table offsets, model.py:157,162).  Samples are bucketed by their context tuple (counting sort, buckets padded
// to whole tiles), so a tile shares ONE scale context -- it reads that context's (mu, a) table, no transcendental per evaluation --
// and ONE mean-offset row c[mk, d]: the thread adds its TM offsets to mu once per element (they change every HW elements), the
// inner product stays at 3 instructions.  (Bucketing by scale context alone and carrying per-sample mean offsets in registers was
// measured first: 4 instructions per evaluation plus an 8 x TM register reload per channel, 1.5-2.7x slower than this.)
#include "common.cuh"
#include "gmm_tc.cuh"
#include <algorithm>

namespace cfpp {
namespace gt {

constexpr int TS = 64;        // samples per tile
constexpr int EC = 32;        // event elements per shared-memory chunk
constexpr int XS = 36;        // x row stride in floats: 16-byte aligned rows, rows sg + 8 i fall in distinct banks
constexpr int SGS = 8;        // sample groups: thread (sg, mg) owns samples sg + 8 i, i < 8, and components mg*TM .. +TM-1

__device__ float log_mix_t(const float* __restrict__ wrow, int K, int k) {   // as gmm.cu:log_mix (torch Categorical + MixtureSameFamily)
  float mx = -INFINITY;
  for (int i = 0; i < K; ++i) mx = fmaxf(mx, wrow[i]);
  float den = 0.f;
  for (int i = 0; i < K; ++i) den += expf(wrow[i] - mx);
  float psum = 0.f;
  for (int i = 0; i < K; ++i) psum += expf(wrow[i] - mx) / den;
  const float eps = 1.1920928955078125e-07f;
  float lmx = -INFINITY;
  for (int i = 0; i < K; ++i) lmx = fmaxf(lmx, logf(fminf(fmaxf(expf(wrow[i] - mx) / den / psum, eps), 1.f - eps)));
  float lse = 0.f, lk = 0.f;
  for (int i = 0; i < K; ++i) {
    const float l = logf(fminf(fmaxf(expf(wrow[i] - mx) / den / psum, eps), 1.f - eps));
    lse += expf(l - lmx);
    if (i == k) lk = l;
  }
  return lk - (lmx + logf(lse));
}

// table layout: [PT: Vs][EP][MKP] float2 (mu, a)   [LB: Vs][MKP] float      EP = E rounded up to EC, MKP = MK rounded up to 4
// (rows e >= E and columns mk >= MK hold (0, 0): they contribute nothing)
__global__ void prepare_kernel(const float* __restrict__ mG, const float* __restrict__ sG, const float* __restrict__ wG,
                               const float* __restrict__ stab, int swidth, int soff, float2* __restrict__ PT, float* __restrict__ LB,
                               int MK, int MKP, int K, int D, int HW, int EP) {
  __shared__ float red[32];
  const int mk = blockIdx.x, v = blockIdx.y, E = D * HW;
  float acc = 0.f;
  if (mk < MK) {
    const float* so = stab ? stab + (int64_t)v * swidth + soff + (int64_t)mk * D : nullptr;
    for (int e = threadIdx.x; e < EP; e += blockDim.x) {
      float2 o = make_float2(0.f, 0.f);
      if (e < E) {
        const float sc = softplus_f(sG[(int64_t)mk * E + e] + (so ? so[e / HW] : 0.f));
        o = make_float2(mG[(int64_t)mk * E + e], 1.f / (2.f * sc * sc));
        acc += logf(sc);
      }
      PT[((int64_t)v * EP + e) * MKP + mk] = o;
    }
    acc = group_sum(acc, blockDim.x, red);
    if (threadIdx.x == 0) LB[v * MKP + mk] = log_mix_t(wG + (mk / K) * K, K, mk % K) - acc - (float)E * kHalfLog2Pi;
  } else {
    for (int e = threadIdx.x; e < EP; e += blockDim.x) PT[((int64_t)v * EP + e) * MKP + mk] = make_float2(0.f, 0.f);
    if (threadIdx.x == 0) LB[v * MKP + mk] = 0.f;
  }
}

// Single-CTA counting sort of the batch by context tuple; buckets padded to whole tiles of ts samples (perm = -1 in the padding).
// key = ctx[b,0] (one feature) or ctx[b,0] * card1 + ctx[b,1] (two features)
__global__ void __launch_bounds__(1024) bucket_kernel(const int64_t* __restrict__ ctx, int n_ctx, int card1, int B, int NB,
                                                      int ts, int* __restrict__ perm, int* __restrict__ tile_vs, int* __restrict__ n_tiles) {
  extern __shared__ int sh[];
  int* cnt = sh; int* base = sh + NB; int* cur = sh + 2 * NB;
  __shared__ int total_tiles;
  for (int k = threadIdx.x; k < NB; k += blockDim.x) { cnt[k] = 0; cur[k] = 0; }
  __syncthreads();
  auto key_of = [&](int b) -> int {
    int k = (int)ctx[(int64_t)b * n_ctx];
    if (n_ctx == 2) k = k * card1 + (int)ctx[(int64_t)b * n_ctx + 1];
    return k < 0 ? 0 : (k >= NB ? NB - 1 : k);
  };
  for (int b = threadIdx.x; b < B; b += blockDim.x) atomicAdd(&cnt[key_of(b)], 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int k = 0; k < NB; ++k) { base[k] = t; t += (cnt[k] + ts - 1) / ts; }
    total_tiles = t; *n_tiles = t;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < NB; k += blockDim.x) {
    const int nt = (cnt[k] + ts - 1) / ts;
    for (int t = 0; t < nt; ++t) tile_vs[base[k] + t] = k;
  }
  for (int i = threadIdx.x; i < total_tiles * ts; i += blockDim.x) perm[i] = -1;
  __syncthreads();
  // stable within a bucket is not required for the result; atomics give an arbitrary but valid order
  for (int b = threadIdx.x; b < B; b += blockDim.x) { const int k = key_of(b); perm[base[k] * ts + atomicAdd(&cur[k], 1)] = b; }
}

struct Args {
  const float* x; int64_t x_bstride;
  const float2* PT; const float* LB;
  const int* perm; const int* tile_vs; const int* n_tiles;      // NULL: identity order, no context, grid.x tiles; tile_vs holds the tile's context key
  int tile_shift;                                               // buckets hold whole tiles of TS << tile_shift samples (n_tiles, tile_vs count those)
  const int* flags; int ftiles;                                 // non-NULL: tile_kernel only recomputes the slices that gmm_tc flagged ([nsplit][ftiles])
  int key_div, scale_in_low;                                    // key -> (mean context, scale context): two features: (key / key_div, key % key_div); one: (key, key)
  const float* mtab; int mwidth, moff;                          // mean offsets of a tile: mtab + mean_ctx * mwidth + moff + mk * D + d
  float* part;                                                  // [nsplit][slots][MKP]
  const float* logp_c; float logp_scale; float* out;
  int B, M, K, MK, MKP, D, HW, E, EP, esplit, nsplit, slots;
};

__device__ __forceinline__ void cp_async16(void* dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst, const void* src, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int TM, bool OFF>
__global__ void __launch_bounds__(256, 2) tile_kernel(const Args a) {     // <= 128 registers: three 160-thread CTAs per SM at M*K = 80
  extern __shared__ float4 gt_smem4[];
  const int tile = blockIdx.x, split = blockIdx.y;
  if (a.n_tiles && (tile >> a.tile_shift) >= *a.n_tiles) return;
  if (a.flags && !a.flags[(int64_t)split * a.ftiles + (tile >> a.tile_shift)]) return;
  const int MKP = a.MKP;
  float* xs = reinterpret_cast<float*>(gt_smem4);                 // [2][TS][XS]
  float2* ps = reinterpret_cast<float2*>(xs + 2 * TS * XS);       // [2][EC][MKP]
  __shared__ int bidx[TS];
  const int tid = threadIdx.x, nthr = blockDim.x;
  for (int i = tid; i < TS; i += nthr) {
    const int slot = tile * TS + i;
    bidx[i] = a.perm ? a.perm[slot] : (slot < a.B ? slot : -1);
  }
  __syncthreads();
  const int key = a.tile_vs ? a.tile_vs[tile >> a.tile_shift] : 0;
  const int vs = a.scale_in_low ? key % a.key_div : key, vm = a.scale_in_low ? key / a.key_div : key;
  const float2* PTv = a.PT + (int64_t)vs * a.EP * MKP;
  const int e_begin = split * a.esplit, e_end = min(a.E, e_begin + a.esplit);
  const int nchunks = (e_end - e_begin + EC - 1) / EC;
  const bool al16 = ((reinterpret_cast<uintptr_t>(a.x) & 15) == 0) && (a.x_bstride % 4 == 0);

  auto load_chunk = [&](int c, int st) {
    const int e0 = e_begin + c * EC;
    float* xd = xs + st * TS * XS;
    if (al16) {
      for (int idx = tid; idx < TS * (EC / 4); idx += nthr) {
        const int row = idx / (EC / 4), q = idx - row * (EC / 4);
        const int b = bidx[row], e = e0 + 4 * q;
        const int valid = b < 0 ? 0 : max(0, min(4, a.E - e)) * 4;           // bytes; the rest of the 16 is zero-filled
        cp_async16(xd + row * XS + 4 * q, a.x + (int64_t)max(b, 0) * a.x_bstride + (valid ? e : 0), valid);
      }
    } else {
      for (int idx = tid; idx < TS * EC; idx += nthr) {
        const int row = idx / EC, q = idx - row * EC;
        const int b = bidx[row], e = e0 + q;
        const int valid = (b < 0 || e >= a.E) ? 0 : 4;
        cp_async4(xd + row * XS + q, a.x + (int64_t)max(b, 0) * a.x_bstride + (valid ? e : 0), valid);
      }
    }
    const float4* src = reinterpret_cast<const float4*>(PTv + (int64_t)e0 * MKP);      // e0 + EC <= EP: the table is padded
    float4* dst = reinterpret_cast<float4*>(ps + st * EC * MKP);
    for (int idx = tid; idx < EC * MKP / 2; idx += nthr) cp_async16(dst + idx, src + idx, 16);
    cp_commit();
  };

  const int sg = tid % SGS, mg = tid / SGS, mk0 = mg * TM;
  float acc[8][TM];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < TM; ++j) acc[i][j] = 0.f;
  float off[TM];                                                   // the tile's mean offsets of the current channel for this thread's components
#pragma unroll
  for (int j = 0; j < TM; ++j) off[j] = 0.f;
  const float* mrow = OFF ? a.mtab + (int64_t)vm * a.mwidth + a.moff : nullptr;
  int reload_e = e_begin;                                          // element index at which the mean offsets change (start of slice, then every channel)

  if (nchunks > 0) load_chunk(0, 0);
  for (int c = 0; c < nchunks; ++c) {
    const int st = c & 1;
    if (c + 1 < nchunks) { load_chunk(c + 1, st ^ 1); cp_wait<1>(); } else { cp_wait<0>(); }
    __syncthreads();
    const float* xr = xs + st * TS * XS + sg * XS;
    const float2* pr = ps + st * EC * MKP + mk0;
    int el = 0;
    while (el < EC) {
      int run = EC - el;                                           // elements until the chunk ends or the channel (mean offsets) changes
      if (OFF) {
        const int e = e_begin + c * EC + el;
        if (e == reload_e) {                                       // first element of a channel (or of this slice)
          const int d = e / a.HW;
          reload_e = (d + 1) * a.HW;
          if (d < a.D) {
#pragma unroll
            for (int j = 0; j < TM; ++j) off[j] = mk0 + j < a.MK ? __ldg(mrow + (mk0 + j) * a.D + d) : 0.f;
          }
        }
        run = min(run, reload_e - e);
      }
      const int el_end = el + run;
#pragma unroll 2
      for (; el < el_end; ++el) {
        float xv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) xv[i] = xr[SGS * i * XS + el];
        float2 p[TM];
        if constexpr (TM == 4) {
          const float4 p01 = *reinterpret_cast<const float4*>(pr + el * MKP), p23 = *reinterpret_cast<const float4*>(pr + el * MKP + 2);
          p[0] = make_float2(p01.x, p01.y); p[1] = make_float2(p01.z, p01.w); p[2] = make_float2(p23.x, p23.y); p[3] = make_float2(p23.z, p23.w);
        } else if constexpr (TM == 2) {
          const float4 p01 = *reinterpret_cast<const float4*>(pr + el * MKP);
          p[0] = make_float2(p01.x, p01.y); p[1] = make_float2(p01.z, p01.w);
        } else {
          p[0] = pr[el * MKP];
        }
#pragma unroll
        for (int j = 0; j < TM; ++j) {
          const float mu = OFF ? p[j].x + off[j] : p[j].x;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float df = xv[i] - mu;
            acc[i][j] = fmaf(-p[j].y * df, df, acc[i][j]);
          }
        }
      }
    }
    __syncthreads();
  }
  // partial sums of this slice
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float* dst = a.part + ((int64_t)split * a.slots + (int64_t)tile * TS + sg + SGS * i) * MKP + mk0;
    if constexpr (TM == 4) *reinterpret_cast<float4*>(dst) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    else if constexpr (TM == 2) *reinterpret_cast<float2*>(dst) = make_float2(acc[i][0], acc[i][1]);
    else dst[0] = acc[i][0];
  }
}

// out[b, m] = logsumexp_k( sum_split part + LB ) (+ logp_scale * logp_c[b]); slices are added in index order.
__global__ void finish_kernel(const Args a) {
  const int64_t total = (int64_t)a.slots * a.M;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int slot = (int)(idx / a.M), m = (int)(idx - (int64_t)slot * a.M);
    const int ts = TS << a.tile_shift;
    if (a.n_tiles && slot >= *a.n_tiles * ts) continue;
    const int b = a.perm ? a.perm[slot] : (slot < a.B ? slot : -1);
    if (b < 0) continue;
    const int key = a.tile_vs ? a.tile_vs[slot / ts] : 0;
    const int vs = a.scale_in_low ? key % a.key_div : key;
    float c[64];
    float mx = -INFINITY;
    for (int k = 0; k < a.K; ++k) {
      float v = 0.f;
      for (int sp = 0; sp < a.nsplit; ++sp) v += a.part[((int64_t)sp * a.slots + slot) * a.MKP + m * a.K + k];
      v += a.LB[vs * a.MKP + m * a.K + k];
      c[k] = v; mx = fmaxf(mx, v);
    }
    float se = 0.f;
    for (int k = 0; k < a.K; ++k) se += expf(c[k] - mx);
    a.out[(int64_t)b * a.M + m] = mx + logf(se) + (a.logp_c ? a.logp_scale * a.logp_c[b] : 0.f);
  }
}

static inline int64_t align_up(int64_t v, int64_t al) { return (v + al - 1) / al * al; }
static inline int mkp_of(int MK) { return (MK + 3) & ~3; }
static inline int ep_of(int E) { return (E + EC - 1) / EC * EC; }
static inline int tm_of(int MKP) { return MKP >= 64 ? 4 : (MKP >= 32 ? 2 : 1); }      // threads = 8 * MKP / TM <= 256
static inline int64_t max_tiles(int B, int n_keys, int ts = TS) { return ((int64_t)B + ts - 1) / ts + (n_keys > 1 ? n_keys : 0); }
// Slices of e per tile: enough CTAs for ~4 rounds of the ~3 CTAs an SM holds (a 1.05-wave grid runs at half speed), counted on the
// expected number of non-empty tiles (buckets are padded by half a tile on average; the launch grid covers the worst case).
static inline int splits_for(int B, int n_keys, int E) {
  const int nch = (E + EC - 1) / EC;
  const int64_t est_tiles = ((int64_t)B + TS - 1) / TS + (n_keys > 1 ? n_keys / 2 : 0);
  int want = (int)((12LL * num_sms() + est_tiles - 1) / est_tiles);
  if (want < 1) want = 1;
  if (want > nch) want = nch;
  const int per = (nch + want - 1) / want;                          // chunks per slice
  return (nch + per - 1) / per;
}

}  // namespace gt
}  // namespace cfpp
using namespace cfpp;

extern "C" int64_t cfpp_gmm_tile_table_bytes(int M, int K, int D, int HW, int n_scale_ctx) {
  const int MK = M * K, MKP = gt::mkp_of(MK), EP = gt::ep_of(D * HW);
  if (MK < 1 || K > 64 || MKP > 128 || n_scale_ctx < 1 || n_scale_ctx > 4096) return -1;
  return gt::align_up((int64_t)n_scale_ctx * EP * MKP * 8, 256) + gt::align_up((int64_t)n_scale_ctx * MKP * 4, 256);
}

extern "C" int cfpp_gmm_tile_prepare(const float* mG, const float* sG, const float* wG, const float* scale_table, int scale_width,
                                     int scale_off, int n_scale_ctx, void* table, int M, int K, int D, int HW, void* stream) {
  CFPP_REQUIRE(cfpp_gmm_tile_table_bytes(M, K, D, HW, n_scale_ctx) > 0, "gmm_tile_prepare: unsupported sizes M=%d K=%d", M, K);
  CFPP_REQUIRE(table && (scale_table || n_scale_ctx == 1), "gmm_tile_prepare: null table");
  const int MK = M * K, MKP = gt::mkp_of(MK), EP = gt::ep_of(D * HW);
  float2* PT = (float2*)table;
  float* LB = (float*)((char*)table + gt::align_up((int64_t)n_scale_ctx * EP * MKP * 8, 256));
  gt::prepare_kernel<<<dim3(MKP, n_scale_ctx), 256, 0, (cudaStream_t)stream>>>(mG, sG, wG, scale_table, scale_width, scale_off, PT, LB, MK, MKP, K, D, HW, EP);
  return check_launch("gmm_tile_prepare");
}

// Workspace: partial sums, bucket permutation, tile keys, tile count and the tensor-core kernel's guard flags, sized for the larger of
// the two geometries (64-sample tiles of tile_kernel, 128-sample tiles of gmm_tc).
struct Workspace { int64_t part, perm, tile_vs, flags; };
static Workspace ws_layout(int B, int M, int K, int D, int HW, int n_keys) {
  const int MKP = gt::mkp_of(M * K), E = D * HW;
  const int64_t t64 = gt::max_tiles(B, n_keys), t128 = gt::max_tiles(B, n_keys, gtc::TS);
  const int64_t ns64 = gt::splits_for(B, n_keys, E), ns128 = gtc::splits_for(B, n_keys, E, M * K);
  Workspace w;
  w.part = gt::align_up(std::max(ns64 * t64 * gt::TS, ns128 * t128 * gtc::TS) * MKP * 4, 256);
  w.perm = gt::align_up(std::max(t64 * gt::TS, t128 * gtc::TS) * 4, 256);
  w.tile_vs = gt::align_up(std::max(t64, t128) * 4, 256);
  w.flags = gt::align_up(ns128 * t128 * 4, 256);
  return w;
}

extern "C" int64_t cfpp_gmm_tile_workspace_bytes(int B, int M, int K, int D, int HW, int n_keys) {
  if (n_keys < 1 || n_keys > 4096) return -1;
  const Workspace w = ws_layout(B, M, K, D, HW, n_keys);
  return w.part + w.perm + w.tile_vs + 256 + w.flags;
}

// Tensor-core path (gmm_tc.cu) when x rows can be read as 16-byte vectors and M*K > 48; the exact tile_kernel otherwise, and for every
// slice whose accuracy guard gmm_tc flags.  tile_kernel spends 3 M*K FP32 instructions per element of x, gmm_tc a fixed conversion of x
// into operands: on one B200 the tensor cores win at M*K = 80 (cfg2: 0.66 -> 0.42 ms per step) and lose at M*K = 8 (cfg4: 0.065 -> 0.085 ms).
extern "C" int cfpp_gmm_tile_logprob(const float* x, int64_t x_bstride, const void* table, const int64_t* ctx, int n_ctx,
                                     const int* cards, const float* mean_table, int mean_width, int mean_off,
                                     const float* logp_c, float logp_scale, float* out, void* workspace,
                                     int64_t workspace_bytes, int B, int M, int K, int D, int HW, void* stream) {
  CFPP_REQUIRE(n_ctx >= 0 && n_ctx <= 2 && (n_ctx == 0 || (ctx && cards)), "gmm_tile: n_ctx=%d (0, 1 or 2 context features)", n_ctx);
  const int n_scale_ctx = n_ctx == 0 ? 1 : cards[n_ctx - 1];
  const int64_t n_keys64 = n_ctx == 0 ? 1 : (n_ctx == 1 ? (int64_t)cards[0] : (int64_t)cards[0] * cards[1]);
  CFPP_REQUIRE(n_keys64 >= 1 && n_keys64 <= 4096, "gmm_tile: %lld context tuples (max 4096)", (long long)n_keys64);
  const int n_keys = (int)n_keys64;
  CFPP_REQUIRE(cfpp_gmm_tile_table_bytes(M, K, D, HW, n_scale_ctx) > 0, "gmm_tile: unsupported sizes M=%d K=%d", M, K);
  CFPP_REQUIRE(table && workspace && workspace_bytes >= cfpp_gmm_tile_workspace_bytes(B, M, K, D, HW, n_keys), "gmm_tile: table / workspace too small");
  CFPP_REQUIRE(!mean_table || n_ctx > 0, "gmm_tile: mean offsets need a context");
  if (B <= 0) return CFPP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int MK = M * K, MKP = gt::mkp_of(MK), E = D * HW, EP = gt::ep_of(E);
  const bool tc = MK > 48 && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && (x_bstride % 4 == 0) && (E % 4 == 0);
  const int ts = tc ? gtc::TS : gt::TS;
  const int64_t tiles = gt::max_tiles(B, n_keys, ts);
  const int nsplit = tc ? gtc::splits_for(B, n_keys, E, MK) : gt::splits_for(B, n_keys, E);
  const int nch = EP / gt::EC, per = (nch + nsplit - 1) / nsplit;
  gt::Args a{};
  a.x = x; a.x_bstride = x_bstride;
  a.PT = (const float2*)table;
  a.LB = (const float*)((const char*)table + gt::align_up((int64_t)n_scale_ctx * EP * MKP * 8, 256));
  const Workspace w = ws_layout(B, M, K, D, HW, n_keys);
  char* p = (char*)workspace;
  a.part = (float*)p; p += w.part;
  int* perm = (int*)p; p += w.perm;
  int* tile_vs = (int*)p; p += w.tile_vs;
  int* n_tiles = (int*)p; p += 256;
  int* flags = (int*)p;
  a.key_div = n_ctx == 2 ? cards[1] : 1; a.scale_in_low = n_ctx == 2 ? 1 : 0;
  a.mtab = mean_table; a.mwidth = mean_width; a.moff = mean_off;
  a.logp_c = logp_c; a.logp_scale = logp_scale; a.out = out;
  a.B = B; a.M = M; a.K = K; a.MK = MK; a.MKP = MKP; a.D = D; a.HW = HW; a.E = E; a.EP = EP;
  a.esplit = per * gt::EC; a.nsplit = nsplit; a.slots = (int)(tiles * ts);
  a.tile_shift = tc ? 1 : 0;
  if (n_ctx > 0) {
    gt::bucket_kernel<<<1, 1024, 3 * n_keys * sizeof(int), st>>>(ctx, n_ctx, n_ctx == 2 ? cards[1] : 1, B, n_keys, ts, perm, tile_vs, n_tiles);
    int rc = check_launch("gmm_tile_bucket");
    if (rc) return rc;
    a.perm = perm; a.tile_vs = tile_vs; a.n_tiles = n_tiles;
  }
  if (tc) {
    gtc::Args g{};
    g.x = x; g.x_bstride = x_bstride; g.PT = a.PT; g.LB = a.LB;
    g.perm = a.perm; g.tile_vs = a.tile_vs; g.n_tiles = a.n_tiles;
    g.key_div = a.key_div; g.scale_in_low = a.scale_in_low;
    g.mtab = mean_table; g.mwidth = mean_width; g.moff = mean_off;
    g.part = a.part; g.flags = flags; g.has_logp = logp_c != nullptr;
    g.B = B; g.K = K; g.MK = MK; g.MKP = MKP; g.N = gtc::n_of(MK); g.D = D; g.HW = HW; g.E = E; g.EP = EP;
    g.esplit = a.esplit; g.nsplit = nsplit; g.slots = a.slots; g.tiles = (int)tiles;
    int rc = gtc::launch(g, st);
    if (rc) return rc;
    a.flags = flags; a.ftiles = (int)tiles;
  }
  const int TM = gt::tm_of(MKP);
  const int threads = gt::SGS * (MKP / TM);
  const size_t smem = (size_t)2 * gt::TS * gt::XS * 4 + (size_t)2 * gt::EC * MKP * 8;
  dim3 grid((unsigned)(tiles << a.tile_shift), nsplit);
  const bool offs = mean_table != nullptr;
#define CFPP_GT_LAUNCH(TMV, OFFV)                                                                                          \
  do {                                                                                                                     \
    static DeviceOnce attr;                                                                                              \
    if (attr.first()) {                                                                                                           \
      cudaFuncSetAttribute(gt::tile_kernel<TMV, OFFV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);           \
      cudaFuncSetAttribute(gt::tile_kernel<TMV, OFFV>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); \
    }                                                                                                                      \
    gt::tile_kernel<TMV, OFFV><<<grid, threads, smem, st>>>(a);                                                            \
  } while (0)
  if (TM == 4) { if (offs) CFPP_GT_LAUNCH(4, true); else CFPP_GT_LAUNCH(4, false); }
  else if (TM == 2) { if (offs) CFPP_GT_LAUNCH(2, true); else CFPP_GT_LAUNCH(2, false); }
  else { if (offs) CFPP_GT_LAUNCH(1, true); else CFPP_GT_LAUNCH(1, false); }
#undef CFPP_GT_LAUNCH
  int rc = check_launch("gmm_tile");
  if (rc) return rc;
  const int64_t total = (int64_t)a.slots * M;
  int64_t blocks = (total + 255) / 256; if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  gt::finish_kernel<<<(int)blocks, 256, 0, st>>>(a);
  return check_launch("gmm_tile_finish");
}
