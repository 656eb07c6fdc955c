// Invertible 1x1 convolution (shared or per-sample weights), ActNorm, their fusion, slogdet and the ActNorm
// data-dependent initialisation statistics.   Reference: layers/conv1x1.py:28-57, layers/actnorm.py:28-60.
#include <stdlib.h>
#include "common.cuh"

namespace cfpp {

// ---------------------------------------------------------------------------------------------------------------
// slogdet: LU with partial pivoting in fp64, one CTA.  A is DxD fp32 row-major.
// ---------------------------------------------------------------------------------------------------------------
__global__ void slogdet_kernel(const float* __restrict__ A, int D, float* __restrict__ out) {
  extern __shared__ double lu[];            // D*D
  __shared__ int piv_row;
  __shared__ double piv_val;
  for (int i = threadIdx.x; i < D * D; i += blockDim.x) lu[i] = (double)A[i];
  __syncthreads();
  double logabs = 0.0;                      // only thread 0's copy is used
  for (int k = 0; k < D; ++k) {
    if (threadIdx.x < 32) {                 // warp 0: arg-max |lu[i][k]| over i >= k
      double best = -1.0; int bi = k;
      for (int i = k + threadIdx.x; i < D; i += 32) { double v = fabs(lu[i * D + k]); if (v > best) { best = v; bi = i; } }
      for (int o = 16; o > 0; o >>= 1) {
        double ob = __shfl_xor_sync(0xffffffffu, best, o); int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
      }
      if (threadIdx.x == 0) { piv_row = bi; piv_val = lu[bi * D + k]; }
    }
    __syncthreads();
    const int pr = piv_row; const double pv = piv_val;
    if (pr != k) for (int j = threadIdx.x; j < D; j += blockDim.x) { double t = lu[k * D + j]; lu[k * D + j] = lu[pr * D + j]; lu[pr * D + j] = t; }
    if (threadIdx.x == 0) logabs += log(fabs(pv));
    __syncthreads();
    if (pv != 0.0) {
      for (int i = k + 1 + threadIdx.x; i < D; i += blockDim.x) {
        const double f = lu[i * D + k] / pv;
        for (int j = k + 1; j < D; ++j) lu[i * D + j] -= f * lu[k * D + j];
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (float)logabs;
}

// ---------------------------------------------------------------------------------------------------------------
// Conv1x1 (+ optional ActNorm epilogue): per sample a (D x D) by (D x HW) product, z[i][p] = sum_j W[i][j] x[j][p].
// The matrix is per sample in specialist mode (assembled from the raw context matrix c) and used for only HW pixels, so
// the kernel is organised around NOT moving it twice: a CTA takes NS samples, assembles their matrices row-major into
// shared memory with coalesced reads of c (the only pass over c), and every thread owns ONE pixel column: its D inputs are
// loaded from HBM straight into registers (coalesced along pixels, never staged), the matrix rows arrive as warp-broadcast
// 128-bit shared loads (4 FMA per load), and outputs are stored coalesced along pixels.  When a sample has few pixels
// (HW = 16) the output rows are split over G thread groups so a CTA still has 256 threads of work per 4 matrices.
// ---------------------------------------------------------------------------------------------------------------
struct Conv1x1Args {
  const float* x; float* z; float* ldj; const float* NN; const float* logabsdet;
  const float* c; const float* logp_c; int contextflow;
  const float* an_t; const float* an_logs; int an_per_sample; const float* an_logp_c; float an_logp_scale;
  int B, D, HW, NS, PT, CPS, NCOLP, G, IR, DR, tiles_per_sample, an_stride;   // CPS = thread columns per sample tile (PT / PX), DR = D rounded up to 4
};

template <int PX> struct PixVec;
template <> struct PixVec<1> { using T = float; };
template <> struct PixVec<2> { using T = float2; };
template <> struct PixVec<4> { using T = float4; };
__device__ __forceinline__ void pv_load(float (&d)[1], const float* p) { d[0] = __ldg(p); }
__device__ __forceinline__ void pv_load(float (&d)[2], const float* p) { const float2 v = __ldg(reinterpret_cast<const float2*>(p)); d[0] = v.x; d[1] = v.y; }
__device__ __forceinline__ void pv_load(float (&d)[4], const float* p) { const float4 v = ldg_stream(reinterpret_cast<const float4*>(p)); d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w; }
__device__ __forceinline__ void pv_store(float* p, const float (&d)[1]) { *p = d[0]; }
__device__ __forceinline__ void pv_store(float* p, const float (&d)[2]) { *reinterpret_cast<float2*>(p) = make_float2(d[0], d[1]); }
__device__ __forceinline__ void pv_store(float* p, const float (&d)[4]) { stg_stream(reinterpret_cast<float4*>(p), make_float4(d[0], d[1], d[2], d[3])); }

// DT = padded matrix width (>= D, multiple of 16), PX = consecutive pixels per thread (register tile along pixels: every matrix
// value fetched from shared memory feeds PX FMAs and the loads / stores of x and z are PX-wide).
template <int DT, int PX>
__global__ void __launch_bounds__(256) conv1x1_kernel(const Conv1x1Args a) {
  extern __shared__ float4 smem4[];
  const int D = a.D, HW = a.HW, DR = a.DR;
  const int nmat = a.c ? a.NS : 1;
  float* Ws = reinterpret_cast<float*>(smem4);                 // [nmat][DR][DT] row-major; rows >= D and columns >= D are zero
  float* sh = Ws + (size_t)nmat * DR * DT;                     // [NS][DR] ActNorm shift
  float* sc = sh + (size_t)a.NS * DR;                          // [NS][DR] ActNorm exp(-logs)
  const int64_t grp = blockIdx.x;                              // group of NS samples x one pixel tile
  const int64_t sg = grp / a.tiles_per_sample;
  const int ptile = (int)(grp - sg * a.tiles_per_sample);
  const int64_t b0 = sg * a.NS;
  const int nS = (int)min((int64_t)a.NS, (int64_t)a.B - b0);
  const int tid = threadIdx.x, nthr = blockDim.x;

  // ---- this thread's PX pixel columns: their D inputs go straight from HBM to registers, issued first so the latency overlaps
  //      the matrix assembly below ----
  const int g = tid / a.NCOLP, col = tid - g * a.NCOLP;
  const int m = col / a.CPS, pl = (col - m * a.CPS) * PX;
  const int p = ptile * a.PT + pl;
  const bool live = col < a.NS * a.CPS && m < nS && p < HW;    // HW % PX == 0 (host): a live thread owns PX real pixels
  const int64_t b = b0 + (live ? m : 0);
  float xc[DT][PX];
  {
    const float* xg = a.x + (b * D) * (int64_t)HW + (live ? p : 0);
#pragma unroll
    for (int j = 0; j < DT; ++j) {
      if (live && j < D) pv_load(xc[j], xg + (int64_t)j * HW);
      else {
#pragma unroll
        for (int q = 0; q < PX; ++q) xc[j][q] = 0.f;
      }
    }
  }

  // ---- matrices: W = NN (shared) or tril(c,-1) + diag(exp(diag c)) [- I + NN]   (conv1x1.py:36-49), row-major in shared memory.
  //      c is streamed exactly once: the NS matrices of this CTA are one contiguous run of floats, read as 128-bit loads with four
  //      loads in flight per thread before any of them is consumed ----
  if (D != DT) {                                                 // padding rows / columns must read as zero
    for (int idx = tid; idx < nmat * DR * DT; idx += nthr) Ws[idx] = 0.f;
    __syncthreads();
  }
  if (!a.c) {
    for (int idx = tid; idx < D * D; idx += nthr) { const int i = idx / D, j = idx - i * D; Ws[i * DT + j] = a.NN[idx]; }
  } else if ((D & 3) == 0) {
    const int D4 = D >> 2, units = nS * D * D4;
    const float4* c4 = reinterpret_cast<const float4*>(a.c + b0 * (int64_t)D * D);
    const float4* n4 = reinterpret_cast<const float4*>(a.NN);
    for (int u0 = tid; u0 < units; u0 += 4 * nthr) {
      float4 cv[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {                // entries strictly above the diagonal are never used (and never produced by cfpp_cn_batch)
        const int u = u0 + k * nthr;
        if (u < units) {
          int row, j0, i;
          if (D == DT) { row = u / (DT / 4); j0 = (u % (DT / 4)) << 2; i = row % DT; }
          else { row = u / D4; j0 = (u - row * D4) << 2; i = row - (row / D) * D; }
          cv[k] = (j0 > i) ? make_float4(0.f, 0.f, 0.f, 0.f) : ldg_stream(c4 + u);
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int u = u0 + k * nthr;
        if (u < units) {
          int row, j0, mm, i;
          if (D == DT) { row = u / (DT / 4); j0 = (u % (DT / 4)) << 2; mm = row / DT; i = row % DT; }     // compile-time divisors
          else { row = u / D4; j0 = (u - row * D4) << 2; mm = row / D; i = row - mm * D; }
          float v[4] = {cv[k].x, cv[k].y, cv[k].z, cv[k].w};
          if (j0 + 3 < i) {}                                               // strictly below the diagonal: W = c
          else if (j0 > i) { v[0] = v[1] = v[2] = v[3] = 0.f; }            // strictly above: 0
          else {
#pragma unroll
            for (int q = 0; q < 4; ++q) { const int j = j0 + q; v[q] = (j < i) ? v[q] : (j == i ? expf(v[q]) : 0.f); }
          }
          if (a.contextflow) {
            const float4 nn = __ldg(n4 + (i * D4 + (j0 >> 2)));
            v[0] += nn.x; v[1] += nn.y; v[2] += nn.z; v[3] += nn.w;
            if (j0 <= i && i <= j0 + 3) v[i - j0] -= 1.f;
          }
          *reinterpret_cast<float4*>(Ws + ((size_t)mm * DR + i) * DT + j0) = make_float4(v[0], v[1], v[2], v[3]);
        }
      }
    }
  } else {
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthr >> 5;
    for (int row = warp; row < nS * D; row += nwarps) {
      const int mm = row / D, i = row - mm * D;
      float* wrow = Ws + ((size_t)mm * DR + i) * DT;
      const float* nrow = a.NN + (size_t)i * D;
      const float* crow = a.c + ((b0 + mm) * D + i) * (int64_t)D;
      for (int j = lane; j < D; j += 32) {
        const float cij = j <= i ? crow[j] : 0.f;
        float v = (j < i) ? cij : (j == i ? expf(cij) : 0.f);
        if (a.contextflow) v = (v - (i == j ? 1.f : 0.f)) + nrow[j];
        wrow[j] = v;
      }
    }
  }
  if (a.an_logs) {
    for (int idx = tid; idx < a.NS * D; idx += nthr) {
      const int mm = idx / D, i = idx - mm * D;
      const int64_t bb = min(b0 + mm, (int64_t)a.B - 1);
      sh[mm * DR + i] = a.an_t[bb * a.an_stride + i];
      sc[mm * DR + i] = expf(-a.an_logs[bb * a.an_stride + i]);
    }
  }
  // ---- per-sample ldj: one warp per sample (only the CTA of the sample's first pixel tile writes it) ----
  if (ptile == 0) {
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthr >> 5;
    for (int ms = warp; ms < nS; ms += nwarps) {
      const int64_t bb = b0 + ms;
      float part = 0.f, part_an = 0.f;
      if (a.c) for (int i = lane; i < D; i += 32) part += a.c[(bb * D + i) * (int64_t)D + i];
      if (a.an_logs) for (int i = lane; i < D; i += 32) part_an += a.an_logs[bb * a.an_stride + i];
      part = warp_sum(part); part_an = warp_sum(part_an);
      if (lane == 0) {
        float l;
        if (a.c) { l = (float)HW * ((a.contextflow ? a.logabsdet[0] : 0.f) + part); if (a.logp_c) l += a.logp_c[bb] * (float)HW; }
        else l = a.logabsdet[0] * (float)HW;
        if (a.an_logs) { l += part_an; if (a.an_logp_c) l += a.an_logp_scale * a.an_logp_c[bb]; }
        a.ldj[bb] = l;
      }
    }
  }
  __syncthreads();
  if (!live) return;

  // ---- 4 output rows x PX pixels per pass; matrix rows arrive as warp-broadcast 128-bit shared loads ----
  const float* Wm = Ws + (a.c ? (size_t)m * DR * DT : 0);
  const float* shm = sh + (size_t)m * DR; const float* scm = sc + (size_t)m * DR;
  float* zg = a.z + (b * D) * (int64_t)HW + p;
  const int i_beg = g * a.IR, i_end = min(DR, i_beg + a.IR);
  const bool an = a.an_logs != nullptr;
  for (int i0 = i_beg; i0 < i_end; i0 += 4) {
    float acc[4][PX];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int q = 0; q < PX; ++q) acc[r][q] = 0.f;
    const float* w0 = Wm + (size_t)i0 * DT;
#pragma unroll
    for (int j = 0; j < DT; j += 4) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float4 w = *reinterpret_cast<const float4*>(w0 + r * DT + j);
#pragma unroll
        for (int q = 0; q < PX; ++q) {
          acc[r][q] = fmaf(w.x, xc[j][q], acc[r][q]); acc[r][q] = fmaf(w.y, xc[j + 1][q], acc[r][q]);
          acc[r][q] = fmaf(w.z, xc[j + 2][q], acc[r][q]); acc[r][q] = fmaf(w.w, xc[j + 3][q], acc[r][q]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = i0 + r;
      if (i < D) {
        if (an) {
          const float t = shm[i], e = scm[i];
#pragma unroll
          for (int q = 0; q < PX; ++q) acc[r][q] = (acc[r][q] - t) * e;
        }
        pv_store(zg + (int64_t)i * HW, acc[r]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// ActNorm alone: elementwise with per-(sample, channel) shift / log-scale.
// ---------------------------------------------------------------------------------------------------------------
__global__ void actnorm_kernel(const float* __restrict__ x, float* __restrict__ z, float* __restrict__ ldj,
                               const float* __restrict__ bt, const float* __restrict__ bl, const float* __restrict__ c,
                               const float* __restrict__ logp_c, float logp_scale, int mode, int B, int D, int HW, bool vec4) {
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (tid < B) {                                                    // ldj[b] = sum_d logs (actnorm.py:58)
    float s = 0.f;
    for (int d = 0; d < D; ++d) {
      float l = (mode != 2) ? bl[d] : 0.f;
      if (mode != 0) l = c[tid * 2 * D + D + d] + l;
      s += l;
    }
    ldj[tid] = s + (logp_c ? logp_scale * logp_c[tid] : 0.f);
  }
  auto coef = [&](int64_t bd, float& t, float& e) {
    const int d = bd % D; const int64_t b = bd / D;
    float tt = (mode != 2) ? bt[d] : 0.f, ll = (mode != 2) ? bl[d] : 0.f;
    if (mode != 0) { tt = c[b * 2 * D + d] + tt; ll = c[b * 2 * D + D + d] + ll; }
    t = tt; e = expf(-ll);
  };
  if (vec4) {
    const int64_t n4 = (int64_t)B * D * HW / 4;
    const int hw4 = HW / 4;
    for (int64_t i = tid; i < n4; i += stride) {
      float t, e; coef(i / hw4, t, e);
      float4 v = ldg_stream(reinterpret_cast<const float4*>(x) + i);
      v.x = (v.x - t) * e; v.y = (v.y - t) * e; v.z = (v.z - t) * e; v.w = (v.w - t) * e;
      stg_stream(reinterpret_cast<float4*>(z) + i, v);
    }
  } else {
    const int64_t n = (int64_t)B * D * HW;
    for (int64_t i = tid; i < n; i += stride) {
      float t, e; coef(i / HW, t, e);
      z[i] = (x[i] - t) * e;
    }
  }
}

// ActNorm.initialize statistics: one CTA per channel, fp64 two-pass (mean, then unbiased variance).
__global__ void actnorm_stats_kernel(const float* __restrict__ x, float* __restrict__ mean, float* __restrict__ logstd,
                                     int B, int D, int HW) {
  __shared__ double red[32];
  __shared__ double mu_s;
  const int d = blockIdx.x;
  const int64_t n = (int64_t)B * HW;
  auto block_sum = [&](double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
    __syncthreads();
    return s;
  };
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += (double)x[((i / HW) * D + d) * (int64_t)HW + (i % HW)];
  const double tot = block_sum(acc);
  if (threadIdx.x == 0) mu_s = tot / (double)n;
  __syncthreads();
  const double mu = mu_s;
  acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = (double)x[((i / HW) * D + d) * (int64_t)HW + (i % HW)] - mu;
    acc += v * v;
  }
  const double ss = block_sum(acc);
  if (threadIdx.x == 0) {
    mean[d] = (float)mu;
    const float sd = (float)sqrt(ss / (double)(n - 1));           // torch.std: unbiased
    logstd[d] = logf(sd + 1e-8f);                                 // actnorm.py:32
  }
}

}  // namespace cfpp
using namespace cfpp;

int cfpp_conv1x1_rt_launch(const float* x, float* z, float* ldj, const float* NN, const float* logabsdet, const float* c, const float* logp_c,
                           int contextflow, const float* an_t, const float* an_logs, int an_stride, const float* an_logp_c, float an_logp_scale,
                           int B, int D, int HW, cudaStream_t st);

extern "C" int cfpp_slogdet(const float* A, int D, float* logabsdet, void* stream) {
  CFPP_REQUIRE(D >= 1 && D <= 128, "slogdet: D=%d outside [1,128]", D);
  static DeviceOnce attr_set;
  if (attr_set.first()) { cudaFuncSetAttribute(slogdet_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 128 * 8); }
  slogdet_kernel<<<1, 128, (size_t)D * D * sizeof(double), (cudaStream_t)stream>>>(A, D, logabsdet);
  return check_launch("slogdet");
}

extern "C" int cfpp_conv1x1_fwd(const float* x, float* z, float* ldj, const float* NN, const float* logabsdet,
                                const float* c, const float* logp_c, int contextflow,
                                const float* an_t, const float* an_logs, int an_per_sample, const float* an_logp_c, float an_logp_scale,
                                int B, int D, int HW, void* stream) {
  CFPP_REQUIRE(D >= 1 && D <= 128 && HW >= 1, "conv1x1: D=%d HW=%d unsupported (D<=128)", D, HW);
  CFPP_REQUIRE((an_t == nullptr) == (an_logs == nullptr), "conv1x1: an_t and an_logs must be given together");
  CFPP_REQUIRE(an_per_sample >= 0 && an_per_sample <= 2, "conv1x1: an_per_sample must be 0, 1 or 2");
  if (B <= 0) return CFPP_OK;
  Conv1x1Args a{x, z, ldj, NN, logabsdet, c, logp_c, contextflow, an_t, an_logs, an_per_sample, an_logp_c, an_logp_scale, B, D, HW};
  a.an_stride = an_per_sample == 0 ? 0 : (an_per_sample == 1 ? D : 2 * D);
  {   // register-tiled kernel (conv1x1_rt.cu) where it measured faster and its tile fits; the column-per-thread kernel below otherwise
    // measured on B200 (B = 8192): shared matrix D=16/32/64 rt 80/57/47 us vs column kernel 61/55/59 us; per-sample matrices
    // rt 100/80/161 us vs 72/86/148 us -- the per-sample assembly of W from c dominates both; rt is used where it wins
    const bool use_rt = c ? (D > 16 && D <= 32) : (D > 32);
    if (use_rt) {
      const int rc = cfpp_conv1x1_rt_launch(x, z, ldj, NN, logabsdet, c, logp_c, contextflow, an_t, an_logs, a.an_stride, an_logp_c, an_logp_scale,
                                            B, D, HW, (cudaStream_t)stream);
      if (rc != CFPP_ERR_UNSUPPORTED) return rc;
    }
  }
  const int DT = D <= 16 ? 16 : D <= 32 ? 32 : D <= 64 ? 64 : D <= 96 ? 96 : 128;
  const bool al16 = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(z)) & 15) == 0;
  int PX = DT == 16 ? 4 : DT == 32 ? 2 : 1;                 // DT * PX = 64 input registers per thread
  while (PX > 1 && (HW % PX != 0 || !al16)) PX >>= 1;
  a.DR = (D + 3) / 4 * 4;
  a.PT = HW < 256 * PX ? HW : 256 * PX;
  a.CPS = (a.PT + PX - 1) / PX;
  a.tiles_per_sample = (HW + a.PT - 1) / a.PT;
  int ns = 256 / a.CPS; if (ns < 1) ns = 1;
  const size_t mat_bytes = (size_t)a.DR * DT * sizeof(float);
  if (c) { const int by_smem = (int)((72 * 1024) / mat_bytes); if (ns > by_smem) ns = by_smem < 1 ? 1 : by_smem; }
  if (ns > B) ns = B;
  a.NS = ns;
  a.NCOLP = (ns * a.CPS + 31) / 32 * 32;
  int G = 256 / a.NCOLP; if (G < 1) G = 1;
  int IR = ((a.DR + G - 1) / G + 3) / 4 * 4;
  G = (a.DR + IR - 1) / IR;
  a.G = G; a.IR = IR;
  const int threads = G * a.NCOLP;
  const size_t smem = (size_t)(c ? ns : 1) * mat_bytes + (size_t)2 * ns * a.DR * sizeof(float);
  CFPP_REQUIRE(threads <= 256 && smem <= 200 * 1024, "conv1x1: tile does not fit (D=%d)", D);
  const int64_t blocks = (int64_t)((B + ns - 1) / ns) * a.tiles_per_sample;
  cudaStream_t st = (cudaStream_t)stream;
#define CFPP_C1(DT_, PX_) do { static DeviceOnce set_; if (set_.first()) { cudaFuncSetAttribute(conv1x1_kernel<DT_, PX_>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); } \
    conv1x1_kernel<DT_, PX_><<<(unsigned)blocks, threads, smem, st>>>(a); } while (0)
  if (DT == 16) { if (PX == 4) CFPP_C1(16, 4); else if (PX == 2) CFPP_C1(16, 2); else CFPP_C1(16, 1); }
  else if (DT == 32) { if (PX == 2) CFPP_C1(32, 2); else CFPP_C1(32, 1); }
  else if (DT == 64) CFPP_C1(64, 1);
  else if (DT == 96) CFPP_C1(96, 1);
  else CFPP_C1(128, 1);
#undef CFPP_C1
  return check_launch("conv1x1_fwd");
}

extern "C" int cfpp_actnorm_fwd(const float* x, float* z, float* ldj, const float* base_t, const float* base_logs, const float* c,
                                const float* logp_c, float logp_scale, int mode, int B, int D, int HW, void* stream) {
  CFPP_REQUIRE(mode >= 0 && mode <= 2, "actnorm: mode %d", mode);
  CFPP_REQUIRE(mode == 0 || c != nullptr, "actnorm: context matrix required for mode %d", mode);
  CFPP_REQUIRE(mode == 2 || (base_t && base_logs), "actnorm: base parameters required");
  if (B <= 0) return CFPP_OK;
  const bool vec4 = (HW % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(z)) % 16 == 0);
  const int64_t n = (int64_t)B * D * HW / (vec4 ? 4 : 1);
  int64_t blocks = (n + 255) / 256;
  const int64_t minb = (B + 255) / 256, cap = (int64_t)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < minb) blocks = minb;
  actnorm_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(x, z, ldj, base_t, base_logs, c, logp_c, logp_scale, mode, B, D, HW, vec4);
  return check_launch("actnorm_fwd");
}

extern "C" int cfpp_actnorm_stats(const float* x, float* mean, float* logstd, int B, int D, int HW, void* stream) {
  CFPP_REQUIRE(B >= 1 && D >= 1 && HW >= 1, "actnorm_stats: bad dims");
  actnorm_stats_kernel<<<D, 256, 0, (cudaStream_t)stream>>>(x, mean, logstd, B, D, HW);
  return check_launch("actnorm_stats");
}
