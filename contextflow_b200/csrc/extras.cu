// Kernels of the rows SURVEY §8(f) lists beside the headline path:
//   * standalone Sigmoid / Softplus flow layers (reference layers/activations.py:228-264): forward, reverse, backward;
//   * StudentMixtureDistribution.log_prob (layers/distributions/student.py:44-111): scoring, and training with every parameter but the
//     frozen degrees of freedom vS;
//   * training pieces of the conventional (concatenated-context) specialists: the per-sample bias + ReLU of the first conditioner
//     convolution (coupling.py:47) and the mixture's own parameter gradients when mG / sG / wG train beside the context offsets
//     (distributions/gaussian.py:146-155 with contextflow = False).
#include <math.h>
#include "common.cuh"

namespace cfpp {
namespace ex {

// ---------------------------------------------------------------------------------------------------------------- activations
// kind 0 = Sigmoid(temperature): z = sigmoid(T x), ldj_i = log T - softplus(-T x) - softplus(T x)          (activations.py:234-238)
// kind 1 = Softplus:             z = softplus(x),  ldj_i = logsigmoid(x) = -softplus(-x)                    (activations.py:252-259)
// rows of D values; one warp per row; ldj[row] = sum over the row in a fixed order (lane-strided partials, shuffle tree).
__global__ void __launch_bounds__(256) act_fwd_kernel(const float* __restrict__ x, float* __restrict__ z, float* __restrict__ ldj,
                                                      const float* __restrict__ temperature, int64_t rows, int D, int kind) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int l = threadIdx.x & 31;
  const float T = kind == 0 ? temperature[0] : 1.f;
  const float logT = kind == 0 ? logf(T) : 0.f;
  float acc = 0.f;
  for (int i = l; i < D; i += 32) {
    const float v = x[row * D + i];
    if (kind == 0) {
      const float t = T * v;
      z[row * D + i] = 1.f / (1.f + expf(-t));
      acc += logT - softplus_f(-t) - softplus_f(t);
    } else {
      z[row * D + i] = softplus_f(v);
      acc += fminf(v, 0.f) - log1pf(expf(-fabsf(v)));            // F.logsigmoid
    }
  }
  acc = warp_sum(acc);
  if (l == 0) ldj[row] = acc;
}

// reverse: Sigmoid: z clamped to [eps, 1 - eps], x = (log z - log1p(-z)) / T (activations.py:240-244; the [0,1] assertion is the
// caller's); Softplus: x = z + log1p(-exp(-max(z, eps))) (activations.py:261-264)
__global__ void __launch_bounds__(256) act_inv_kernel(const float* __restrict__ z, float* __restrict__ x, const float* __restrict__ temperature,
                                                      int64_t n, float eps, int kind) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = z[i];
  if (kind == 0) {
    const float c = fminf(fmaxf(v, eps), 1.f - eps);
    x[i] = (1.f / temperature[0]) * (logf(c) - log1pf(-c));
  } else {
    x[i] = v + log1pf(-expf(-fmaxf(v, eps)));
  }
}

// backward: dx = dz * dz/dx + dldj[row] * d ldj_i / dx
//   Sigmoid:  dz/dx = T z (1 - z),  d ldj_i/dx = T (1 - 2 z)        Softplus: dz/dx = sigmoid(x),  d ldj_i/dx = sigmoid(-x)
__global__ void __launch_bounds__(256) act_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dz, const float* __restrict__ dldj,
                                                      float* __restrict__ dx, const float* __restrict__ temperature, int64_t n, int D, int kind) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = x[i], gz = dz ? dz[i] : 0.f, gl = dldj ? dldj[i / D] : 0.f;
  if (kind == 0) {
    const float T = temperature[0];
    const float s = 1.f / (1.f + expf(-T * v));
    dx[i] = gz * T * s * (1.f - s) + gl * T * (1.f - 2.f * s);
  } else {
    const float s = 1.f / (1.f + expf(-v));
    dx[i] = gz * s + gl * (1.f - s);
  }
}

// ---------------------------------------------------------------------------------------------------- Student-t mixture
// tables per (m, k, e): Gaussian {mu, 1/sigma, -log sigma - log sqrt(2 pi)}, Student {mu, 1/(sigma sqrt(df)), -(df + 1)/2, -Z},
//   Z = log sigma + 0.5 log df + 0.5 log pi + lgamma(df / 2) - lgamma((df + 1) / 2)            (torch.distributions.StudentT.log_prob)
// mixture weights: softmax over dim 0 of w (M, K) (student.py:78-79), renormalised along K by Categorical(probs=...)
__global__ void __launch_bounds__(256) student_prep_kernel(const float* __restrict__ mG, const float* __restrict__ sG, const float* __restrict__ mS,
                                                           const float* __restrict__ sS, const float* __restrict__ vS, float* __restrict__ tab, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float sg = softplus_f(sG[i]), ss = softplus_f(sS[i]), df = softplus_f(vS[i]);
  float* t = tab + i * 8;
  t[0] = mG[i]; t[1] = 1.f / sg; t[2] = -logf(sg) - kHalfLog2Pi;
  t[3] = mS[i]; t[4] = 1.f / (ss * sqrtf(df)); t[5] = -0.5f * (df + 1.f);
  t[6] = -(logf(ss) + 0.5f * logf(df) + 0.57236494292470008707f + lgammaf(0.5f * df) - lgammaf(0.5f * (df + 1.f)));
  t[7] = 0.f;
}

// log mixture weights (M, K) for both families: lw[f][m][k] = log( softmax_0(w)[m,k] / sum_k softmax_0(w)[m,k] )
__global__ void student_weights_kernel(const float* __restrict__ wG, const float* __restrict__ wS, float* __restrict__ lw, int M, int K) {
  const int f = blockIdx.x;
  const float* w = f == 0 ? wG : wS;
  for (int m = threadIdx.x; m < M; m += blockDim.x) {
    float tot = 0.f;
    for (int k = 0; k < K; ++k) {
      float mx = -INFINITY;
      for (int j = 0; j < M; ++j) mx = fmaxf(mx, w[j * K + k]);
      float se = 0.f;
      for (int j = 0; j < M; ++j) se += expf(w[j * K + k] - mx);
      const float p = expf(w[m * K + k] - mx) / se;
      lw[(f * M + m) * K + k] = p;
      tot += p;
    }
    for (int k = 0; k < K; ++k) lw[(f * M + m) * K + k] = logf(lw[(f * M + m) * K + k] / tot);
  }
}

// one CTA per (sample, mixture): component sums over the D*H*W elements in a fixed order, then the two log-sum-exps.  resp (training):
// the responsibilities softmax_k of both families, resp[b, m, f, k] (f = 0 Gaussian, 1 Student-t); NULL for scoring.
constexpr int kStuMaxK = 32;
__global__ void __launch_bounds__(256) student_logprob_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ tab,
                                                              const float* __restrict__ lw, float* __restrict__ logp, float* __restrict__ resp,
                                                              int M, int K, int n) {
  __shared__ float red[2][kStuMaxK][8];
  const int64_t b = blockIdx.x;
  const int m = blockIdx.y, w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const float* xb = x + b * x_bstride;
  for (int k = 0; k < K; ++k) {
    const float* t = tab + ((int64_t)(m * K + k) * n) * 8;
    float ag = 0.f, as = 0.f;
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const float4 p0 = *reinterpret_cast<const float4*>(t + (int64_t)e * 8), p1 = *reinterpret_cast<const float4*>(t + (int64_t)e * 8 + 4);
      const float v = xb[e];
      const float yg = (v - p0.x) * p0.y;
      ag += fmaf(-0.5f * yg, yg, p0.z);
      const float ys = (v - p0.w) * p1.x;
      as += fmaf(p1.y, log1pf(ys * ys), p1.z);
    }
    ag = warp_sum(ag); as = warp_sum(as);
    if (l == 0) { red[0][k][w] = ag; red[1][k][w] = as; }
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    const int f = threadIdx.x;
    float comp[kStuMaxK];
    float mx = -INFINITY;
    for (int k = 0; k < K; ++k) {
      float s = 0.f;
      for (int i = 0; i < 8; ++i) s += red[f][k][i];
      comp[k] = s + lw[(f * M + m) * K + k];
      mx = fmaxf(mx, comp[k]);
    }
    float se = 0.f;
    for (int k = 0; k < K; ++k) se += expf(comp[k] - mx);
    const float lse = mx + logf(se);
    red[f][0][0] = lse;
    if (resp)
      for (int k = 0; k < K; ++k) resp[((b * M + m) * 2 + f) * K + k] = expf(comp[k] - lse);
  }
  __syncthreads();
  if (threadIdx.x == 0) logp[b * M + m] = red[0][0][0] + red[1][0][0];
}

// ---------------------------------------------------------------------------------------------- Student-t mixture, training
// With w[b, f, mk] = g[b, m] resp[b, m, f, k] and the table's yg = (x - mG) / sg, t = (x - mS) / (ss sqrt(df)) = y / sqrt(df),
// u = t / (1 + t^2):
//   dx[b, e] = sum_mk  -wG yg / sg  +  wS (2 t5 t4) u                 (t4 = 1 / (ss sqrt(df)), t5 = -(df + 1) / 2)
//            = sum_mk  -wG (x - mG) / sg^2  -  wS (df + 1) y / (ss (df + y^2))
//   dmG = sum_b wG yg / sg,         dsG = sum_b wG (yg^2 - 1) / sg * sigmoid(sG)
//   dmS = -2 t5 t4 sum_b wS u,      dsS = sum_b wS ((df + 1) t u - 1) / ss * sigmoid(sS)
// dx: a CTA holds kStuDxS samples and one slice of elements, so every table entry read from L2 serves kStuDxS samples; the block of
// samples of blockIdx.y == 0 also writes w to wbuf for the parameter sums.
constexpr int kStuDxS = 8, kStuDxThreads = 128, kStuMaxMK = 768;
__global__ void __launch_bounds__(kStuDxThreads) student_dx_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ tab,
                                                                   const float* __restrict__ resp, const float* __restrict__ g,
                                                                   float* __restrict__ wbuf, float* __restrict__ dx, int64_t dx_bstride,
                                                                   int B, int M, int K, int n) {
  extern __shared__ float sw[];                        // [kStuDxS][2][MK]
  const int MK = M * K, b0 = blockIdx.x * kStuDxS;
  for (int i = threadIdx.x; i < kStuDxS * 2 * MK; i += blockDim.x) {
    const int s = i / (2 * MK), r = i - s * 2 * MK, f = r / MK, mk = r - f * MK, m = mk / K, k = mk - m * K;
    const int64_t b = b0 + s;
    float v = 0.f;
    if (b < B) {
      v = g[b * M + m] * resp[((b * M + m) * 2 + f) * K + k];
      if (blockIdx.y == 0) wbuf[b * 2 * MK + r] = v;
    }
    sw[i] = v;
  }
  if (!dx) return;
  __syncthreads();
  const int e = blockIdx.y * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float xv[kStuDxS], acc[kStuDxS];
#pragma unroll
  for (int s = 0; s < kStuDxS; ++s) { xv[s] = b0 + s < B ? x[(int64_t)(b0 + s) * x_bstride + e] : 0.f; acc[s] = 0.f; }
  for (int mk = 0; mk < MK; ++mk) {
    const float4 p0 = __ldg(reinterpret_cast<const float4*>(tab + ((int64_t)mk * n + e) * 8));
    const float4 p1 = __ldg(reinterpret_cast<const float4*>(tab + ((int64_t)mk * n + e) * 8 + 4));
    const float ag = p0.y * p0.y, cs = 2.f * p1.y * p1.x;
#pragma unroll
    for (int s = 0; s < kStuDxS; ++s) {
      const float wg = sw[s * 2 * MK + mk], ws = sw[s * 2 * MK + MK + mk];
      acc[s] = fmaf(wg * ag, p0.x - xv[s], acc[s]);
      const float t = (xv[s] - p0.w) * p1.x;
      acc[s] = fmaf(ws * cs, __fdividef(t, fmaf(t, t, 1.f)), acc[s]);
    }
  }
#pragma unroll
  for (int s = 0; s < kStuDxS; ++s)
    if (b0 + s < B) dx[(int64_t)(b0 + s) * dx_bstride + e] = acc[s];
}

// Partial parameter sums over a chunk of samples: grid (n / 256, MK / kStuPT, chunks); a thread owns one element and kStuPT (m, k)
// pairs; part[chunk][mk][e] = {sum wG yg, sum wG (yg^2 - 1), sum wS u, sum wS ((df + 1) t u - 1)}
constexpr int kStuPT = 8;
__global__ void __launch_bounds__(256) student_psum_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ tab,
                                                           const float* __restrict__ wbuf, float4* __restrict__ part, int B, int MK, int n,
                                                           int per_chunk) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int mk0 = blockIdx.y * kStuPT, chunk = blockIdx.z;
  const int b0 = chunk * per_chunk, b1 = min(B, b0 + per_chunk);
  if (e >= n) return;
  float mg[kStuPT], ig[kStuPT], ms[kStuPT], is[kStuPT], nu1[kStuPT], a0[kStuPT], a1[kStuPT], a2[kStuPT], a3[kStuPT];
#pragma unroll
  for (int j = 0; j < kStuPT; ++j) {
    const int mk = min(mk0 + j, MK - 1);
    const float* t = tab + ((int64_t)mk * n + e) * 8;
    mg[j] = t[0]; ig[j] = t[1]; ms[j] = t[3]; is[j] = t[4]; nu1[j] = -2.f * t[5];
    a0[j] = a1[j] = a2[j] = a3[j] = 0.f;
  }
  for (int b = b0; b < b1; ++b) {
    const float xv = x[(int64_t)b * x_bstride + e];
    const float* w = wbuf + (int64_t)b * 2 * MK + mk0;
#pragma unroll
    for (int j = 0; j < kStuPT; ++j) {
      const bool in = mk0 + j < MK;
      const float wg = in ? __ldg(w + j) : 0.f, ws = in ? __ldg(w + MK + j) : 0.f;
      const float yg = (xv - mg[j]) * ig[j];
      a0[j] = fmaf(wg, yg, a0[j]);
      a1[j] = fmaf(wg, fmaf(yg, yg, -1.f), a1[j]);
      const float t = (xv - ms[j]) * is[j];
      const float u = __fdividef(t, fmaf(t, t, 1.f));
      a2[j] = fmaf(ws, u, a2[j]);
      a3[j] = fmaf(ws, fmaf(nu1[j] * t, u, -1.f), a3[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < kStuPT; ++j)
    if (mk0 + j < MK) part[((int64_t)chunk * MK + mk0 + j) * n + e] = make_float4(a0[j], a1[j], a2[j], a3[j]);
}

// the chunks' partial sums added in chunk order, then the per-element factors of the parameter gradients
__global__ void __launch_bounds__(256) student_finish_kernel(const float4* __restrict__ part, const float* __restrict__ tab,
                                                             const float* __restrict__ sG, const float* __restrict__ sS,
                                                             float* __restrict__ dmG, float* __restrict__ dsG, float* __restrict__ dmS,
                                                             float* __restrict__ dsS, int64_t total, int chunks) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < chunks; ++c) {
      const float4 p = part[(int64_t)c * total + i];
      s.x += p.x; s.y += p.y; s.z += p.z; s.w += p.w;
    }
    const float* t = tab + i * 8;
    const float rg = sG[i], rs = sS[i];
    dmG[i] = t[1] * s.x;
    dsG[i] = t[1] * s.y * (1.f / (1.f + expf(-rg)));
    dmS[i] = -2.f * t[5] * t[4] * s.z;
    dsS[i] = s.w / softplus_f(rs) * (1.f / (1.f + expf(-rs)));
  }
}

// G[f, mk] = sum_b w[b, f, mk], one CTA per (f, mk), fixed order
__global__ void __launch_bounds__(256) student_gsum_kernel(const float* __restrict__ wbuf, float* __restrict__ G, int B, int MK2) {
  __shared__ float red[32];
  const int i = blockIdx.x;
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) s += wbuf[(int64_t)b * MK2 + i];
  s = group_sum(s, blockDim.x, red);
  if (threadIdx.x == 0) G[i] = s;
}

// Mixture-weight gradients, one CTA per family.  logw[m, k] = log(q[m, k]), q = p / P_m, P_m = sum_k p[m, k], p = softmax over m of
// w[:, k]; with G = dL/dlogw:
//   dw[j, k] = G[j, k] - p[j, k] C_k - T_j q[j, k] + p[j, k] U_k,   C_k = sum_m G[m, k], T_m = sum_k G[m, k], U_k = sum_m T_m q[m, k].
// M = 1: p = 1 exactly, C = G and U = T q, so dw is exactly 0.
__global__ void __launch_bounds__(256) student_wgrad_kernel(const float* __restrict__ wG, const float* __restrict__ wS, const float* __restrict__ Gs,
                                                            float* __restrict__ dwG, float* __restrict__ dwS, int M, int K) {
  extern __shared__ float sh[];
  const int f = blockIdx.x, MK = M * K;
  const float* w = f ? wS : wG;
  const float* G = Gs + f * MK;
  float* dw = f ? dwS : dwG;
  float* p = sh; float* q = p + MK; float* T = q + MK; float* Cs = T + M; float* U = Cs + K;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float mx = -INFINITY;
    for (int m = 0; m < M; ++m) mx = fmaxf(mx, w[m * K + k]);
    float se = 0.f;
    for (int m = 0; m < M; ++m) se += expf(w[m * K + k] - mx);
    float c = 0.f;
    for (int m = 0; m < M; ++m) { p[m * K + k] = expf(w[m * K + k] - mx) / se; c += G[m * K + k]; }
    Cs[k] = c;
  }
  __syncthreads();
  for (int m = threadIdx.x; m < M; m += blockDim.x) {
    float P = 0.f, t = 0.f;
    for (int k = 0; k < K; ++k) { P += p[m * K + k]; t += G[m * K + k]; }
    for (int k = 0; k < K; ++k) q[m * K + k] = p[m * K + k] / P;
    T[m] = t;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float u = 0.f;
    for (int m = 0; m < M; ++m) u += T[m] * q[m * K + k];
    U[k] = u;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < MK; i += blockDim.x) {
    const int m = i / K, k = i - m * K;
    dw[i] = G[i] - p[i] * Cs[k] - T[m] * q[i] + p[i] * U[k];
  }
}

// --------------------------------------------------------------------------------------- conventional specialists, training
// a[b, c, :] = relu(a[b, c, :] + bias[b, c]) in place: the first conditioner convolution of coupling.py:47 is W1[:, :D] x0 plus the
// per-sample term b1 + W1[:, D:] CN(c)
__global__ void __launch_bounds__(256) bias_rows_relu_kernel(float* __restrict__ a, const float* __restrict__ bias, int64_t rows, int HW) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float bv = bias[row];
  for (int i = threadIdx.x & 31; i < HW; i += 32) a[row * HW + i] = fmaxf(a[row * HW + i] + bv, 0.f);
}

// dmG, dsG (M, K, D, HW): one thread per element, samples in order (deterministic):
//   mu = mG + c_m[b, m, k, d], sigma = softplus(sG + c_s[b, m, k, d]), coef = g[b, m] resp[b, m, k]
//   dmu = coef (x - mu) / sigma^2,   dspre = coef ((x - mu)^2 / sigma^3 - 1 / sigma) sigmoid(sG + c_s)
__global__ void __launch_bounds__(256) gmm_ctx_param_bwd_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ mG,
                                                                const float* __restrict__ sG, const float* __restrict__ c, const float* __restrict__ resp,
                                                                const float* __restrict__ g, float* __restrict__ dmG, float* __restrict__ dsG,
                                                                int B, int M, int K, int D, int HW) {
  const int n = D * HW, MK = M * K;
  const int e = blockIdx.x * blockDim.x + threadIdx.x, mk = blockIdx.y;
  if (e >= n) return;
  const int d = e / HW, m = mk / K;
  const float m0 = mG[(int64_t)mk * n + e], s0 = sG[(int64_t)mk * n + e];
  float am = 0.f, as = 0.f;
  for (int64_t b = 0; b < B; ++b) {
    const float coef = g[b * M + m] * resp[b * MK + mk];
    const float* cb = c + b * 2 * MK * D;
    const float mu = m0 + cb[mk * D + d], sp = s0 + cb[(int64_t)MK * D + mk * D + d];
    const float s = softplus_f(sp), inv = 1.f / s, df = x[b * x_bstride + e] - mu;
    const float r = df * inv;
    am += coef * r * inv;
    as += coef * (r * r - 1.f) * inv * (1.f / (1.f + expf(-sp)));
  }
  dmG[(int64_t)mk * n + e] = am;
  dsG[(int64_t)mk * n + e] = as;
}

// dwG[m, k] = sum_b g[b, m] (resp[b, m, k] - softmax(wG[m, :])[k])
__global__ void gmm_ctx_weight_bwd_kernel(const float* __restrict__ wG, const float* __restrict__ resp, const float* __restrict__ g,
                                          float* __restrict__ dwG, int B, int M, int K) {
  const int mk = blockIdx.x * blockDim.x + threadIdx.x;
  if (mk >= M * K) return;
  const int m = mk / K;
  float mx = -INFINITY;
  for (int j = 0; j < K; ++j) mx = fmaxf(mx, wG[m * K + j]);
  float se = 0.f;
  for (int j = 0; j < K; ++j) se += expf(wG[m * K + j] - mx);
  const float pi = expf(wG[mk] - mx) / se;
  float acc = 0.f;
  for (int64_t b = 0; b < B; ++b) acc += g[b * M + m] * (resp[b * M * K + mk] - pi);
  dwG[mk] = acc;
}

}  // namespace ex
}  // namespace cfpp
using namespace cfpp;

extern "C" int cfpp_activation_fwd(const float* x, float* z, float* ldj, const float* temperature, int64_t rows, int D, int kind, void* stream) {
  CFPP_REQUIRE((kind == 0 || kind == 1) && D >= 1 && (kind == 1 || temperature), "activation_fwd: kind=%d D=%d", kind, D);
  if (rows <= 0) return CFPP_OK;
  ex::act_fwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, z, ldj, temperature, rows, D, kind);
  return check_launch("activation_fwd");
}

extern "C" int cfpp_activation_inv(const float* z, float* x, const float* temperature, int64_t n, float eps, int kind, void* stream) {
  CFPP_REQUIRE((kind == 0 || kind == 1) && (kind == 1 || temperature), "activation_inv: kind=%d", kind);
  if (n <= 0) return CFPP_OK;
  ex::act_inv_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(z, x, temperature, n, eps, kind);
  return check_launch("activation_inv");
}

extern "C" int cfpp_activation_bwd(const float* x, const float* dz, const float* dldj, float* dx, const float* temperature, int64_t rows, int D,
                                   int kind, void* stream) {
  CFPP_REQUIRE((kind == 0 || kind == 1) && D >= 1 && (kind == 1 || temperature), "activation_bwd: kind=%d D=%d", kind, D);
  const int64_t n = rows * D;
  if (n <= 0) return CFPP_OK;
  ex::act_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, dz, dldj, dx, temperature, n, D, kind);
  return check_launch("activation_bwd");
}

extern "C" int64_t cfpp_student_table_floats(int M, int K, int n) { return ((int64_t)M * K * n) * 8 + (int64_t)2 * M * K; }

extern "C" int cfpp_student_prep(const float* mG, const float* sG, const float* wG, const float* mS, const float* sS, const float* wS,
                                 const float* vS, float* table, int M, int K, int n, void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && K <= ex::kStuMaxK && n >= 1, "student_prep: M=%d K=%d (<= %d) n=%d", M, K, ex::kStuMaxK, n);
  const int64_t tot = (int64_t)M * K * n;
  ex::student_prep_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(mG, sG, mS, sS, vS, table, tot);
  int rc = check_launch("student_prep");
  if (rc != CFPP_OK) return rc;
  ex::student_weights_kernel<<<2, 64, 0, (cudaStream_t)stream>>>(wG, wS, table + tot * 8, M, K);
  return check_launch("student_weights");
}

extern "C" int cfpp_student_logprob(const float* x, const float* table, float* logp, int B, int M, int K, int n, void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && K <= ex::kStuMaxK && n >= 1, "student_logprob: M=%d K=%d (<= %d) n=%d", M, K, ex::kStuMaxK, n);
  if (B <= 0) return CFPP_OK;
  ex::student_logprob_kernel<<<dim3(B, M), 256, 0, (cudaStream_t)stream>>>(x, n, table, table + (int64_t)M * K * n * 8, logp, nullptr, M, K, n);
  return check_launch("student_logprob");
}

extern "C" int cfpp_student_train_fwd(const float* x, int64_t x_bstride, const float* table, float* logp, float* resp, int B, int M, int K,
                                      int n, void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && K <= ex::kStuMaxK && M * K <= ex::kStuMaxMK && n >= 1 && resp,
               "student_train_fwd: M=%d K=%d (<= %d, M*K <= %d) n=%d", M, K, ex::kStuMaxK, ex::kStuMaxMK, n);
  if (B <= 0) return CFPP_OK;
  ex::student_logprob_kernel<<<dim3(B, M), 256, 0, (cudaStream_t)stream>>>(x, x_bstride, table, table + (int64_t)M * K * n * 8, logp, resp,
                                                                           M, K, n);
  return check_launch("student_train_fwd");
}

// Samples per chunk of the parameter sums: a function of the shapes only, so that a step is bit-identical run to run.  Enough chunks
// for about four CTAs per SM of a B200 at the shapes of the priors (cfg4's 26x8x1 mixture has a single CTA per chunk).
static void student_chunks(int B, int MK, int n, int* chunks, int* per_chunk) {
  const int64_t ctas = (int64_t)((n + 255) / 256) * ((MK + ex::kStuPT - 1) / ex::kStuPT);
  int64_t c = (592 + ctas - 1) / ctas;
  c = c < 8 ? 8 : (c > 512 ? 512 : c);
  if (c > B) c = B > 0 ? B : 1;
  *per_chunk = (int)((B + c - 1) / c);
  *chunks = *per_chunk > 0 ? (int)((B + *per_chunk - 1) / *per_chunk) : 1;
}

static int64_t align4(int64_t v) { return (v + 3) / 4 * 4; }

extern "C" int64_t cfpp_student_train_bwd_workspace_floats(int B, int M, int K, int n) {
  int chunks, per_chunk;
  const int MK = M * K;
  student_chunks(B, MK, n, &chunks, &per_chunk);
  return align4((int64_t)B * 2 * MK + 2 * MK) + (int64_t)chunks * MK * n * 4;
}

extern "C" int cfpp_student_train_bwd(const float* x, int64_t x_bstride, const float* table, const float* sG, const float* wG, const float* sS,
                                      const float* wS, const float* resp, const float* g, float* dx, int64_t dx_bstride, float* dmG,
                                      float* dsG, float* dwG, float* dmS, float* dsS, float* dwS, float* workspace, int B, int M, int K, int n,
                                      void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && K <= ex::kStuMaxK && M * K <= ex::kStuMaxMK && n >= 1 && B >= 1 && workspace,
               "student_train_bwd: B=%d M=%d K=%d (<= %d, M*K <= %d) n=%d", B, M, K, ex::kStuMaxK, ex::kStuMaxMK, n);
  const bool params = dmG != nullptr;
  CFPP_REQUIRE(!params || (dsG && dwG && dmS && dsS && dwS && sG && wG && sS && wS), "student_train_bwd: all six parameter gradients or none");
  const int MK = M * K;
  int chunks, per_chunk;
  student_chunks(B, MK, n, &chunks, &per_chunk);
  float* wbuf = workspace;
  float* G = wbuf + (int64_t)B * 2 * MK;
  float4* part = reinterpret_cast<float4*>(workspace + align4((int64_t)B * 2 * MK + 2 * MK));
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned eslices = dx ? (unsigned)((n + ex::kStuDxThreads - 1) / ex::kStuDxThreads) : 1u;
  ex::student_dx_kernel<<<dim3((unsigned)((B + ex::kStuDxS - 1) / ex::kStuDxS), eslices), ex::kStuDxThreads,
                          (size_t)ex::kStuDxS * 2 * MK * sizeof(float), st>>>(x, x_bstride, table, resp, g, wbuf, dx, dx_bstride, B, M, K, n);
  int rc = check_launch("student_train_dx");
  if (rc != CFPP_OK || !params) return rc;
  ex::student_psum_kernel<<<dim3((n + 255) / 256, (MK + ex::kStuPT - 1) / ex::kStuPT, chunks), 256, 0, st>>>(x, x_bstride, table, wbuf, part,
                                                                                                            B, MK, n, per_chunk);
  if ((rc = check_launch("student_train_psum")) != CFPP_OK) return rc;
  const int64_t total = (int64_t)MK * n;
  ex::student_finish_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(part, table, sG, sS, dmG, dsG, dmS, dsS, total, chunks);
  if ((rc = check_launch("student_train_finish")) != CFPP_OK) return rc;
  ex::student_gsum_kernel<<<2 * MK, 256, 0, st>>>(wbuf, G, B, 2 * MK);
  if ((rc = check_launch("student_train_gsum")) != CFPP_OK) return rc;
  ex::student_wgrad_kernel<<<2, 256, (size_t)(2 * MK + M + 2 * K) * sizeof(float), st>>>(wG, wS, G, dwG, dwS, M, K);
  return check_launch("student_train_wgrad");
}

extern "C" int cfpp_bias_rows_relu(float* a, const float* bias, int B, int C, int HW, void* stream) {
  CFPP_REQUIRE(C >= 1 && HW >= 1, "bias_rows_relu: C=%d HW=%d", C, HW);
  const int64_t rows = (int64_t)B * C;
  if (rows <= 0) return CFPP_OK;
  ex::bias_rows_relu_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(a, bias, rows, HW);
  return check_launch("bias_rows_relu");
}

extern "C" int cfpp_gmm_ctx_param_bwd(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG, const float* c,
                                      const float* resp, const float* g, float* dmG, float* dsG, float* dwG, int B, int M, int K, int D, int HW,
                                      void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && D >= 1 && HW >= 1 && c && dmG && dsG && dwG, "gmm_ctx_param_bwd: M=%d K=%d D=%d HW=%d", M, K, D, HW);
  const int n = D * HW;
  ex::gmm_ctx_param_bwd_kernel<<<dim3((n + 255) / 256, M * K), 256, 0, (cudaStream_t)stream>>>(x, x_bstride, mG, sG, c, resp, g, dmG, dsG, B, M, K, D, HW);
  int rc = check_launch("gmm_ctx_param_bwd");
  if (rc != CFPP_OK) return rc;
  ex::gmm_ctx_weight_bwd_kernel<<<(M * K + 127) / 128, 128, 0, (cudaStream_t)stream>>>(wG, resp, g, dwG, B, M, K);
  return check_launch("gmm_ctx_weight_bwd");
}
