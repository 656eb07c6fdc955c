// Training direction (SURVEY §8f-1): the activation-saving conditioner forward and the backward kernels of the context-free
// (generalist) conv stack -- Coupling (layers/coupling.py:39-66), its conv conditioner (:26-29), ActNorm (layers/actnorm.py:37-60),
// Conv1x1 (layers/conv1x1.py:52-55), the mixture base (layers/distributions/gaussian.py:142-161) and the (B,M) log-det accumulation
// (layers/flowsequential.py:20-27).  What the reference obtains from torch autograd over experiment_ad.py:204-213.
// First version: FP32 CUDA cores, one CTA per sample with the sample resident in shared memory; every reduction over the batch is
// two-stage with a fixed order (no atomics): gradients are bit-identical run to run.
#include <math.h>
#include <stdlib.h>
#include <stdint.h>
#include "common.cuh"

namespace cfpp {
namespace bw {

__device__ __forceinline__ int reflect_idx(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

// ---------------------------------------------------------------------------------------------------------------
// Coupling backward.  Forward: t = h[:, :Ch], r = h[:, Ch:]; ls = 2 tanh(r/2); z1 = x1 e^{ls} + t; ldj = sum ls.
//   dx0 = dz0 (the conditioner's contribution is added by its own backward); dx1 = dz1 e^{ls};
//   dt = dz1; dr = (dz1 x1 e^{ls} + dldj[b]) (1 - tanh^2(r/2)).          20*C*HW bytes per sample.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) coupling_bwd_kernel(const float* __restrict__ x, const float* __restrict__ h, const float* __restrict__ add,
                                                           const float* __restrict__ dz, const float* __restrict__ dldj,
                                                           float* __restrict__ dx, float* __restrict__ dh, int B, int C, int HW, int G) {
  const int spc = blockDim.x / G;
  const int s = threadIdx.x / G, g = threadIdx.x % G;
  const int64_t b = (int64_t)blockIdx.x * spc + s;
  if (b >= B) return;
  const int64_t n = (int64_t)(C / 2) * HW;
  const float* xb = x + b * 2 * n; const float* hb = h + b * 2 * n; const float* gb = dz + b * 2 * n;
  float* dxb = dx + b * 2 * n; float* dhb = dh + b * 2 * n;
  const float gl = dldj ? dldj[b] : 0.f;
  const float* ab = add ? add + b * C + C / 2 : nullptr;        // additive context term of the scale half (coupling.py:45)
  for (int64_t i = g; i < n; i += G) {
    const float r = hb[n + i] + (ab ? ab[i / HW] : 0.f), x1 = xb[n + i], g0 = gb[i], g1 = gb[n + i];
    const float th = tanhf(r * 0.5f);
    const float sc = expf(2.0f * th);
    dxb[i] = g0;
    dxb[n + i] = g1 * sc;
    dhb[i] = g1;
    dhb[n + i] = (g1 * x1 * sc + gl) * (1.0f - th * th);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// ActNorm backward (context-free).  Forward: z = (x - t) e^{-logs}; ldj[b] = sum_d logs.
//   dx = dz e^{-logs};  dt[d] = -sum_{b,p} dz e^{-logs};  dlogs[d] = -sum_{b,p} dz z + sum_b dldj[b].
// grid (D, chunks): a CTA walks channel d of a contiguous chunk of samples; partial[(chunk*D + d)*2 + {0,1}]; finish sums in order.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) actnorm_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dz,
                                                          const float* __restrict__ t, const float* __restrict__ logs,
                                                          float* __restrict__ dx, float* __restrict__ partial, int B, int D, int HW, int per_chunk) {
  __shared__ float red[32];
  const int d = blockIdx.x, chunk = blockIdx.y;
  const int b0 = chunk * per_chunk, b1 = min(B, b0 + per_chunk);
  const float e = expf(-logs[d]), tt = t[d];
  float a0 = 0.f, a1 = 0.f;
  const int64_t total = (int64_t)(b1 - b0) * HW;
  for (int64_t i = threadIdx.x; i < total; i += blockDim.x) {
    const int64_t b = b0 + i / HW; const int p = (int)(i % HW);
    const int64_t o = (b * D + d) * HW + p;
    const float g = dz[o], ge = g * e;
    if (dx) dx[o] = ge;
    a0 -= ge;
    a1 -= g * ((x[o] - tt) * e);
  }
  a0 = group_sum(a0, blockDim.x, red);
  a1 = group_sum(a1, blockDim.x, red);
  if (threadIdx.x == 0) { partial[((int64_t)chunk * D + d) * 2] = a0; partial[((int64_t)chunk * D + d) * 2 + 1] = a1; }
}

__global__ void actnorm_bwd_finish_kernel(const float* __restrict__ partial, const float* __restrict__ dldj, float* __restrict__ dt,
                                          float* __restrict__ dlogs, int B, int D, int chunks) {
  __shared__ float red[32];
  float s = 0.f;                                                    // sum_b dldj[b], fixed order per thread then tree
  if (dldj) for (int b = threadIdx.x; b < B; b += blockDim.x) s += dldj[b];
  s = group_sum(s, blockDim.x, red);
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float a0 = 0.f, a1 = 0.f;
    for (int c = 0; c < chunks; ++c) { a0 += partial[((int64_t)c * D + d) * 2]; a1 += partial[((int64_t)c * D + d) * 2 + 1]; }
    dt[d] = a0; dlogs[d] = a1 + s;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Generic small convolution family, NCHW, "same" reflect padding (KH, KW in {1,3}), torch weight layout (Cout, Cin, KH, KW).
// One CTA per sample; the sample's input planes live in shared memory.  Used for the conditioner in training mode (the three
// convolutions as separate launches so that the post-ReLU activations are saved) and, with 1x1 kernels, for Conv1x1's backward.
// ---------------------------------------------------------------------------------------------------------------
constexpr int CG = 4;        // channels per thread
constexpr int PXT = 4;       // pixels per thread

__host__ __device__ inline int odd_stride(int n) { return n | 1; }   // odd row strides: channel rows start in different banks

// Stage the first C channels of sample b with a reflect halo of (PH, PW): dst[c * S + (y + PH) * Wp + (x + PW)], Wp = W + 2 PW.
template <int PH, int PW>
__device__ __forceinline__ void stage_reflect(float* dst, const float* __restrict__ src, int C, int H, int Wd, int S, bool relu_in = false) {
  const int Hp = H + 2 * PH, Wp = Wd + 2 * PW, HW = H * Wd;
  for (int i = threadIdx.x; i < C * Hp * Wp; i += blockDim.x) {
    const int c = i / (Hp * Wp), r = i - c * (Hp * Wp);
    const int yp = r / Wp, xp = r - yp * Wp;
    const float v = src[c * HW + reflect_idx(yp - PH, H) * Wd + reflect_idx(xp - PW, Wd)];
    dst[c * S + r] = relu_in ? fmaxf(v, 0.f) : v;
  }
}

// out[b,co,p] = [relu](bias[co] + sum_{ci,kh,kw} W[co,ci,kh,kw] in[b,ci,reflect(p + (kh,kw) - pad)]).
// Thread = PXT pixels x CG output channels: per (ci, tap) 4 warp-uniform weight loads + 4 shared loads feed 16 FMAs.
template <int KH, int KW>
__global__ void __launch_bounds__(256) conv2d_fwd_kernel(const float* __restrict__ in, int64_t in_bstride, const float* __restrict__ W,
                                                         const float* __restrict__ bias, float* __restrict__ out,
                                                         int Cin, int Cout, int H, int Wd, int relu) {
  constexpr int PH = KH / 2, PW = KW / 2, KK = KH * KW;
  extern __shared__ float sm[];
  const int HW = H * Wd, Wp = Wd + 2 * PW, S = odd_stride((H + 2 * PH) * Wp);
  const int64_t b = blockIdx.x;
  stage_reflect<PH, PW>(sm, in + b * in_bstride, Cin, H, Wd, S, (relu & 2) != 0);     // relu bit 1: ReLU on the INPUT (pre-activation blocks)
  relu &= 1;                                                                           // relu bit 0: ReLU on the output
  __syncthreads();
  const int ncg = (Cout + CG - 1) / CG, nslot = (HW + PXT - 1) / PXT;
  for (int item = threadIdx.x; item < nslot * ncg; item += blockDim.x) {
    const int slot = item % nslot, co0 = (item / nslot) * CG;
    int pb[PXT];
#pragma unroll
    for (int j = 0; j < PXT; ++j) { int p = slot + j * nslot; if (p >= HW) p = HW - 1; const int y = p / Wd; pb[j] = y * Wp + (p - y * Wd); }
    float acc[PXT][CG];
#pragma unroll
    for (int c = 0; c < CG; ++c) {
      const float bv = (bias && co0 + c < Cout) ? bias[co0 + c] : 0.f;
#pragma unroll
      for (int j = 0; j < PXT; ++j) acc[j][c] = bv;
    }
    const int nc = min(CG, Cout - co0);
    for (int ci = 0; ci < Cin; ++ci) {
      const float* sp = sm + ci * S;
      const float* wp = W + ((int64_t)co0 * Cin + ci) * KK;
#pragma unroll
      for (int kh = 0; kh < KH; ++kh)
#pragma unroll
        for (int kw = 0; kw < KW; ++kw) {
          float w[CG];
#pragma unroll
          for (int c = 0; c < CG; ++c) w[c] = c < nc ? __ldg(wp + (int64_t)c * Cin * KK + kh * KW + kw) : 0.f;
#pragma unroll
          for (int j = 0; j < PXT; ++j) {
            const float v = sp[pb[j] + kh * Wp + kw];
#pragma unroll
            for (int c = 0; c < CG; ++c) acc[j][c] = fmaf(w[c], v, acc[j][c]);
          }
        }
    }
#pragma unroll
    for (int j = 0; j < PXT; ++j) {
      const int p = slot + j * nslot;
      if (p >= HW) continue;
#pragma unroll
      for (int c = 0; c < CG; ++c)
        if (c < nc) out[(b * Cout + co0 + c) * HW + p] = relu ? fmaxf(acc[j][c], 0.f) : acc[j][c];
    }
  }
}

// Gradient w.r.t. the convolution's input.  Phase 1: dpad[ci,u] = sum_{co,kh,kw} W[co,ci,kh,kw] dout0[co, u - (kh,kw)] over the PADDED
// domain u (dout staged with a zero halo of (KH-1, KW-1), so no bounds checks), register tile PXT x CG, into shared memory.
// Phase 2: fold the reflect halo back (the adjoint of reflect padding): din[q] = sum of dpad over the positions that read q,
// times (act > 0), stored or accumulated.  With 1x1 kernels phase 1 writes straight to global memory.
template <int KH, int KW>
__global__ void __launch_bounds__(256) conv2d_bwd_data_kernel(const float* __restrict__ dout, const float* __restrict__ W,
                                                              const float* __restrict__ act, int64_t act_bstride,
                                                              float* __restrict__ din, int64_t din_bstride, int accumulate,
                                                              int Cin, int Cout, int H, int Wd) {
  constexpr int PH = KH / 2, PW = KW / 2, KK = KH * KW, ZH = KH - 1, ZW = KW - 1;
  extern __shared__ float sm[];
  const int HW = H * Wd;
  const int Hp = H + 2 * PH, Wp = Wd + 2 * PW;                 // padded domain of the forward input
  const int Hz = H + 2 * ZH, Wz = Wd + 2 * ZW;                 // dout with a zero halo
  const int Sz = odd_stride(Hz * Wz), Sp = odd_stride(Hp * Wp);
  float* sz = sm;                                              // Cout * Sz
  float* spad = sm + Cout * Sz;                                // Cin * Sp (unused for 1x1)
  const int64_t b = blockIdx.x;
  if (KK == 1 && (HW & 3) == 0 && (reinterpret_cast<uintptr_t>(dout) & 15) == 0) {
    // no halo: a straight copy.  128-bit loads, four per thread in flight -- with one scalar load per thread and iteration the kernel ran at
    // the latency of its own staging loop (0.6 TB/s at B = 8192 on the conditioner's 1x1 layers)
    const float4* src4 = reinterpret_cast<const float4*>(dout + b * (int64_t)Cout * HW);
    const int n4 = Cout * HW / 4, step = blockDim.x;
    for (int i0 = threadIdx.x; i0 < n4; i0 += 4 * step) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = i0 + u * step < n4 ? __ldg(src4 + i0 + u * step) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = 4 * (i0 + u * step);
        if (e < 4 * n4) { const int c = e / HW; float* d = sz + c * Sz + (e - c * HW); d[0] = v[u].x; d[1] = v[u].y; d[2] = v[u].z; d[3] = v[u].w; }
      }
    }
  } else {
    for (int i = threadIdx.x; i < Cout * Hz * Wz; i += blockDim.x) {
      const int c = i / (Hz * Wz), r = i - c * (Hz * Wz);
      const int y = r / Wz - ZH, x = r % Wz - ZW;
      sz[c * Sz + r] = (y >= 0 && y < H && x >= 0 && x < Wd) ? dout[(b * Cout + c) * HW + y * Wd + x] : 0.f;
    }
  }
  __syncthreads();
  const int NP = Hp * Wp;
  const int ncg = (Cin + CG - 1) / CG, nslot = (NP + PXT - 1) / PXT;
  for (int item = threadIdx.x; item < nslot * ncg; item += blockDim.x) {
    const int slot = item % nslot, ci0 = (item / nslot) * CG;
    int ub[PXT];
#pragma unroll
    for (int j = 0; j < PXT; ++j) {
      int u = slot + j * nslot; if (u >= NP) u = NP - 1;
      const int uy = u / Wp, ux = u - uy * Wp;
      ub[j] = (uy + ZH) * Wz + (ux + ZW);                      // dout0 index of tap (0,0); tap (kh,kw) reads ub - kh*Wz - kw
    }
    float acc[PXT][CG];
#pragma unroll
    for (int j = 0; j < PXT; ++j)
#pragma unroll
      for (int c = 0; c < CG; ++c) acc[j][c] = 0.f;
    const int nc = min(CG, Cin - ci0);
    for (int co = 0; co < Cout; ++co) {
      const float* gp = sz + co * Sz;
      const float* wp = W + ((int64_t)co * Cin + ci0) * KK;
#pragma unroll
      for (int kh = 0; kh < KH; ++kh)
#pragma unroll
        for (int kw = 0; kw < KW; ++kw) {
          float w[CG];
#pragma unroll
          for (int c = 0; c < CG; ++c) w[c] = c < nc ? __ldg(wp + c * KK + kh * KW + kw) : 0.f;
#pragma unroll
          for (int j = 0; j < PXT; ++j) {
            const float g = gp[ub[j] - kh * Wz - kw];
#pragma unroll
            for (int c = 0; c < CG; ++c) acc[j][c] = fmaf(w[c], g, acc[j][c]);
          }
        }
    }
#pragma unroll
    for (int j = 0; j < PXT; ++j) {
      const int u = slot + j * nslot;
      if (u >= NP) continue;
#pragma unroll
      for (int c = 0; c < CG; ++c) {
        if (c >= nc) continue;
        if (KK == 1) {
          float v = acc[j][c];
          if (act && !(act[b * act_bstride + (int64_t)(ci0 + c) * HW + u] > 0.f)) v = 0.f;
          float* o = din + b * din_bstride + (int64_t)(ci0 + c) * HW + u;
          *o = accumulate ? *o + v : v;
        } else {
          spad[(ci0 + c) * Sp + u] = acc[j][c];
        }
      }
    }
  }
  if (KK == 1) return;
  __syncthreads();
  for (int i = threadIdx.x; i < Cin * HW; i += blockDim.x) {
    const int ci = i / HW, q = i - ci * HW;
    const int qy = q / Wd, qx = q - qy * Wd;
    int uy[3], ux[3]; int ny = 0, nx = 0;                      // padded rows / columns whose reflection is (qy, qx)
    uy[ny++] = qy + PH; if (PH == 1 && qy == 1) uy[ny++] = 0; if (PH == 1 && qy == H - 2) uy[ny++] = H + 1;
    ux[nx++] = qx + PW; if (PW == 1 && qx == 1) ux[nx++] = 0; if (PW == 1 && qx == Wd - 2) ux[nx++] = Wd + 1;
    float v = 0.f;
    for (int a = 0; a < ny; ++a)
      for (int c = 0; c < nx; ++c) v += spad[ci * Sp + uy[a] * Wp + ux[c]];
    if (act && !(act[b * act_bstride + (int64_t)ci * HW + q] > 0.f)) v = 0.f;
    float* o = din + b * din_bstride + (int64_t)ci * HW + q;
    *o = accumulate ? *o + v : v;
  }
}

// H = W = 1 with a 1x1 kernel: the FC / CouplingFC layers of the context-encoder flows (`x.view(-1, D, 1, 1)`, coupling.py:83-91 of the
// reference) at widths of 10-40 channels.  One CTA per sample would leave 256 threads with a few hundred MACs and a grid of B CTAs per
// launch (36 encoders x 14 such launches per training step); here a CTA takes kRowsPerCta samples as rows of a small matrix product:
//   FWD : out[b, o] = [relu](bias[o] + sum_i W[o, i] [relu_in](in[b, i]))          (o = co, i = ci)
//   !FWD: out[b, o] (+)= [act[b, o] > 0] sum_i W[i, o] in[b, i]                    (o = ci, i = co: the gradient w.r.t. the input)
// the weight matrix sits in shared memory as [i][o] (threads of a warp = consecutive o: conflict-free), the sample rows as [s][i].
// Summation order per output = i ascending, as in the per-sample kernels (bit-identical results).
constexpr int kRowsPerCta = 16;                                // 512 CTAs at B = 8192: the launch is latency-bound, not work-bound
template <bool FWD>
__global__ void __launch_bounds__(256) conv_rows_kernel(const float* __restrict__ in, int64_t in_bstride, const float* __restrict__ W,
                                                        const float* __restrict__ bias, const float* __restrict__ act, int64_t act_bstride,
                                                        float* __restrict__ out, int64_t out_bstride, int accumulate,
                                                        int B, int NI, int NO, int relu) {
  extern __shared__ float smr[];
  const int NOp = NO | 1, NIp = NI | 1;
  float* Ms = smr;                                             // [NI][NOp]
  float* Xs = smr + (size_t)NI * NOp;                          // [kRowsPerCta][NIp]
  const int64_t b0 = (int64_t)blockIdx.x * kRowsPerCta;
  const int nS = (int)min((int64_t)kRowsPerCta, (int64_t)B - b0);
  for (int idx = threadIdx.x; idx < NI * NO; idx += 256) {
    const int o = FWD ? idx / NI : idx % NO, i = FWD ? idx - o * NI : idx / NO;      // W is (Cout, Cin): FWD (o, i), else (i, o); idx runs along W
    Ms[i * NOp + o] = __ldg(W + idx);
  }
  const bool relu_in = FWD && (relu & 2) != 0;
  for (int idx = threadIdx.x; idx < nS * NI; idx += 256) {
    const int sI = idx / NI, i = idx - sI * NI;
    const float v = __ldg(in + (b0 + sI) * in_bstride + i);
    Xs[sI * NIp + i] = relu_in ? fmaxf(v, 0.f) : v;
  }
  __syncthreads();
  for (int item = threadIdx.x; item < nS * NO; item += 256) {
    const int sI = item / NO, o = item - sI * NO;
    const float* xr = Xs + sI * NIp;
    const float* mr = Ms + o;
    float acc = (FWD && bias) ? __ldg(bias + o) : 0.f;
    for (int i = 0; i < NI; ++i) acc = fmaf(mr[i * NOp], xr[i], acc);
    const int64_t b = b0 + sI;
    if (FWD) {
      out[b * out_bstride + o] = (relu & 1) ? fmaxf(acc, 0.f) : acc;
    } else {
      if (act && !(act[b * act_bstride + o] > 0.f)) acc = 0.f;
      float* op = out + b * out_bstride + o;
      *op = accumulate ? *op + acc : acc;
    }
  }
}

// Weight / bias gradient of the same H = W = 1 layers: dW[co, ci] = sum_b dout[b, co] in[b, ci], db[co] = sum_b dout[b, co].  A CTA owns a
// chunk of samples (tiles of kRowsW rows of `in` and `dout` staged in shared memory), a thread up to 8 entries of dW; the chunks' partial
// sums go to the workspace and chunk_sum_kernel adds them in a fixed order (deterministic, no atomics) -- the per-sample family's scheme
// with 64 samples per CTA instead of ~14 spread over 256 mostly idle threads.
constexpr int kRowsW = 64, kRowsWEntries = 8;
__global__ void __launch_bounds__(256) conv_rows_bwd_weight_kernel(const float* __restrict__ in, int64_t in_bstride, const float* __restrict__ dout,
                                                                   float* __restrict__ partW, float* __restrict__ partb,
                                                                   int B, int Cin, int Cout, int per_chunk) {
  extern __shared__ float smw[];
  const int CIp = Cin | 1, COp = Cout | 1, nW = Cin * Cout;
  float* Xs = smw;                                             // [kRowsW][CIp]
  float* Gs = smw + (size_t)kRowsW * CIp;                      // [kRowsW][COp]
  const int tid = threadIdx.x;
  const int64_t b_lo = (int64_t)blockIdx.x * per_chunk;
  const int64_t b_hi = min((int64_t)B, b_lo + per_chunk);
  int xo[kRowsWEntries], go[kRowsWEntries];
  float acc[kRowsWEntries];
#pragma unroll
  for (int k = 0; k < kRowsWEntries; ++k) {
    const int idx = tid + k * 256, co = idx < nW ? idx / Cin : 0;
    go[k] = co; xo[k] = idx < nW ? idx - co * Cin : 0; acc[k] = 0.f;
  }
  float accb = 0.f;
  for (int64_t b0 = b_lo; b0 < b_hi; b0 += kRowsW) {
    const int nS = (int)min((int64_t)kRowsW, b_hi - b0);
    for (int idx = tid; idx < nS * Cin; idx += 256) { const int sI = idx / Cin, i = idx - sI * Cin; Xs[sI * CIp + i] = __ldg(in + (b0 + sI) * in_bstride + i); }
    for (int idx = tid; idx < nS * Cout; idx += 256) { const int sI = idx / Cout, o = idx - sI * Cout; Gs[sI * COp + o] = __ldg(dout + (b0 + sI) * Cout + o); }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kRowsWEntries; ++k) {
      if (tid + k * 256 < nW) {
        const float* gp = Gs + go[k];
        const float* xp = Xs + xo[k];
        float a = acc[k];
        for (int sI = 0; sI < nS; ++sI) a = fmaf(gp[sI * COp], xp[sI * CIp], a);
        acc[k] = a;
      }
    }
    if (partb && tid < Cout) for (int sI = 0; sI < nS; ++sI) accb += Gs[sI * COp + tid];
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < kRowsWEntries; ++k)
    if (tid + k * 256 < nW) partW[(int64_t)blockIdx.x * nW + tid + k * 256] = acc[k];
  if (partb && tid < Cout) partb[(int64_t)blockIdx.x * Cout + tid] = accb;
}

// Register-tiled 3x3 form of the kernel above (the conditioner's middle convolution: 94 % of its backward-data flops).  Same two phases
// and the same summation order per output (co outer, taps inner: results are bit-identical to the generic tile), but a thread owns TP
// CONSECUTIVE padded positions of one row x 4 input channels.  Per output channel co: 3 rows x (TP + 2) staged gradients arrive by
// 128/64-bit shared loads (rows of WzP columns, a multiple of 4, so every group starts 16-byte aligned) and the 4 x 9 weights
// W[co, ci0..ci0+3, :, :] are 36 contiguous floats = nine 128-bit warp-uniform loads; together they feed 36 TP FMAs (TP = 4: 144 FMAs per 15
// loads, against 16 per 8 in the generic tile).  TP = 6 covers a whole padded row of a 4-wide image with one group.
template <int TP>
__global__ void __launch_bounds__(256, 2) conv2d_bwd_data3_kernel(const float* __restrict__ dout, const float* __restrict__ W,
                                                                  const float* __restrict__ act, int64_t act_bstride,
                                                                  float* __restrict__ din, int64_t din_bstride, int accumulate,
                                                                  int Cin, int Cout, int H, int Wd, int NG, int WzP) {
  constexpr int NV = TP + 2;                                   // staged gradients per row that TP positions x 3 column taps read
  extern __shared__ __align__(16) float sm3[];
  const int HW = H * Wd, Hp = H + 2, Wp = Wd + 2, Hz = H + 4;
  const int SzC = Hz * WzP, Sp = odd_stride(Hp * Wp);
  float* sz = sm3;                                             // [Cout][Hz][WzP]: dout at (y + 2, x + 2), zeros elsewhere
  float* spad = sm3 + (size_t)Cout * SzC + 4;                  // [Cin][Sp]; the 4 floats between are zero: with TP = 4 rows are stored WITHOUT
                                                               // padding (WzP = 4 NG: the groups of a warp read consecutive 16-byte chunks, no bank
                                                               // conflicts) and the last group's two extra columns wrap into the next row's zero halo
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x;
  {   // stage dout: LPR lanes per staged row (a power of two >= WzP when WzP <= 32), four rows in flight per thread
    const int LPR = WzP <= 8 ? 8 : WzP <= 16 ? 16 : 32, RPW = 32 / LPR;
    const int lane = tid & 31, warp = tid >> 5;
    const int lr = lane / LPR, lc = lane - lr * LPR;
    const int rows = Cout * Hz, rstep = 8 * RPW;
    const float* src0 = dout + b * (int64_t)Cout * HW;
    if (tid < 4) sz[(size_t)Cout * SzC + tid] = 0.f;
    for (int col = lc; col < WzP; col += LPR) {
      const int x = col - 2;
      const bool xin = x >= 0 && x < Wd;
      for (int row0 = warp * RPW + lr; row0 < rows; row0 += 4 * rstep) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int row = row0 + u * rstep;
          const int c = row / Hz, y = row - c * Hz - 2;
          v[u] = (row < rows && xin && y >= 0 && y < H) ? __ldg(src0 + ((int64_t)c * H + y) * Wd + x) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int row = row0 + u * rstep;
          if (row < rows) sz[(size_t)row * WzP + col] = v[u];
        }
      }
    }
  }
  __syncthreads();
  const int npg = Hp * NG, nitems = npg * (Cin >> 2);
  for (int item = tid; item < nitems; item += 256) {
    const int cg = item / npg, pgi = item - cg * npg;
    const int uy = pgi / NG, ux0 = (pgi - uy * NG) * TP, ci0 = cg * 4;
    const float* gp = sz + uy * WzP + ux0;                     // tap row kh reads staged row uy + 2 - kh, tap column kw reads column ux + 2 - kw
    const float4* wq = reinterpret_cast<const float4*>(W + (int64_t)ci0 * 9);
    const int wstep = Cin * 9 / 4;                             // float4s between consecutive co (Cin % 4 == 0)
    float acc[4][TP];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int j = 0; j < TP; ++j) acc[c][j] = 0.f;
    float4 wn[9];                                              // the weights of the next output channel are requested one iteration ahead
#pragma unroll
    for (int q = 0; q < 9; ++q) wn[q] = __ldg(wq + q);
#pragma unroll 2
    for (int co = 0; co < Cout; ++co) {                        // unrolled by two: the (w, wn) register sets swap roles instead of being copied
      float w[36];
#pragma unroll
      for (int q = 0; q < 9; ++q) { w[4 * q] = wn[q].x; w[4 * q + 1] = wn[q].y; w[4 * q + 2] = wn[q].z; w[4 * q + 3] = wn[q].w; }
      wq += co + 1 < Cout ? wstep : 0;                         // the last iteration re-reads its own row (in bounds, unused)
#pragma unroll
      for (int q = 0; q < 9; ++q) wn[q] = __ldg(wq + q);
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        const float* r = gp + (2 - kh) * WzP;
        float v[NV];
        {
          const float4 t = *reinterpret_cast<const float4*>(r);
          v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        }
        if (NV == 6) { const float2 t = *reinterpret_cast<const float2*>(r + 4); v[4] = t.x; v[5] = t.y; }
        else { const float4 t = *reinterpret_cast<const float4*>(r + 4); v[4] = t.x; v[5] = t.y; v[NV - 2] = t.z; v[NV - 1] = t.w; }
#pragma unroll
        for (int kw = 0; kw < 3; ++kw)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float wv = w[c * 9 + kh * 3 + kw];
#pragma unroll
            for (int j = 0; j < TP; ++j) acc[c][j] = fmaf(wv, v[j + 2 - kw], acc[c][j]);
          }
      }
      gp += SzC;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int j = 0; j < TP; ++j)
        if (ux0 + j < Wp) spad[(ci0 + c) * Sp + uy * Wp + ux0 + j] = acc[c][j];
  }
  __syncthreads();
#pragma unroll 4
  for (int i = tid; i < Cin * HW; i += 256) {                  // fold the reflect halo back, mask, store (the generic kernel's summation order)
    const int ci = i / HW, q = i - ci * HW;
    const int qy = q / Wd, qx = q - qy * Wd;
    const float* sp = spad + ci * Sp;
    auto rowsum = [&](int uyv, float v) {
      const float* r = sp + uyv * Wp;
      v += r[qx + 1];
      if (qx == 1) v += r[0];
      if (qx == Wd - 2) v += r[Wd + 1];
      return v;
    };
    float v = rowsum(qy + 1, 0.f);
    if (qy == 1) v = rowsum(0, v);
    if (qy == H - 2) v = rowsum(H + 1, v);
    if (act && !(__ldg(act + b * act_bstride + (int64_t)ci * HW + q) > 0.f)) v = 0.f;
    float* o = din + b * din_bstride + (int64_t)ci * HW + q;
    *o = accumulate ? *o + v : v;
  }
}

// dW[co,ci,tap] += sum_{b in chunk, p} dout[b,co,p] in[b,ci,reflect(p + tap - pad)];  db[co] += sum dout.
// grid (chunks, co blocks).  A CTA stages, per sample, the reflect-padded input planes and NCO rows of dout; thread = one input
// channel x PPT output channels (the 3x3 input window is loaded once per pixel and reused by the PPT rows), accumulators live in
// registers across the samples of the chunk, then one store per weight into the chunk's slice of the workspace; a finishing kernel adds
// the chunks in order, so the gradient is bit-identical run to run (no atomics).
constexpr int PPT = 4;

template <int KH, int KW>
__global__ void __launch_bounds__(256) conv2d_bwd_weight_kernel(const float* __restrict__ in, int64_t in_bstride, const float* __restrict__ dout,
                                                                float* __restrict__ dW, float* __restrict__ db,
                                                                int B, int Cin, int Cout, int H, int Wd, int NCO, int per_chunk) {
  // dW / db here are the workspace slices: [chunk][Cout*Cin*KK] and [chunk][Cout]
  constexpr int PH = KH / 2, PW = KW / 2, KK = KH * KW;
  dW += (int64_t)blockIdx.x * Cout * Cin * KK;
  if (db) db += (int64_t)blockIdx.x * Cout;
  extern __shared__ float sm[];
  const int HW = H * Wd, Wp = Wd + 2 * PW, S = odd_stride((H + 2 * PH) * Wp), Sg = odd_stride(HW);
  float* sin_ = sm;                                   // Cin * S
  float* sd = sm + Cin * S;                           // NCO * Sg
  const int co0 = blockIdx.y * NCO;
  const int nco = min(NCO, Cout - co0);
  const int b0 = blockIdx.x * per_chunk, b1 = min(B, b0 + per_chunk);
  const int cpp = 256 / Cin;                          // output channels covered per pass of the CTA (Cin <= 256)
  const int ci = threadIdx.x % Cin, cog = threadIdx.x / Cin;
  const bool live = cog < cpp;
  float acc[PPT][KK];
#pragma unroll
  for (int k = 0; k < PPT; ++k)
#pragma unroll
    for (int t = 0; t < KK; ++t) acc[k][t] = 0.f;
  float bsum = 0.f;
  for (int b = b0; b < b1; ++b) {
    __syncthreads();
    stage_reflect<PH, PW>(sin_, in + (int64_t)b * in_bstride, Cin, H, Wd, S);
    for (int i = threadIdx.x; i < nco * HW; i += blockDim.x) { const int c = i / HW; sd[c * Sg + (i - c * HW)] = dout[((int64_t)b * Cout + co0) * HW + i]; }
    __syncthreads();
    if ((int)threadIdx.x < nco) { float s = 0.f; for (int p = 0; p < HW; ++p) s += sd[threadIdx.x * Sg + p]; bsum += s; }
    if (!live) continue;
    const float* ip = sin_ + ci * S;
    const float* gp[PPT];
    bool on[PPT];
#pragma unroll
    for (int k = 0; k < PPT; ++k) { const int co = cog + k * cpp; on[k] = co < nco; gp[k] = sd + (on[k] ? co : 0) * Sg; }
    if (on[PPT - 1]) {                                   // all PPT output channels of this thread exist
      for (int y = 0; y < H; ++y)
        for (int x = 0; x < Wd; ++x) {
          float v[KK];
#pragma unroll
          for (int kh = 0; kh < KH; ++kh)
#pragma unroll
            for (int kw = 0; kw < KW; ++kw) v[kh * KW + kw] = ip[(y + kh) * Wp + x + kw];
          const int p = y * Wd + x;
#pragma unroll
          for (int k = 0; k < PPT; ++k) {
            const float g = gp[k][p];
#pragma unroll
            for (int t = 0; t < KK; ++t) acc[k][t] = fmaf(g, v[t], acc[k][t]);
          }
        }
    } else {                                             // narrow layers (Cout < channels per pass x PPT): only the live ones
      for (int y = 0; y < H; ++y)
        for (int x = 0; x < Wd; ++x) {
          float v[KK];
#pragma unroll
          for (int kh = 0; kh < KH; ++kh)
#pragma unroll
            for (int kw = 0; kw < KW; ++kw) v[kh * KW + kw] = ip[(y + kh) * Wp + x + kw];
          const int p = y * Wd + x;
#pragma unroll
          for (int k = 0; k < PPT; ++k) {
            if (!on[k]) break;
            const float g = gp[k][p];
#pragma unroll
            for (int t = 0; t < KK; ++t) acc[k][t] = fmaf(g, v[t], acc[k][t]);
          }
        }
    }
  }
  if (live) {
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
      const int co = cog + k * cpp;
      if (co >= nco) continue;
#pragma unroll
      for (int t = 0; t < KK; ++t) dW[((int64_t)(co0 + co) * Cin + ci) * KK + t] = acc[k][t];
    }
  }
  if (db && (int)threadIdx.x < nco) db[co0 + threadIdx.x] = bsum;
}

// out[i] = sum_c part[c][i]: a CTA covers 32 consecutive outputs; warp w sums chunks w, w+8, ..., the eight warp partials are added
// in warp order -- a fixed order, so the result is deterministic
__global__ void __launch_bounds__(256) chunk_sum_kernel(const float* __restrict__ part, float* __restrict__ out, int64_t n, int chunks) {
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int64_t i0 = (int64_t)blockIdx.x * 32; i0 < n; i0 += (int64_t)gridDim.x * 32) {
    const int64_t i = i0 + lane;
    float s = 0.f;
    if (i < n) for (int c = w; c < chunks; c += 8) s += part[(int64_t)c * n + i];
    red[w][lane] = s;
    __syncthreads();
    if (w == 0 && i < n) { float t = 0.f; for (int q = 0; q < 8; ++q) t += red[q][lane]; out[i] = t; }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Context-conditioned (specialist) layers, backward w.r.t. the input and the raw context-network output (conv1x1.py:31-50,
// actnorm.py:42-58).  The frozen generalist parameters get no gradient in --contextflow mode (requires_grad False in the reference).
// Conv1x1: W_b = tril(c,-1) + diag(exp(diag c)) [- I + NN];  z = W_b x;  ldj = HW (sum diag c [+ logabsdet NN]) + HW logp_c.
//   dx = W_b^T dz;  G = dz x^T;  dc[i][j] = G[i][j] (j < i),  exp(c_ii) G[i][i] + HW dldj[b] (j == i),  0 (j > i).
// One CTA per sample: x, dz (D x HW, odd row stride) and W_b in shared memory.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv1x1_ctx_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dz, const float* __restrict__ c,
                                                              const float* __restrict__ NN, int contextflow, const float* __restrict__ dldj,
                                                              float* __restrict__ dx, float* __restrict__ dc, int D, int HW) {
  extern __shared__ float sm[];
  const int S = HW | 1, SW = D | 1;
  float* xs = sm; float* gs = xs + D * S; float* Wb = gs + D * S;          // Wb[i * SW + j]
  const int64_t b = blockIdx.x;
  const float* cb = c + b * D * D;
  for (int i = threadIdx.x; i < D * HW; i += blockDim.x) {
    const int d = i / HW, p = i - d * HW;
    xs[d * S + p] = x[b * D * HW + i]; gs[d * S + p] = dz[b * D * HW + i];
  }
  for (int e = threadIdx.x; e < D * D; e += blockDim.x) {
    const int i = e / D, j = e - i * D;
    float v = j < i ? cb[e] : (j == i ? expf(cb[e]) : 0.f);
    if (contextflow) v = (v - (i == j ? 1.f : 0.f)) + NN[e];
    Wb[i * SW + j] = v;
  }
  __syncthreads();
  if (dx)
    for (int e = threadIdx.x; e < D * HW; e += blockDim.x) {
      const int j = e / HW, p = e - j * HW;
      float acc = 0.f;
      for (int i = 0; i < D; ++i) acc = fmaf(Wb[i * SW + j], gs[i * S + p], acc);
      dx[b * D * HW + e] = acc;
    }
  const float gl = dldj ? dldj[b] * (float)HW : 0.f;
  for (int e = threadIdx.x; e < D * D; e += blockDim.x) {
    const int i = e / D, j = e - i * D;
    float v = 0.f;
    if (j <= i) {
      float acc = 0.f;
      for (int p = 0; p < HW; ++p) acc = fmaf(gs[i * S + p], xs[j * S + p], acc);
      v = j < i ? acc : expf(cb[e]) * acc + gl;
    }
    dc[b * D * D + e] = v;
  }
}

// ActNorm with per-sample context terms: t_b = [NN_t +] c[b,:D], logs_b = [NN_logs +] c[b,D:];  z = (x - t_b) e^{-logs_b};
// ldj[b] = sum_d logs_b + HW logp_c.   dx = dz e^{-logs_b};  dc[b,d] = -sum_p dz e^{-logs_b};  dc[b,D+d] = -sum_p dz z + dldj[b].
// One CTA per sample, one warp per channel.
__global__ void __launch_bounds__(256) actnorm_ctx_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dz, const float* __restrict__ c,
                                                              const float* __restrict__ base_t, const float* __restrict__ base_logs,
                                                              const float* __restrict__ dldj, float* __restrict__ dx, float* __restrict__ dc,
                                                              int D, int HW) {
  const int64_t b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const float gl = dldj ? dldj[b] : 0.f;
  for (int d = warp; d < D; d += nw) {
    const float t = c[b * 2 * D + d] + (base_t ? base_t[d] : 0.f);
    const float e = expf(-(c[b * 2 * D + D + d] + (base_logs ? base_logs[d] : 0.f)));
    const int64_t o = (b * D + d) * HW;
    float a0 = 0.f, a1 = 0.f;
    for (int p = lane; p < HW; p += 32) {
      const float g = dz[o + p], ge = g * e;
      if (dx) dx[o + p] = ge;
      a0 -= ge;
      a1 -= g * ((x[o + p] - t) * e);
    }
    a0 = warp_sum(a0); a1 = warp_sum(a1);
    if (lane == 0) { dc[b * 2 * D + d] = a0; dc[b * 2 * D + D + d] = a1 + gl; }
  }
}

// elementwise ReLU mask: g *= (act > 0)
__global__ void relu_mask_kernel(float* __restrict__ g, const float* __restrict__ act, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (!(act[i] > 0.f)) g[i] = 0.f;
}

// Conv1x1's log-det term: dNN[i][j] += HW * (sum_b dldj[b]) * inv[j][i]     (d log|det A| / dA = A^-T), one CTA.
__global__ void logdet_grad_kernel(float* __restrict__ dNN, const float* __restrict__ inv, const float* __restrict__ dldj, int B, int D, float HW) {
  __shared__ float red[32];
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) s += dldj[b];
  s = group_sum(s, blockDim.x, red);
  for (int e = threadIdx.x; e < D * D; e += blockDim.x) { const int i = e / D, j = e - i * D; dNN[e] += HW * s * inv[j * D + i]; }
}

// out[b] = sum_m g[b,m]: the gradient a (B,) or (B,1) log-det term receives from the (B,M) accumulation (flowsequential.py:23).
__global__ void rowsum_kernel(const float* __restrict__ g, float* __restrict__ out, int B, int M) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int m = 0; m < M; ++m) s += g[(int64_t)b * M + m];
    out[b] = s;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Mixture base, training direction (context-free).  prep: sigma = softplus(sG), a = 1/sigma^2, cst[m,k] = log_softmax-weights
// - sum_e log sigma - n/2 log 2pi.  resp: comp[b,mk] = cst - 1/2 sum_e a (x-mu)^2; logp[b,m] = lse_k; r = softmax_k.
// dx[b,e] = -sum_mk w a (x - mu), w[b,mk] = g[b,m] r[b,mk].   Parameter sums S0 = sum_b w, S1 = sum_b w x, S2 = sum_b w x^2:
//   dmu = a (S1 - mu S0); dsigma = (S2 - 2 mu S1 + mu^2 S0) / sigma^3 - S0 / sigma; dsG = dsigma * sigmoid(sG);
//   dmix = S0; dwG[m,j] = dmix[m,j] - softmax(wG)[m,j] sum_k dmix[m,k]   (the eps clamp of Categorical(probs) is inactive).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gmm_prep_kernel(const float* __restrict__ sG, const float* __restrict__ wG, float* __restrict__ inv_var,
                                                       float* __restrict__ cst, int M, int K, int n) {
  __shared__ float red[32];
  const int mk = blockIdx.x, m = mk / K, k = mk - m * K;
  float acc = 0.f;
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const float s = softplus_f(sG[(int64_t)mk * n + e]);
    inv_var[(int64_t)mk * n + e] = 1.0f / (s * s);
    acc += logf(s);
  }
  acc = group_sum(acc, blockDim.x, red);
  if (threadIdx.x == 0) {
    float mx = -INFINITY;
    for (int j = 0; j < K; ++j) mx = fmaxf(mx, wG[m * K + j]);
    float se = 0.f;
    for (int j = 0; j < K; ++j) se += expf(wG[m * K + j] - mx);
    cst[mk] = (wG[mk] - mx - logf(se)) - acc - (float)n * kHalfLog2Pi;
  }
}

constexpr int kMaxMK = 256;

// one CTA per sample: warps loop over the (m,k) pairs, lanes over the elements of the sample held in shared memory
__global__ void __launch_bounds__(256) gmm_resp_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ mG,
                                                       const float* __restrict__ inv_var, const float* __restrict__ cst,
                                                       float* __restrict__ logp, float* __restrict__ resp, int M, int K, int n) {
  extern __shared__ float sx[];                        // n floats, then M*K comp values
  float* comp = sx + n;
  const int64_t b = blockIdx.x;
  for (int e = threadIdx.x; e < n; e += blockDim.x) sx[e] = x[b * x_bstride + e];
  __syncthreads();
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int mk = w; mk < M * K; mk += nw) {
    const float* mu = mG + (int64_t)mk * n; const float* a = inv_var + (int64_t)mk * n;
    float acc = 0.f;
    for (int e = l; e < n; e += 32) { const float d = sx[e] - __ldg(mu + e); acc = fmaf(d * d, __ldg(a + e), acc); }
    acc = warp_sum(acc);
    if (l == 0) comp[mk] = cst[mk] - 0.5f * acc;
  }
  __syncthreads();
  for (int m = threadIdx.x; m < M; m += blockDim.x) {
    float mx = -INFINITY;
    for (int k = 0; k < K; ++k) mx = fmaxf(mx, comp[m * K + k]);
    float se = 0.f;
    for (int k = 0; k < K; ++k) se += expf(comp[m * K + k] - mx);
    const float lp = mx + logf(se);
    logp[b * M + m] = lp;
    if (resp) for (int k = 0; k < K; ++k) resp[(b * M + m) * K + k] = expf(comp[m * K + k] - lp);
  }
}

// w[b,mk] = g[b,m] * resp[b,mk] (in place into wbuf);  dx[b,e] = -sum_mk w a (x - mu).   One CTA per sample.
__global__ void __launch_bounds__(256) gmm_dx_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ mG,
                                                     const float* __restrict__ inv_var, const float* __restrict__ resp, const float* __restrict__ g,
                                                     float* __restrict__ wbuf, float* __restrict__ dx, int64_t dx_bstride, int M, int K, int n) {
  __shared__ float sw[kMaxMK];
  const int64_t b = blockIdx.x;
  const int MK = M * K;
  for (int i = threadIdx.x; i < MK; i += blockDim.x) {
    const float v = g[b * M + i / K] * resp[b * MK + i];
    sw[i] = v; wbuf[b * MK + i] = v;
  }
  __syncthreads();
  if (!dx) return;
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const float xv = x[b * x_bstride + e];
    float acc = 0.f;
    for (int mk = 0; mk < MK; ++mk) acc = fmaf(sw[mk] * __ldg(inv_var + (int64_t)mk * n + e), __ldg(mG + (int64_t)mk * n + e) - xv, acc);
    dx[b * dx_bstride + e] = acc;
  }
}

// Partial sums over a chunk of samples: grid (n / 256, MK / MKT, chunks); thread = one element e, MKT pairs in registers.
constexpr int MKT = 8;
__global__ void __launch_bounds__(256) gmm_psum_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ wbuf,
                                                       float* __restrict__ part, int B, int MK, int n, int per_chunk) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int mk0 = blockIdx.y * MKT;
  const int chunk = blockIdx.z;
  const int b0 = chunk * per_chunk, b1 = min(B, b0 + per_chunk);
  float s1[MKT], s2[MKT];
#pragma unroll
  for (int j = 0; j < MKT; ++j) { s1[j] = 0.f; s2[j] = 0.f; }
  if (e < n) {
    for (int b = b0; b < b1; ++b) {
      const float xv = x[(int64_t)b * x_bstride + e], xx = xv * xv;
      const float* wp = wbuf + (int64_t)b * MK + mk0;
#pragma unroll
      for (int j = 0; j < MKT; ++j) {
        const float w = (mk0 + j < MK) ? __ldg(wp + j) : 0.f;
        s1[j] = fmaf(w, xv, s1[j]); s2[j] = fmaf(w, xx, s2[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < MKT; ++j)
      if (mk0 + j < MK) {
        float* o = part + (((int64_t)chunk * MK + mk0 + j) * n + e) * 2;
        o[0] = s1[j]; o[1] = s2[j];
      }
  }
}

// S0[mk] = sum_b w[b,mk] in fixed order (one CTA per mk), then dwG by the first thread of the last... kept separate for clarity.
__global__ void __launch_bounds__(256) gmm_s0_kernel(const float* __restrict__ wbuf, float* __restrict__ S0, int B, int MK) {
  __shared__ float red[32];
  const int mk = blockIdx.x;
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) s += wbuf[(int64_t)b * MK + mk];
  s = group_sum(s, blockDim.x, red);
  if (threadIdx.x == 0) S0[mk] = s;
}

__global__ void __launch_bounds__(256) gmm_finish_kernel(const float* __restrict__ part, const float* __restrict__ S0, const float* __restrict__ mG,
                                                         const float* __restrict__ sG, const float* __restrict__ wG,
                                                         float* __restrict__ dmG, float* __restrict__ dsG, float* __restrict__ dwG,
                                                         int M, int K, int n, int chunks) {
  const int MK = M * K;
  const int64_t total = (int64_t)MK * n;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int mk = (int)(i / n);
    float s1 = 0.f, s2 = 0.f;
    for (int c = 0; c < chunks; ++c) { const float* p = part + ((int64_t)c * total + i) * 2; s1 += p[0]; s2 += p[1]; }
    const float s0 = S0[mk], mu = mG[i], raw = sG[i];
    const float sg = softplus_f(raw);
    const float a = 1.0f / (sg * sg);
    dmG[i] = a * (s1 - mu * s0);
    const float q = s2 - 2.0f * mu * s1 + mu * mu * s0;              // sum_b w (x - mu)^2
    const float dsig = q * a / sg - s0 / sg;
    dsG[i] = dsig * (1.0f / (1.0f + expf(-raw)));
  }
  if (blockIdx.x == 0)
    for (int i = threadIdx.x; i < MK; i += blockDim.x) {
      const int m = i / K;
      float mx = -INFINITY, tot = 0.f;
      for (int k = 0; k < K; ++k) { mx = fmaxf(mx, wG[m * K + k]); tot += S0[m * K + k]; }
      float se = 0.f;
      for (int k = 0; k < K; ++k) se += expf(wG[m * K + k] - mx);
      dwG[i] = S0[i] - expf(wG[i] - mx) / se * tot;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Mixture with per-sample context offsets (gaussian.py:146-155: c = context_net(ctx), 'b (p m k d)': mean + c[0], softplus(sG + c[1])),
// training direction.  General in the context structure: c (B, 2*M*K*D) is the materialised lookup; the table gradients are a
// scatter of dc by context value (embed_scatter below).  One CTA per sample; sigma is recomputed where it is needed.
// ---------------------------------------------------------------------------------------------------------------
// Optional cheap transcendental forms for the per-sample-offset mixture (CFPP_GMM_FAST=1; ncu profiles/r2av_ncu_full_gmm_ctx.txt: both kernels
// are issue-bound at 92 % / 89 % issue-active with 125-240 instructions per element, almost all of them library expf / log1pf / logf / IEEE
// division).  softplus(raw) = log(1 + e^raw): e^raw by ex2.approx; for t = e^raw >= 0.5 the sum 1 + t >= 1.5 is far enough from 1 for
// lg2.approx's absolute error (2^-21.4) to stay below 1e-6 relative, smaller t keeps log1pf; reciprocals by rcp.approx.  Measured (cfg2,
// B = 8192, graphed training step): 105.8 -> 98.7 ms; the loss is unchanged to 1e-6 relative, but three of the reference gradient fixtures
// (context-network biases, cancelling sums over the batch) move from < 3e-4 to 5e-4 of the gradient's largest entry -- past the 2e-4 gate
// of tests/test_oracle_golden_training.py -- so the library forms stay the DEFAULT and the fast forms are an explicit choice.
// (A mode matrix over the single pieces -- exponential, logarithms, reciprocal, the forward's df^2 / s^2 by division -- showed that each
// of them except the reciprocal matters to those three fixtures.)  FAST is a template parameter: a run-time switch inside the 125-instruction
// element loop cost 15-20 % of either kernel.
template <bool FAST>
__device__ __forceinline__ float rcp_sel(float x) {
  if (!FAST) return 1.0f / x;
  float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
}
template <bool FAST>
__device__ __forceinline__ void softplus_sig(float raw, float& s, float& sig) {
  const bool big = raw > 20.f;                                 // F.softplus's threshold: s = raw, sigmoid = 1 to fp32
  const float a = big ? 0.f : raw;
  const float t = FAST ? __expf(a) : expf(a), u = 1.f + t;
  s = big ? raw : ((FAST && t >= 0.5f) ? __logf(u) : log1pf(t));
  sig = big ? 1.f : (FAST ? t * rcp_sel<true>(u) : t / u);
}
inline bool gmm_fast_mode() { const char* f = getenv("CFPP_GMM_FAST"); return f && f[0] == '1'; }

template <bool FAST>
__global__ void __launch_bounds__(256) gmm_ctx_fwd_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ mG,
                                                          const float* __restrict__ sG, const float* __restrict__ wG, const float* __restrict__ c,
                                                          float* __restrict__ logp, float* __restrict__ resp, int M, int K, int D, int HW) {
  extern __shared__ float sx[];                        // n floats, then M*K comp values
  const int n = D * HW, MK = M * K;
  float* comp = sx + n;
  const int64_t b = blockIdx.x;
  for (int e = threadIdx.x; e < n; e += blockDim.x) sx[e] = x[b * x_bstride + e];
  __syncthreads();
  const float* cm = c + b * 2 * MK * D; const float* cs = cm + (int64_t)MK * D;
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int hw_shift = (HW & (HW - 1)) == 0 ? __ffs(HW) - 1 : -1;     // HW a power of two (every image level): d = e >> shift, no division per element
  for (int mk = w; mk < MK; mk += nw) {
    float acc = 0.f;
    for (int e = l; e < n; e += 32) {
      const int d = hw_shift >= 0 ? e >> hw_shift : e / HW;
      const float mu = mG[(int64_t)mk * n + e] + cm[mk * D + d];
      float s, sig;
      softplus_sig<FAST>(sG[(int64_t)mk * n + e] + cs[mk * D + d], s, sig);
      const float df = sx[e] - mu;
      float quad;
      if (!FAST) quad = -0.5f * df * df / (s * s);
      else { const float q = df * rcp_sel<true>(s); quad = -0.5f * q * q; }
      acc += quad - (FAST ? __logf(s) : logf(s));
    }
    acc = warp_sum(acc);
    if (l == 0) {
      const int m = mk / K;
      float mx = -INFINITY;
      for (int j = 0; j < K; ++j) mx = fmaxf(mx, wG[m * K + j]);
      float se = 0.f;
      for (int j = 0; j < K; ++j) se += expf(wG[m * K + j] - mx);
      comp[mk] = acc + (wG[mk] - mx - logf(se)) - (float)n * kHalfLog2Pi;
    }
  }
  __syncthreads();
  for (int m = threadIdx.x; m < M; m += blockDim.x) {
    float mx = -INFINITY;
    for (int k = 0; k < K; ++k) mx = fmaxf(mx, comp[m * K + k]);
    float se = 0.f;
    for (int k = 0; k < K; ++k) se += expf(comp[m * K + k] - mx);
    const float lp = mx + logf(se);
    logp[b * M + m] = lp;
    for (int k = 0; k < K; ++k) resp[(b * M + m) * K + k] = expf(comp[m * K + k] - lp);
  }
}

// w[b,mk] = g[b,m] resp[b,mk];  dx[b,e] = sum_mk w (mu - x) / s^2;  dc_mean[b,mk,d] = sum_hw w (x - mu) / s^2;
// dc_scale[b,mk,d] = sum_hw w ((x - mu)^2 / s^3 - 1/s) sigmoid(sG + cs).   Warp per (mk, d): lanes over hw, shuffle-tree sums.
template <bool FAST>
__global__ void __launch_bounds__(256) gmm_ctx_bwd_kernel(const float* __restrict__ x, int64_t x_bstride, const float* __restrict__ mG,
                                                          const float* __restrict__ sG, const float* __restrict__ c, const float* __restrict__ resp,
                                                          const float* __restrict__ g, float* __restrict__ dx, int64_t dx_bstride,
                                                          float* __restrict__ dc, int M, int K, int D, int HW, int dx_partials) {
  extern __shared__ float sx[];                        // n floats x, M*K weights, then (dx_partials) one partial dx row of n floats per warp
  const int n = D * HW, MK = M * K;
  float* sw = sx + n;
  float* dxp = sw + MK;                                // [8][n]
  const int64_t b = blockIdx.x;
  for (int e = threadIdx.x; e < n; e += blockDim.x) sx[e] = x[b * x_bstride + e];
  for (int i = threadIdx.x; i < MK; i += blockDim.x) sw[i] = g[b * M + i / K] * resp[b * MK + i];
  const bool part = dx && dx_partials;
  if (part) for (int i = threadIdx.x; i < 8 * n; i += blockDim.x) dxp[i] = 0.f;
  __syncthreads();
  const float* cm = c + b * 2 * MK * D; const float* cs = cm + (int64_t)MK * D;
  float* dcm = dc + b * 2 * MK * D; float* dcs = dcm + (int64_t)MK * D;
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  // HW < 32 (a power of two: the 4x4 level): a warp takes 32 / HW pairs per pass, one segment of HW lanes each, and reduces inside the
  // segments -- instead of leaving half the lanes idle and paying one full-warp reduction per pair.
  const int SEG = (HW < 32 && (HW & (HW - 1)) == 0) ? HW : 32, PP = 32 / SEG;
  const int sub = l / SEG, hl = l - sub * SEG;
  for (int pair0 = w * PP; pair0 < MK * D; pair0 += nw * PP) {
    const int pair = pair0 + sub;
    const bool live = pair < MK * D;
    const int mk = live ? pair / D : 0, d = live ? pair - mk * D : 0;
    const float wt = sw[mk], om = live ? cm[pair] : 0.f, os = live ? cs[pair] : 0.f;
    float a0 = 0.f, a1 = 0.f;
    for (int hw = hl; live && hw < HW; hw += SEG) {
      const int e = d * HW + hw;
      const float raw = sG[(int64_t)mk * n + e] + os;
      // softplus and its derivative from ONE exponential: t = e^raw, s = log1p(t), sigmoid(raw) = t / (1 + t); 1 / s once, its powers by
      // multiplication
      float s, sig;
      softplus_sig<FAST>(raw, s, sig);
      const float df = sx[e] - (mG[(int64_t)mk * n + e] + om);
      const float rs = rcp_sel<FAST>(s), is2 = rs * rs;
      a0 += df * is2;
      a1 += (df * df * is2 - 1.0f) * rs * sig;
      if (part) dxp[w * n + e] -= wt * df * is2;       // this warp's share of dx[e] = sum_mk w (mu - x) / s^2 (one lane per e: no race)
    }
    if (SEG == 32) { a0 = warp_sum(a0); a1 = warp_sum(a1); }
    else for (int off = SEG >> 1; off > 0; off >>= 1) { a0 += __shfl_xor_sync(0xffffffffu, a0, off); a1 += __shfl_xor_sync(0xffffffffu, a1, off); }
    if (hl == 0 && live) { dcm[pair] = wt * a0; dcs[pair] = wt * a1; }
  }
  if (!dx) return;
  if (!part) {                                         // samples too large for eight partial rows: second pass, sigma recomputed per element
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const int d = e / HW;
      float acc = 0.f;
      for (int mk = 0; mk < MK; ++mk) {
        const float s = softplus_f(sG[(int64_t)mk * n + e] + cs[mk * D + d]);
        acc -= sw[mk] * (sx[e] - (mG[(int64_t)mk * n + e] + cm[mk * D + d])) / (s * s);
      }
      dx[b * dx_bstride + e] = acc;
    }
    return;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < n; e += blockDim.x) {  // the eight warp partials in warp order: deterministic
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) acc += dxp[q * n + e];
    dx[b * dx_bstride + e] = acc;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Encoder flows, training direction: the base draw and the variational-dequantisation epilogue as elementwise (B, C) kernels.
// ConditionalGaussianDistribution.sample (gaussian.py:263-270): c = [mean | log_scale] (B, 2C); x = mean + exp(ls) eps;
//   logq[b] = sum_d (-1/2 log 2pi - ls - 1/2 eps^2)   (the reference evaluates -1/2 exp(-2 ls) (x - mean)^2, which is eps^2).
//   backward: dc_mean = dx; dc_ls = dx eps exp(ls) - dlogq[b].
// VariationalCatDequantization.forward (dequantize.py:107-116) with Sigmoid (activations.py:231-235, temperature 1):
//   z = (x + sigmoid(u)) / qbins;  ldj[b] = ldj_const + sum_d (-softplus(-u) - softplus(u)) - qu[b].
//   backward: du = dz / qbins * s (1 - s) + dldj[b] (1 - 2 s);  dqu = -dldj.
// ---------------------------------------------------------------------------------------------------------------
__global__ void cond_gauss_fwd_kernel(const float* __restrict__ c, const float* __restrict__ eps, float* __restrict__ x, float* __restrict__ logq, int B, int C) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int d = 0; d < C; ++d) {
      const float ls = c[(int64_t)b * 2 * C + C + d], e = eps[(int64_t)b * C + d];
      x[(int64_t)b * C + d] = c[(int64_t)b * 2 * C + d] + expf(ls) * e;
      acc += -kHalfLog2Pi - ls - 0.5f * e * e;
    }
    logq[b] = acc;
  }
}
__global__ void cond_gauss_bwd_kernel(const float* __restrict__ c, const float* __restrict__ eps, const float* __restrict__ dx,
                                      const float* __restrict__ dlogq, float* __restrict__ dc, int B, int C) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (int64_t)B * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / C; const int d = (int)(i - b * C);
    const float g = dx ? dx[i] : 0.f;
    dc[b * 2 * C + d] = g;
    dc[b * 2 * C + C + d] = g * eps[i] * expf(c[b * 2 * C + C + d]) - (dlogq ? dlogq[b] : 0.f);
  }
}
// mode 0 vardeq: z = (xcat + s) / qbins, ldj = const + act - qu;  mode 1 argmax (dequantize.py:239-268): z = s * sign (sign = 2 bit - 1,
// passed in xcat as +-1), ldj = act - qu;  mode 2 probsample (:152-160): z = s, ldj = act + qu.   s = sigmoid(u), act = sum(-softplus(-u) - softplus(u)).
__global__ void vardeq_fwd_kernel(const float* __restrict__ u, const float* __restrict__ qu, const int64_t* __restrict__ xcat, const float* __restrict__ qbins,
                                  float ldj_const, int mode, float* __restrict__ z, float* __restrict__ ldj, int B, int C) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int d = 0; d < C; ++d) {
      const float v = u[(int64_t)b * C + d];
      const float s = 1.0f / (1.0f + expf(-v));
      z[(int64_t)b * C + d] = mode == 0 ? ((float)xcat[(int64_t)b * C + d] + s) / qbins[d] : mode == 1 ? s * (float)xcat[(int64_t)b * C + d] : s;
      acc += -softplus_f(-v) - softplus_f(v);
    }
    ldj[b] = mode == 2 ? (ldj_const + acc) + qu[b] : (ldj_const + acc) - qu[b];
  }
}
__global__ void vardeq_bwd_kernel(const float* __restrict__ u, const int64_t* __restrict__ xcat, const float* __restrict__ qbins, int mode,
                                  const float* __restrict__ dz, const float* __restrict__ dldj,
                                  float* __restrict__ du, float* __restrict__ dqu, int B, int C) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (int64_t)B * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / C; const int d = (int)(i - b * C);
    const float s = 1.0f / (1.0f + expf(-u[i]));
    const float gl = dldj ? dldj[b] : 0.f;
    const float mul = mode == 0 ? 1.0f / qbins[d] : mode == 1 ? (float)xcat[i] : 1.0f;
    du[i] = (dz ? dz[i] * mul * s * (1.0f - s) : 0.f) + gl * (1.0f - 2.0f * s);
    if (d == 0) dqu[b] = mode == 2 ? gl : -gl;
  }
}

// dTable[v][col] = sum over the samples whose context feature equals v (bucket order given by a stable sort), of dc[b][col0 + col]
__global__ void __launch_bounds__(256) embed_scatter_kernel(const float* __restrict__ dc, int64_t dc_stride, int col0, const int64_t* __restrict__ perm,
                                                            const int64_t* __restrict__ offsets, float* __restrict__ dtable, int width) {
  // CTA = one table row v x 32 columns; the 8 warps take the bucket's samples round-robin (8 rows in flight per column), their partial
  // sums are added in warp order: a fixed summation order, so the result is deterministic
  __shared__ float red[8][32];
  const int v = blockIdx.x;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int col = blockIdx.y * 32 + lane;
  const int64_t i1 = offsets[v + 1];
  float s = 0.f;
  if (col < width)
    for (int64_t i = offsets[v] + w; i < i1; i += 8) s += dc[perm[i] * dc_stride + col0 + col];
  red[w][lane] = s;
  __syncthreads();
  if (w == 0 && col < width) {
    float t = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) t += red[q][lane];
    dtable[(int64_t)v * width + col] = t;
  }
}

inline int grid1d(int64_t n, int per_thread = 1) {
  int64_t blocks = (n + 256LL * per_thread - 1) / (256LL * per_thread);
  const int64_t cap = (int64_t)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

inline bool conv_rows_enabled() {
  const char* e = getenv("CFPP_CONV_ROWS");                    // 0: keep the per-sample kernels for H = W = 1 (A/B switch; same results bit for bit)
  return !(e && e[0] == '0');
}

inline bool bwd_data3_enabled() {
  const char* e = getenv("CFPP_BWD_DATA3");                    // read per call: the tests flip it to compare the two routes bit for bit
  return !(e && e[0] == '0');
}

template <typename Kern>
inline bool want_smem(Kern k, size_t bytes) {
  if (bytes <= 48 * 1024) return true;
  if (bytes > 200 * 1024) return false;
  return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess;
}

}  // namespace bw
}  // namespace cfpp
using namespace cfpp;
using namespace cfpp::bw;

extern "C" int cfpp_coupling_bwd(const float* x, const float* h, const float* add, const float* dz, const float* dldj, float* dx, float* dh,
                                 int B, int C, int HW, void* stream) {
  CFPP_REQUIRE(C >= 2 && C % 2 == 0 && HW >= 1, "coupling_bwd: C=%d must be even, HW=%d", C, HW);
  if (B <= 0) return CFPP_OK;
  const int64_t n = (int64_t)(C / 2) * HW;
  int G = 32;
  while (G < 256 && G * 4 < n) G <<= 1;
  const int spc = 256 / G;
  coupling_bwd_kernel<<<(B + spc - 1) / spc, 256, 0, (cudaStream_t)stream>>>(x, h, add, dz, dldj, dx, dh, B, C, HW, G);
  return check_launch("coupling_bwd");
}

extern "C" int64_t cfpp_actnorm_bwd_workspace_floats(int B, int D) {
  int chunks = (num_sms() * 4 + D - 1) / D; if (chunks < 1) chunks = 1; if (chunks > B) chunks = B > 0 ? B : 1;
  return (int64_t)chunks * D * 2;
}

extern "C" int cfpp_actnorm_bwd(const float* x, const float* dz, const float* dldj, const float* t, const float* logs,
                                float* dx, float* dt, float* dlogs, float* workspace, int B, int D, int HW, void* stream) {
  CFPP_REQUIRE(D >= 1 && HW >= 1 && B >= 1, "actnorm_bwd: B=%d D=%d HW=%d", B, D, HW);
  int chunks = (num_sms() * 4 + D - 1) / D; if (chunks < 1) chunks = 1; if (chunks > B) chunks = B;
  const int per_chunk = (B + chunks - 1) / chunks;
  chunks = (B + per_chunk - 1) / per_chunk;
  actnorm_bwd_kernel<<<dim3(D, chunks), 256, 0, (cudaStream_t)stream>>>(x, dz, t, logs, dx, workspace, B, D, HW, per_chunk);
  int rc = check_launch("actnorm_bwd");
  if (rc != CFPP_OK) return rc;
  actnorm_bwd_finish_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(workspace, dldj, dt, dlogs, B, D, chunks);
  return check_launch("actnorm_bwd_finish");
}

#define CFPP_CONV_DISPATCH(KH, KW, ...)                                                   \
  do {                                                                                    \
    if (KH == 1 && KW == 1) { constexpr int kKH = 1, kKW = 1; __VA_ARGS__; }              \
    else if (KH == 3 && KW == 3) { constexpr int kKH = 3, kKW = 3; __VA_ARGS__; }         \
    else if (KH == 3 && KW == 1) { constexpr int kKH = 3, kKW = 1; __VA_ARGS__; }         \
    else { constexpr int kKH = 1, kKW = 3; __VA_ARGS__; }                                 \
  } while (0)

static inline bool conv_shape_ok(int H, int Wd, int KH, int KW) {
  return (KH == 1 || KH == 3) && (KW == 1 || KW == 3) && (KH == 1 || H >= 2) && (KW == 1 || Wd >= 2);
}

extern "C" int cfpp_conv2d_fwd(const float* in, int64_t in_bstride, const float* W, const float* bias, float* out,
                               int B, int Cin, int Cout, int H, int Wd, int KH, int KW, int relu, void* stream) {
  CFPP_REQUIRE(conv_shape_ok(H, Wd, KH, KW), "conv2d: kernel %dx%d on %dx%d", KH, KW, H, Wd);
  if (B <= 0) return CFPP_OK;
  if (H * Wd == 1 && KH == 1 && KW == 1 && conv_rows_enabled()) {
    const size_t smr = ((size_t)Cin * (Cout | 1) + (size_t)kRowsPerCta * (Cin | 1)) * sizeof(float);
    if (want_smem(conv_rows_kernel<true>, smr)) {
      conv_rows_kernel<true><<<(B + kRowsPerCta - 1) / kRowsPerCta, 256, smr, (cudaStream_t)stream>>>(in, in_bstride, W, bias, nullptr, 0, out, Cout, 0, B, Cin, Cout, relu);
      return check_launch("conv2d_fwd");
    }
  }
  const size_t smem = (size_t)Cin * odd_stride((H + 2 * (KH / 2)) * (Wd + 2 * (KW / 2))) * sizeof(float);
  CFPP_CONV_DISPATCH(KH, KW, {
    CFPP_REQUIRE(want_smem(conv2d_fwd_kernel<kKH, kKW>, smem), "conv2d_fwd: sample of %zu bytes exceeds shared memory", smem);
    conv2d_fwd_kernel<kKH, kKW><<<B, 256, smem, (cudaStream_t)stream>>>(in, in_bstride, W, bias, out, Cin, Cout, H, Wd, relu);
  });
  return check_launch("conv2d_fwd");
}

extern "C" int cfpp_conv2d_bwd_data(const float* dout, const float* W, const float* act, int64_t act_bstride, float* din, int64_t din_bstride,
                                    int accumulate, int B, int Cin, int Cout, int H, int Wd, int KH, int KW, void* stream) {
  CFPP_REQUIRE(conv_shape_ok(H, Wd, KH, KW), "conv2d: kernel %dx%d on %dx%d", KH, KW, H, Wd);
  if (B <= 0) return CFPP_OK;
  if (H * Wd == 1 && KH == 1 && KW == 1 && conv_rows_enabled()) {
    const size_t smr = ((size_t)Cout * (Cin | 1) + (size_t)kRowsPerCta * (Cout | 1)) * sizeof(float);
    if (want_smem(conv_rows_kernel<false>, smr)) {
      conv_rows_kernel<false><<<(B + kRowsPerCta - 1) / kRowsPerCta, 256, smr, (cudaStream_t)stream>>>(dout, Cout, W, nullptr, act, act_bstride, din, din_bstride, accumulate, B, Cout, Cin, 0);
      return check_launch("conv2d_bwd_data");
    }
  }
  if (KH == 3 && KW == 3 && Cin % 4 == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0 && bwd_data3_enabled()) {
    // register-tiled 3x3 route; CFPP_BWD_DATA3=0 keeps the generic tile (same results bit for bit: an A/B switch for timing)
    const int TP = Wd + 2 <= 6 ? 6 : 4;
    const int NG = (Wd + 2 + TP - 1) / TP, WzP = TP == 4 ? 4 * NG : 8;
    const size_t smem3 = ((size_t)Cout * (H + 4) * WzP + 4 + (size_t)Cin * odd_stride((H + 2) * (Wd + 2))) * sizeof(float);
    bool ok = false;
#define CFPP_BD3(TP_) do { auto kern = conv2d_bwd_data3_kernel<TP_>; \
      if ((ok = want_smem(kern, smem3))) { \
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);   /* two samples resident per SM */ \
        kern<<<B, 256, smem3, (cudaStream_t)stream>>>(dout, W, act, act_bstride, din, din_bstride, accumulate, Cin, Cout, H, Wd, NG, WzP); } } while (0)
    if (TP == 6) CFPP_BD3(6); else CFPP_BD3(4);
#undef CFPP_BD3
    if (ok) return check_launch("conv2d_bwd_data");
  }
  const size_t smem = ((size_t)Cout * odd_stride((H + 2 * (KH - 1)) * (Wd + 2 * (KW - 1))) +
                       (KH * KW == 1 ? 0 : (size_t)Cin * odd_stride((H + 2 * (KH / 2)) * (Wd + 2 * (KW / 2))))) * sizeof(float);
  CFPP_CONV_DISPATCH(KH, KW, {
    CFPP_REQUIRE(want_smem(conv2d_bwd_data_kernel<kKH, kKW>, smem), "conv2d_bwd_data: sample of %zu bytes exceeds shared memory", smem);
    conv2d_bwd_data_kernel<kKH, kKW><<<B, 256, smem, (cudaStream_t)stream>>>(dout, W, act, act_bstride, din, din_bstride, accumulate, Cin, Cout, H, Wd);
  });
  return check_launch("conv2d_bwd_data");
}

static inline void bwd_weight_plan(int B, int Cin, int Cout, int& NCO, int& coblocks, int& chunks, int& per_chunk) {
  NCO = (256 / (Cin > 0 ? Cin : 1)) * PPT; if (NCO > Cout) NCO = Cout; if (NCO < 1) NCO = 1;
  coblocks = (Cout + NCO - 1) / NCO;
  chunks = (num_sms() * 4 + coblocks - 1) / coblocks; if (chunks > B) chunks = B; if (chunks < 1) chunks = 1;
  per_chunk = (B + chunks - 1) / chunks; if (per_chunk < 1) per_chunk = 1;
  chunks = B > 0 ? (B + per_chunk - 1) / per_chunk : 1;
}

extern "C" int64_t cfpp_conv2d_bwd_weight_workspace_floats(int B, int Cin, int Cout, int KH, int KW) {
  int NCO, coblocks, chunks, per_chunk;
  bwd_weight_plan(B, Cin, Cout, NCO, coblocks, chunks, per_chunk);
  return (int64_t)chunks * ((int64_t)Cout * Cin * KH * KW + Cout);
}

extern "C" int cfpp_conv2d_bwd_weight(const float* in, int64_t in_bstride, const float* dout, float* dW, float* db, float* workspace,
                                      int B, int Cin, int Cout, int H, int Wd, int KH, int KW, void* stream) {
  CFPP_REQUIRE(conv_shape_ok(H, Wd, KH, KW), "conv2d: kernel %dx%d on %dx%d", KH, KW, H, Wd);
  CFPP_REQUIRE(Cin >= 1 && Cin <= 256, "conv2d_bwd_weight: Cin=%d outside [1,256]", Cin);
  const int KK = KH * KW, HW = H * Wd;
  const int64_t nW = (int64_t)Cout * Cin * KK;
  if (B <= 0) {
    cudaMemsetAsync(dW, 0, (size_t)nW * sizeof(float), (cudaStream_t)stream);
    if (db) cudaMemsetAsync(db, 0, (size_t)Cout * sizeof(float), (cudaStream_t)stream);
    return CFPP_OK;
  }
  CFPP_REQUIRE(workspace != nullptr, "conv2d_bwd_weight: workspace required (cfpp_conv2d_bwd_weight_workspace_floats)");
  int NCO, coblocks, chunks, per_chunk;
  bwd_weight_plan(B, Cin, Cout, NCO, coblocks, chunks, per_chunk);
  if (HW == 1 && KK == 1 && nW <= 256 * kRowsWEntries && Cout <= 256 && conv_rows_enabled()) {
    int chunks_r = (B + kRowsW - 1) / kRowsW; if (chunks_r > chunks) chunks_r = chunks;          // never more partial slices than the workspace holds
    const int per_r = (B + chunks_r - 1) / chunks_r;
    chunks_r = (B + per_r - 1) / per_r;
    float* pW = workspace; float* pb = workspace + (int64_t)chunks_r * nW;
    const size_t smw = (size_t)kRowsW * ((Cin | 1) + (Cout | 1)) * sizeof(float);
    if (want_smem(conv_rows_bwd_weight_kernel, smw)) {
      conv_rows_bwd_weight_kernel<<<chunks_r, 256, smw, (cudaStream_t)stream>>>(in, in_bstride, dout, pW, db ? pb : nullptr, B, Cin, Cout, per_r);
      int rc = check_launch("conv2d_bwd_weight");
      if (rc != CFPP_OK) return rc;
      chunk_sum_kernel<<<(unsigned)((nW + 31) / 32), 256, 0, (cudaStream_t)stream>>>(pW, dW, nW, chunks_r);
      if ((rc = check_launch("conv2d_bwd_weight_sum")) != CFPP_OK) return rc;
      if (db) {
        chunk_sum_kernel<<<(Cout + 31) / 32, 256, 0, (cudaStream_t)stream>>>(pb, db, Cout, chunks_r);
        rc = check_launch("conv2d_bwd_bias_sum");
      }
      return rc;
    }
  }
  float* partW = workspace; float* partb = workspace + (int64_t)chunks * nW;
  const size_t smem = ((size_t)Cin * odd_stride((H + 2 * (KH / 2)) * (Wd + 2 * (KW / 2))) + (size_t)NCO * odd_stride(HW)) * sizeof(float);
  const dim3 grid(chunks, coblocks);
  CFPP_CONV_DISPATCH(KH, KW, {
    CFPP_REQUIRE(want_smem(conv2d_bwd_weight_kernel<kKH, kKW>, smem), "conv2d_bwd_weight: tile of %zu bytes exceeds shared memory", smem);
    conv2d_bwd_weight_kernel<kKH, kKW><<<grid, 256, smem, (cudaStream_t)stream>>>(in, in_bstride, dout, partW, db ? partb : nullptr, B, Cin, Cout, H, Wd, NCO, per_chunk);
  });
  int rc = check_launch("conv2d_bwd_weight");
  if (rc != CFPP_OK) return rc;
  chunk_sum_kernel<<<(unsigned)((nW + 31) / 32), 256, 0, (cudaStream_t)stream>>>(partW, dW, nW, chunks);
  if ((rc = check_launch("conv2d_bwd_weight_sum")) != CFPP_OK) return rc;
  if (db) {
    chunk_sum_kernel<<<(Cout + 31) / 32, 256, 0, (cudaStream_t)stream>>>(partb, db, Cout, chunks);
    rc = check_launch("conv2d_bwd_bias_sum");
  }
  return rc;
}

extern "C" int cfpp_conv1x1_ctx_bwd(const float* x, const float* dz, const float* c, const float* NN, int contextflow, const float* dldj,
                                    float* dx, float* dc, int B, int D, int HW, void* stream) {
  CFPP_REQUIRE(D >= 1 && HW >= 1 && c && dc && (!contextflow || NN), "conv1x1_ctx_bwd: D=%d HW=%d", D, HW);
  if (B <= 0) return CFPP_OK;
  const size_t smem = ((size_t)2 * D * (HW | 1) + (size_t)D * (D | 1)) * sizeof(float);
  CFPP_REQUIRE(want_smem(conv1x1_ctx_bwd_kernel, smem), "conv1x1_ctx_bwd: sample of %zu bytes exceeds shared memory", smem);
  conv1x1_ctx_bwd_kernel<<<B, 256, smem, (cudaStream_t)stream>>>(x, dz, c, NN, contextflow, dldj, dx, dc, D, HW);
  return check_launch("conv1x1_ctx_bwd");
}

extern "C" int cfpp_actnorm_ctx_bwd(const float* x, const float* dz, const float* c, const float* base_t, const float* base_logs,
                                    const float* dldj, float* dx, float* dc, int B, int D, int HW, void* stream) {
  CFPP_REQUIRE(D >= 1 && HW >= 1 && c && dc, "actnorm_ctx_bwd: D=%d HW=%d", D, HW);
  if (B <= 0) return CFPP_OK;
  actnorm_ctx_bwd_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(x, dz, c, base_t, base_logs, dldj, dx, dc, D, HW);
  return check_launch("actnorm_ctx_bwd");
}

extern "C" int cfpp_gmm_ctx_train_fwd(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG, const float* c,
                                      float* logp, float* resp, int B, int M, int K, int D, int HW, void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && M * K <= kMaxMK && D >= 1 && HW >= 1 && c, "gmm_ctx_train: M*K=%d exceeds %d", M * K, kMaxMK);
  if (B <= 0) return CFPP_OK;
  const size_t smem = ((size_t)D * HW + M * K) * sizeof(float);
  CFPP_REQUIRE(gmm_fast_mode() ? want_smem(gmm_ctx_fwd_kernel<true>, smem) : want_smem(gmm_ctx_fwd_kernel<false>, smem), "gmm_ctx_train_fwd: sample of %zu bytes exceeds shared memory", smem);
  if (gmm_fast_mode()) gmm_ctx_fwd_kernel<true><<<B, 256, smem, (cudaStream_t)stream>>>(x, x_bstride, mG, sG, wG, c, logp, resp, M, K, D, HW);
  else gmm_ctx_fwd_kernel<false><<<B, 256, smem, (cudaStream_t)stream>>>(x, x_bstride, mG, sG, wG, c, logp, resp, M, K, D, HW);
  return check_launch("gmm_ctx_train_fwd");
}

extern "C" int cfpp_gmm_ctx_train_bwd(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* c, const float* resp,
                                      const float* g, float* dx, int64_t dx_bstride, float* dc, int B, int M, int K, int D, int HW, void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && M * K <= kMaxMK && D >= 1 && HW >= 1 && c && dc, "gmm_ctx_train_bwd: M*K=%d", M * K);
  if (B <= 0) return CFPP_OK;
  size_t smem = ((size_t)D * HW * (dx ? 9 : 1) + M * K) * sizeof(float);
  int partials = dx ? 1 : 0;
  const bool fast = gmm_fast_mode();
  auto fits = [&](size_t bytes) { return fast ? want_smem(gmm_ctx_bwd_kernel<true>, bytes) : want_smem(gmm_ctx_bwd_kernel<false>, bytes); };
  if (dx && !fits(smem)) {                              // eight partial dx rows do not fit: keep the sample only and recompute sigma for dx
    partials = 0;
    smem = ((size_t)D * HW + M * K) * sizeof(float);
  }
  CFPP_REQUIRE(fits(smem), "gmm_ctx_train_bwd: sample of %zu bytes exceeds shared memory", smem);
  if (fast) gmm_ctx_bwd_kernel<true><<<B, 256, smem, (cudaStream_t)stream>>>(x, x_bstride, mG, sG, c, resp, g, dx, dx_bstride, dc, M, K, D, HW, partials);
  else gmm_ctx_bwd_kernel<false><<<B, 256, smem, (cudaStream_t)stream>>>(x, x_bstride, mG, sG, c, resp, g, dx, dx_bstride, dc, M, K, D, HW, partials);
  return check_launch("gmm_ctx_train_bwd");
}

extern "C" int cfpp_cond_gauss_fwd(const float* c, const float* eps, float* x, float* logq, int B, int C, void* stream) {
  CFPP_REQUIRE(C >= 1, "cond_gauss: C=%d", C);
  if (B <= 0) return CFPP_OK;
  cond_gauss_fwd_kernel<<<grid1d(B), 256, 0, (cudaStream_t)stream>>>(c, eps, x, logq, B, C);
  return check_launch("cond_gauss_fwd");
}
extern "C" int cfpp_cond_gauss_bwd(const float* c, const float* eps, const float* dx, const float* dlogq, float* dc, int B, int C, void* stream) {
  CFPP_REQUIRE(C >= 1, "cond_gauss: C=%d", C);
  if (B <= 0) return CFPP_OK;
  cond_gauss_bwd_kernel<<<grid1d((int64_t)B * C), 256, 0, (cudaStream_t)stream>>>(c, eps, dx, dlogq, dc, B, C);
  return check_launch("cond_gauss_bwd");
}
extern "C" int cfpp_vardeq_fwd(const float* u, const float* qu, const int64_t* xcat, const float* qbins, float ldj_const, int mode, float* z, float* ldj,
                               int B, int C, void* stream) {
  CFPP_REQUIRE(C >= 1 && mode >= 0 && mode <= 2 && (mode == 2 || xcat) && (mode != 0 || qbins), "vardeq: C=%d mode=%d", C, mode);
  if (B <= 0) return CFPP_OK;
  vardeq_fwd_kernel<<<grid1d(B), 256, 0, (cudaStream_t)stream>>>(u, qu, xcat, qbins, ldj_const, mode, z, ldj, B, C);
  return check_launch("vardeq_fwd");
}
extern "C" int cfpp_vardeq_bwd(const float* u, const int64_t* xcat, const float* qbins, int mode, const float* dz, const float* dldj, float* du, float* dqu,
                               int B, int C, void* stream) {
  CFPP_REQUIRE(C >= 1 && mode >= 0 && mode <= 2 && (mode == 2 || xcat) && (mode != 0 || qbins), "vardeq: C=%d mode=%d", C, mode);
  if (B <= 0) return CFPP_OK;
  vardeq_bwd_kernel<<<grid1d((int64_t)B * C), 256, 0, (cudaStream_t)stream>>>(u, xcat, qbins, mode, dz, dldj, du, dqu, B, C);
  return check_launch("vardeq_bwd");
}

extern "C" int cfpp_embed_scatter(const float* dc, int64_t dc_stride, int col0, const int64_t* perm, const int64_t* offsets, float* dtable,
                                  int cardinality, int width, void* stream) {
  CFPP_REQUIRE(cardinality >= 1 && width >= 1 && perm && offsets, "embed_scatter: card=%d width=%d", cardinality, width);
  embed_scatter_kernel<<<dim3(cardinality, (width + 31) / 32), 256, 0, (cudaStream_t)stream>>>(dc, dc_stride, col0, perm, offsets, dtable, width);
  return check_launch("embed_scatter");
}

extern "C" int cfpp_relu_mask(float* g, const float* act, int64_t n, void* stream) {
  if (n <= 0) return CFPP_OK;
  relu_mask_kernel<<<grid1d(n, 4), 256, 0, (cudaStream_t)stream>>>(g, act, n);
  return check_launch("relu_mask");
}

extern "C" int cfpp_logdet_grad(float* dNN, const float* inv, const float* dldj, int B, int D, int HW, void* stream) {
  CFPP_REQUIRE(D >= 1 && D <= 128 && dldj, "logdet_grad: D=%d", D);
  logdet_grad_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(dNN, inv, dldj, B, D, (float)HW);
  return check_launch("logdet_grad");
}

extern "C" int cfpp_rowsum(const float* g, float* out, int B, int M, void* stream) {
  if (B <= 0) return CFPP_OK;
  rowsum_kernel<<<grid1d(B), 256, 0, (cudaStream_t)stream>>>(g, out, B, M);
  return check_launch("rowsum");
}

extern "C" int cfpp_gmm_train_prep(const float* sG, const float* wG, float* inv_var, float* cst, int M, int K, int n, void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && M * K <= kMaxMK && n >= 1, "gmm_train: M*K=%d exceeds %d", M * K, kMaxMK);
  gmm_prep_kernel<<<M * K, 256, 0, (cudaStream_t)stream>>>(sG, wG, inv_var, cst, M, K, n);
  return check_launch("gmm_train_prep");
}

extern "C" int cfpp_gmm_train_fwd(const float* x, int64_t x_bstride, const float* mG, const float* inv_var, const float* cst,
                                  float* logp, float* resp, int B, int M, int K, int n, void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && M * K <= kMaxMK && n >= 1, "gmm_train: M*K=%d exceeds %d", M * K, kMaxMK);
  if (B <= 0) return CFPP_OK;
  const size_t smem = ((size_t)n + M * K) * sizeof(float);
  CFPP_REQUIRE(want_smem(gmm_resp_kernel, smem), "gmm_train_fwd: sample of %zu bytes exceeds shared memory", smem);
  gmm_resp_kernel<<<B, 256, smem, (cudaStream_t)stream>>>(x, x_bstride, mG, inv_var, cst, logp, resp, M, K, n);
  return check_launch("gmm_train_fwd");
}

extern "C" int64_t cfpp_gmm_train_bwd_workspace_floats(int B, int M, int K, int n) {
  int chunks = 8; if (chunks > B) chunks = B > 0 ? B : 1;
  return (int64_t)B * M * K + (int64_t)M * K + (int64_t)chunks * M * K * n * 2;
}

extern "C" int cfpp_gmm_train_bwd(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG, const float* inv_var,
                                  const float* resp, const float* g, float* dx, int64_t dx_bstride, float* dmG, float* dsG, float* dwG,
                                  float* workspace, int B, int M, int K, int n, void* stream) {
  CFPP_REQUIRE(M >= 1 && K >= 1 && M * K <= kMaxMK && n >= 1 && B >= 1, "gmm_train_bwd: B=%d M*K=%d", B, M * K);
  const int MK = M * K;
  int chunks = 8; if (chunks > B) chunks = B;
  const int per_chunk = (B + chunks - 1) / chunks;
  chunks = (B + per_chunk - 1) / per_chunk;
  float* wbuf = workspace; float* S0 = wbuf + (int64_t)B * MK; float* part = S0 + MK;
  cudaStream_t st = (cudaStream_t)stream;
  gmm_dx_kernel<<<B, 256, 0, st>>>(x, x_bstride, mG, inv_var, resp, g, wbuf, dx, dx_bstride, M, K, n);
  int rc = check_launch("gmm_train_dx");
  if (rc != CFPP_OK || !dmG) return rc;
  gmm_psum_kernel<<<dim3((n + 255) / 256, (MK + MKT - 1) / MKT, chunks), 256, 0, st>>>(x, x_bstride, wbuf, part, B, MK, n, per_chunk);
  if ((rc = check_launch("gmm_train_psum")) != CFPP_OK) return rc;
  gmm_s0_kernel<<<MK, 256, 0, st>>>(wbuf, S0, B, MK);
  if ((rc = check_launch("gmm_train_s0")) != CFPP_OK) return rc;
  gmm_finish_kernel<<<grid1d((int64_t)MK * n), 256, 0, st>>>(part, S0, mG, sG, wG, dmG, dsG, dwG, M, K, n, chunks);
  return check_launch("gmm_train_finish");
}
