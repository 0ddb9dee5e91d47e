// GDN / IGDN forward and backward, fp32 CUDA-core path (correctness baseline + any-C fallback).
//
// Replaces the TF graph of tensorflow_compression/python/layers/gdn.py:371-421
//   u = relu(x) | x ; p = |u|^alpha ; n = beta + p . gamma ; m = n^eps ; y = u / m  |  u * m
// and TF autodiff of it (the reference has no hand-written gradient).
//
// Layout: x, y [n_pix, C] row-major (channels-last, the only layout the models use), gamma [C, C]
// with gamma[j, i] = weight of input channel j in the pool of output channel i.
//
// Kernel shape (persistent, one CTA per SM): gamma lives in shared memory for the whole launch; a
// CTA walks 64-pixel tiles; warp w owns 8 pixels, lane l owns output channels {l + 32 m}; the pool
// tile is read with 128-bit broadcast loads (4 input channels at a time), gamma rows with
// conflict-free scalar loads.  The tcgen05 tensor-core path lives in gdn_tc.cu.
#include <algorithm>

#include "common.cuh"

namespace tfcb {
namespace {

constexpr int kTM = 64;        // pixels per tile
constexpr int kThreads = 256;  // 8 warps x 8 pixels
constexpr int kPixPerWarp = 8;

struct GdnFlags {
  bool inverse, rectify;
  int alpha_mode;  // 1, 2, or 0 = generic powf
  int eps_mode;    // 1 -> identity, 2 -> sqrt, 0 = generic powf
  float alpha, eps;
};

__device__ __forceinline__ float pool_of(float x, const GdnFlags& f) {
  const float u = f.rectify ? fmaxf(x, 0.f) : x;
  if (f.alpha_mode == 1) return f.rectify ? u : fabsf(u);
  if (f.alpha_mode == 2) return u * u;
  return powf(u, f.alpha);  // `inputs ** alpha`, gdn.py:388
}

__device__ __forceinline__ float norm_of(float n, const GdnFlags& f) {
  if (f.eps_mode == 1) return n;
  if (f.eps_mode == 2) return sqrtf(n);
  return powf(n, f.eps);
}

// d pool / d u
__device__ __forceinline__ float dpool_du(float u, const GdnFlags& f) {
  if (f.alpha_mode == 1) {
    if (f.rectify) return 1.f;
    return (u > 0.f) ? 1.f : ((u < 0.f) ? -1.f : 0.f);  // TF's abs gradient is sign()
  }
  if (f.alpha_mode == 2) return 2.f * u;
  return f.alpha * powf(u, f.alpha - 1.f);
}

// d L / d n  given upstream g, for one element
__device__ __forceinline__ float dl_dn(float g, float u, float n, const GdnFlags& f) {
  if (!f.inverse) {
    // y = u * n^-eps
    if (f.eps_mode == 1) return -g * u / (n * n);
    if (f.eps_mode == 2) return -0.5f * g * u / (n * sqrtf(n));
    return -f.eps * g * u * powf(n, -f.eps - 1.f);
  }
  if (f.eps_mode == 1) return g * u;
  if (f.eps_mode == 2) return 0.5f * g * u / sqrtf(n);
  return f.eps * g * u * powf(n, f.eps - 1.f);
}

// ---------------------------------------------------------------------------------------------
// Tiled contraction  acc[pix][m] = sum_j  A[pix][j] * W[j][lane + 32 m]
// A: smem tile [kTM][C + 4] (row padded so that the 8 rows of a warp hit different banks for the
// 128-bit broadcast loads), W: smem [C][C].
// ---------------------------------------------------------------------------------------------
template <int CPL>
__device__ __forceinline__ void contract(const float* __restrict__ A, const float* __restrict__ W, int C,
                                         int lda, int warp, int lane, float (&acc)[kPixPerWarp][CPL]) {
#pragma unroll
  for (int p = 0; p < kPixPerWarp; ++p)
#pragma unroll
    for (int m = 0; m < CPL; ++m) acc[p][m] = 0.f;
  const float* a0 = A + (warp * kPixPerWarp) * lda;
  for (int j = 0; j < C; j += 4) {
    float4 a[kPixPerWarp];
#pragma unroll
    for (int p = 0; p < kPixPerWarp; ++p) a[p] = *reinterpret_cast<const float4*>(a0 + p * lda + j);
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      float w[CPL];
#pragma unroll
      for (int m = 0; m < CPL; ++m) w[m] = W[(j + jj) * C + lane + 32 * m];
#pragma unroll
      for (int p = 0; p < kPixPerWarp; ++p) {
        const float av = jj == 0 ? a[p].x : (jj == 1 ? a[p].y : (jj == 2 ? a[p].z : a[p].w));
#pragma unroll
        for (int m = 0; m < CPL; ++m) acc[p][m] = fmaf(av, w[m], acc[p][m]);
      }
    }
  }
}

template <int CPL>
__global__ void __launch_bounds__(kThreads, 1)
gdn_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
               float* __restrict__ y, long long n_pix, GdnFlags f) {
  constexpr int C = CPL * 32;
  constexpr int LDA = C + 4;
  extern __shared__ __align__(16) float smem[];
  float* W = smem;          // [C][C]
  float* A = smem + C * C;  // [kTM][LDA]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < C * C; i += kThreads) W[i] = gamma[i];
  float b[CPL];
#pragma unroll
  for (int m = 0; m < CPL; ++m) b[m] = beta[lane + 32 * m];

  const long long n_tiles = (n_pix + kTM - 1) / kTM;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const long long p0 = t * kTM;
    __syncthreads();  // previous tile fully consumed (also covers the W fill)
    for (int i = tid; i < kTM * (C / 4); i += kThreads) {
      const int r = i / (C / 4), c4 = i % (C / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p0 + r < n_pix) v = __ldg(reinterpret_cast<const float4*>(x + (p0 + r) * C) + c4);
      v.x = pool_of(v.x, f);
      v.y = pool_of(v.y, f);
      v.z = pool_of(v.z, f);
      v.w = pool_of(v.w, f);
      *reinterpret_cast<float4*>(A + r * LDA + 4 * c4) = v;
    }
    __syncthreads();
    float acc[kPixPerWarp][CPL];
    contract<CPL>(A, W, C, LDA, warp, lane, acc);
#pragma unroll
    for (int p = 0; p < kPixPerWarp; ++p) {
      const long long pix = p0 + warp * kPixPerWarp + p;
      if (pix < n_pix) {
#pragma unroll
        for (int m = 0; m < CPL; ++m) {
          const int ch = lane + 32 * m;
          const float xv = __ldg(x + pix * C + ch);
          const float u = f.rectify ? fmaxf(xv, 0.f) : xv;
          const float nm = norm_of(b[m] + acc[p][m], f);
          y[pix * C + ch] = f.inverse ? u * nm : u / nm;
        }
      }
    }
  }
}

// Any-C fallback: one warp per pixel, lanes stride over output channels.
__global__ void gdn_fwd_generic_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, float* __restrict__ y,
                                       long long n_pix, int C, GdnFlags f) {
  const long long pix = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pix >= n_pix) return;
  const float* xr = x + pix * C;
  for (int i = lane; i < C; i += 32) {
    float n = 0.f;
    for (int j = 0; j < C; ++j) n = fmaf(pool_of(xr[j], f), gamma[(long long)j * C + i], n);
    n = beta[i] + n;
    const float u = f.rectify ? fmaxf(xr[i], 0.f) : xr[i];
    const float nm = norm_of(n, f);
    y[pix * C + i] = f.inverse ? u * nm : u / nm;
  }
}

// ---------------------------------------------------------------------------------------------
// Backward
//   B1: n = beta + p.gamma ; q = dL/dn ; dx_direct = g / m (or g * m) ; writes q (workspace), dx.
//   B2: dp = q . gamma^T ; dx += dpool/du * dp ; rectify mask.
//   B3: per-CTA partial dgamma[j,i] = sum_pix p_j q_i and dbeta_i = sum_pix q_i ; B4 reduces them.
// ---------------------------------------------------------------------------------------------
template <int CPL>
__global__ void __launch_bounds__(kThreads, 1)
gdn_bwd_q_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                 const float* __restrict__ dy, float* __restrict__ q, float* __restrict__ dx, long long n_pix,
                 GdnFlags f) {
  constexpr int C = CPL * 32;
  constexpr int LDA = C + 4;
  extern __shared__ __align__(16) float smem[];
  float* W = smem;
  float* A = smem + C * C;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < C * C; i += kThreads) W[i] = gamma[i];
  float b[CPL];
#pragma unroll
  for (int m = 0; m < CPL; ++m) b[m] = beta[lane + 32 * m];
  const long long n_tiles = (n_pix + kTM - 1) / kTM;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const long long p0 = t * kTM;
    __syncthreads();
    for (int i = tid; i < kTM * (C / 4); i += kThreads) {
      const int r = i / (C / 4), c4 = i % (C / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p0 + r < n_pix) v = __ldg(reinterpret_cast<const float4*>(x + (p0 + r) * C) + c4);
      v.x = pool_of(v.x, f);
      v.y = pool_of(v.y, f);
      v.z = pool_of(v.z, f);
      v.w = pool_of(v.w, f);
      *reinterpret_cast<float4*>(A + r * LDA + 4 * c4) = v;
    }
    __syncthreads();
    float acc[kPixPerWarp][CPL];
    contract<CPL>(A, W, C, LDA, warp, lane, acc);
#pragma unroll
    for (int p = 0; p < kPixPerWarp; ++p) {
      const long long pix = p0 + warp * kPixPerWarp + p;
      if (pix < n_pix) {
#pragma unroll
        for (int m = 0; m < CPL; ++m) {
          const int ch = lane + 32 * m;
          const float xv = __ldg(x + pix * C + ch);
          const float g = __ldg(dy + pix * C + ch);
          const float u = f.rectify ? fmaxf(xv, 0.f) : xv;
          const float n = b[m] + acc[p][m];
          const float nm = norm_of(n, f);
          q[pix * C + ch] = dl_dn(g, u, n, f);
          dx[pix * C + ch] = f.inverse ? g * nm : g / nm;
        }
      }
    }
  }
}

template <int CPL>
__global__ void __launch_bounds__(kThreads, 1)
gdn_bwd_dx_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ q,
                  float* __restrict__ dx, long long n_pix, GdnFlags f) {
  constexpr int C = CPL * 32;
  constexpr int LDA = C + 4;
  extern __shared__ __align__(16) float smem[];
  float* W = smem;  // gamma^T: W[i][j] = gamma[j][i]
  float* A = smem + C * C;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int idx = tid; idx < C * C; idx += kThreads) {
    const int i = idx / C, j = idx % C;
    W[idx] = gamma[j * C + i];
  }
  const long long n_tiles = (n_pix + kTM - 1) / kTM;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const long long p0 = t * kTM;
    __syncthreads();
    for (int i = tid; i < kTM * (C / 4); i += kThreads) {
      const int r = i / (C / 4), c4 = i % (C / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p0 + r < n_pix) v = __ldg(reinterpret_cast<const float4*>(q + (p0 + r) * C) + c4);
      *reinterpret_cast<float4*>(A + r * LDA + 4 * c4) = v;
    }
    __syncthreads();
    float acc[kPixPerWarp][CPL];
    contract<CPL>(A, W, C, LDA, warp, lane, acc);
#pragma unroll
    for (int p = 0; p < kPixPerWarp; ++p) {
      const long long pix = p0 + warp * kPixPerWarp + p;
      if (pix < n_pix) {
#pragma unroll
        for (int m = 0; m < CPL; ++m) {
          const int ch = lane + 32 * m;
          const float xv = __ldg(x + pix * C + ch);
          const float u = f.rectify ? fmaxf(xv, 0.f) : xv;
          float d = dx[pix * C + ch] + dpool_du(u, f) * acc[p][m];
          if (f.rectify && !(xv > 0.f)) d = 0.f;
          dx[pix * C + ch] = d;
        }
      }
    }
  }
}

// dgamma partials: CTA b owns pixel tiles b, b + grid, ...; thread (tj, ti) owns a (C/16)x(C/16)
// block of dgamma, accumulated in registers over 32-pixel slabs staged in shared memory.
template <int CPL>
__global__ void __launch_bounds__(256, 1)
gdn_bwd_dgamma_kernel(const float* __restrict__ x, const float* __restrict__ q, float* __restrict__ part_g,
                      float* __restrict__ part_b, long long n_pix, GdnFlags f) {
  constexpr int C = CPL * 32;
  constexpr int R = C / 16;  // rows/cols per thread
  constexpr int SL = 32;     // pixels per slab
  __shared__ __align__(16) float P[SL][C];
  __shared__ __align__(16) float Q[SL][C];
  const int tid = threadIdx.x;
  const int tj = tid / 16, ti = tid % 16;
  float acc[R][R];
#pragma unroll
  for (int a = 0; a < R; ++a)
#pragma unroll
    for (int b = 0; b < R; ++b) acc[a][b] = 0.f;
  float bsum = 0.f;  // thread tid < C owns dbeta[tid]
  const long long n_slabs = (n_pix + SL - 1) / SL;
  for (long long s = blockIdx.x; s < n_slabs; s += gridDim.x) {
    const long long p0 = s * SL;
    __syncthreads();
    for (int i = tid; i < SL * (C / 4); i += 256) {
      const int r = i / (C / 4), c4 = i % (C / 4);
      float4 xv = make_float4(0.f, 0.f, 0.f, 0.f), qv = xv;
      if (p0 + r < n_pix) {
        xv = __ldg(reinterpret_cast<const float4*>(x + (p0 + r) * C) + c4);
        qv = __ldg(reinterpret_cast<const float4*>(q + (p0 + r) * C) + c4);
        xv.x = pool_of(xv.x, f);
        xv.y = pool_of(xv.y, f);
        xv.z = pool_of(xv.z, f);
        xv.w = pool_of(xv.w, f);
      }
      *reinterpret_cast<float4*>(&P[r][4 * c4]) = xv;
      *reinterpret_cast<float4*>(&Q[r][4 * c4]) = qv;
    }
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < SL; ++r) {
      float pj[R], qi[R];
#pragma unroll
      for (int a = 0; a < R; ++a) pj[a] = P[r][tj + 16 * a];
#pragma unroll
      for (int b = 0; b < R; ++b) qi[b] = Q[r][ti + 16 * b];
#pragma unroll
      for (int a = 0; a < R; ++a)
#pragma unroll
        for (int b = 0; b < R; ++b) acc[a][b] = fmaf(pj[a], qi[b], acc[a][b]);
    }
    if (tid < C) {
#pragma unroll 8
      for (int r = 0; r < SL; ++r) bsum += Q[r][tid];
    }
  }
  float* pg = part_g + (long long)blockIdx.x * C * C;
#pragma unroll
  for (int a = 0; a < R; ++a)
#pragma unroll
    for (int b = 0; b < R; ++b) pg[(tj + 16 * a) * C + ti + 16 * b] = acc[a][b];
  if (tid < C) part_b[(long long)blockIdx.x * C + tid] = bsum;
}

__global__ void reduce_partials_kernel(const float* __restrict__ part, int n_parts, long long n,
                                       float* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  // pairwise-ish: accumulate in double for a stable, order-deterministic result
  double s = 0.0;
  for (int p = 0; p < n_parts; ++p) s += (double)part[(long long)p * n + i];
  out[i] = (float)s;
}

// Any-C fallback backward: one CTA per launch slice, straightforward loops (small C only).
__global__ void gdn_bwd_generic_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, const float* __restrict__ dy,
                                       float* __restrict__ q, float* __restrict__ dx, long long n_pix, int C,
                                       GdnFlags f) {
  const long long pix = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pix >= n_pix) return;
  const float* xr = x + pix * C;
  for (int i = lane; i < C; i += 32) {
    float n = 0.f;
    for (int j = 0; j < C; ++j) n = fmaf(pool_of(xr[j], f), gamma[(long long)j * C + i], n);
    n = beta[i] + n;
    const float u = f.rectify ? fmaxf(xr[i], 0.f) : xr[i];
    const float g = dy[pix * C + i];
    q[pix * C + i] = dl_dn(g, u, n, f);
    const float nm = norm_of(n, f);
    dx[pix * C + i] = f.inverse ? g * nm : g / nm;
  }
  __syncwarp();
  for (int j = lane; j < C; j += 32) {
    float dp = 0.f;
    for (int i = 0; i < C; ++i) dp = fmaf(gamma[(long long)j * C + i], q[pix * C + i], dp);
    const float xv = xr[j];
    const float u = f.rectify ? fmaxf(xv, 0.f) : xv;
    float d = dx[pix * C + j] + dpool_du(u, f) * dp;
    if (f.rectify && !(xv > 0.f)) d = 0.f;
    dx[pix * C + j] = d;
  }
}

__global__ void gdn_bwd_generic_dgamma_kernel(const float* __restrict__ x, const float* __restrict__ q,
                                              float* __restrict__ dgamma, float* __restrict__ dbeta,
                                              long long n_pix, int C, GdnFlags f) {
  // one thread per (j, i) entry; extra C threads do dbeta.  Small C only.
  const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e < (long long)C * C) {
    const int j = (int)(e / C), i = (int)(e % C);
    double s = 0.0;
    for (long long p = 0; p < n_pix; ++p) s += (double)pool_of(x[p * C + j], f) * (double)q[p * C + i];
    dgamma[e] = (float)s;
  } else if (e < (long long)C * C + C) {
    const int i = (int)(e - (long long)C * C);
    double s = 0.0;
    for (long long p = 0; p < n_pix; ++p) s += (double)q[p * C + i];
    dbeta[i] = (float)s;
  }
}

// Gradients of the two scalar exponents (only needed when they are trainable, gdn.py:345-367): one warp per pixel,
//   n_i = beta_i + sum_j p_j gamma[j, i],   q_i = dL/dn_i,   dp_j = sum_i gamma[j, i] q_i
//   dL/depsilon = sum q_i n_i ln(n_i) / epsilon        (m = n^epsilon:  dL/dm * dm/depsilon = q * n * ln n / epsilon)
//   dL/dalpha   = sum dp_j p_j ln(u_j)                 (p = u^alpha, u > 0)
// Self-contained (recomputes n and q): the fused tensor-core backward does not keep q.  Per-block partials
// [blocks][2], reduced in a fixed order by reduce_partials_kernel.
__global__ void __launch_bounds__(128) gdn_bwd_exponents_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, const float* __restrict__ dy,
                                                                float* __restrict__ part, long long n_pix, int C,
                                                                GdnFlags f) {
  extern __shared__ float qs[];  // [4 warps][C]
  __shared__ float red[4][2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* q = qs + warp * C;
  float dal = 0.f, dep = 0.f;
  for (long long pix = blockIdx.x * 4ll + warp; pix < n_pix; pix += 4ll * gridDim.x) {
    const float* xr = x + pix * C;
    for (int i = lane; i < C; i += 32) {
      float n = 0.f;
      for (int j = 0; j < C; ++j) n = fmaf(pool_of(xr[j], f), gamma[(long long)j * C + i], n);
      n = beta[i] + n;
      const float u = f.rectify ? fmaxf(xr[i], 0.f) : xr[i];
      const float qi = dl_dn(dy[pix * C + i], u, n, f);
      q[i] = qi;
      dep += qi * n * logf(n) / f.eps;
    }
    __syncwarp();
    for (int j = lane; j < C; j += 32) {
      float dp = 0.f;
      for (int i = 0; i < C; ++i) dp = fmaf(gamma[(long long)j * C + i], q[i], dp);
      const float u = f.rectify ? fmaxf(xr[j], 0.f) : xr[j];
      if (u > 0.f) dal += dp * pool_of(xr[j], f) * logf(u);
    }
    __syncwarp();
  }
  for (int o = 16; o > 0; o >>= 1) {
    dal += __shfl_xor_sync(0xFFFFFFFFu, dal, o);
    dep += __shfl_xor_sync(0xFFFFFFFFu, dep, o);
  }
  if (lane == 0) {
    red[warp][0] = dal;
    red[warp][1] = dep;
  }
  __syncthreads();
  if (threadIdx.x < 2)
    part[(long long)blockIdx.x * 2 + threadIdx.x] = red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x];
}

constexpr int kExpGrid = 1184;  // blocks of the exponent-gradient kernel (8 per SM)

int parse_flags(int flags, float alpha, float eps, GdnFlags* f) {
  f->inverse = (flags & TFCB_GDN_INVERSE) != 0;
  f->rectify = (flags & TFCB_GDN_RECTIFY) != 0;
  f->alpha = alpha;
  f->eps = eps;
  f->alpha_mode = (alpha == 1.f) ? 1 : ((alpha == 2.f) ? 2 : 0);
  f->eps_mode = (eps == 1.f) ? 1 : ((eps == 0.5f) ? 2 : 0);
  // trainable exponents: the reference takes `inputs ** alpha` / `norm_pool ** epsilon` whatever the current value
  // (gdn.py:380-388,406-411: the fixed-exponent shortcuts apply only when the parameter is not callable)
  if (flags & TFCB_GDN_POW_ALPHA) f->alpha_mode = 0;
  if (flags & TFCB_GDN_POW_EPSILON) f->eps_mode = 0;
  return TFCB_OK;
}

bool fast_c(int C) { return C % 32 == 0 && C >= 32 && C <= 192; }

size_t fast_smem(int C) { return ((size_t)C * C + (size_t)kTM * (C + 4)) * sizeof(float); }

template <typename K>
int set_smem(K kernel, size_t bytes) {
  TFCB_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return TFCB_OK;
}

}  // namespace

// gdn_tc.cu: the tensor-core kernels; *handled = false where none takes the call
int gdn_tc_forward(int io, const void* x, const float* gamma, const float* beta, void* y, long long n_pix, int C,
                   int flags, float alpha, float eps, cudaStream_t s, bool* handled);
int gdn_tc_backward(int io, const void* x, const float* gamma, const float* beta, const void* dy, void* dx, float* q_ws,
                    float* part_g, float* part_b, int* n_parts, long long n_pix, int C, int flags, float alpha, float eps,
                    cudaStream_t s, bool* handled);

}  // namespace tfcb

using namespace tfcb;

#define DISPATCH_CPL(C, ...)                                   \
  switch ((C) / 32) {                                          \
    case 1: { constexpr int CPL = 1; __VA_ARGS__; } break;     \
    case 2: { constexpr int CPL = 2; __VA_ARGS__; } break;     \
    case 3: { constexpr int CPL = 3; __VA_ARGS__; } break;     \
    case 4: { constexpr int CPL = 4; __VA_ARGS__; } break;     \
    case 5: { constexpr int CPL = 5; __VA_ARGS__; } break;     \
    case 6: { constexpr int CPL = 6; __VA_ARGS__; } break;     \
    default: return fail(TFCB_INVALID_ARGUMENT, "unsupported channel count %d", (C)); \
  }

namespace {

// One forward for every activation type io (0 float32, 1 float16, 2 bfloat16).  The tensor cores take what tc_rule
// (gdn_tc.cu) admits; the rest of the float32 calls run the fp32 kernels, and 16-bit calls have no other kernel.
int gdn_forward(int io, const void* x_dev, const float* gamma_dev, const float* beta_dev, void* y_dev, int64_t n_pix,
                int C, int flags, float alpha, float epsilon, void* stream) {
  if (n_pix < 0 || C <= 0) return fail(TFCB_INVALID_ARGUMENT, "bad GDN shape: n_pix=%lld C=%d", (long long)n_pix, C);
  if (n_pix == 0) return TFCB_OK;
  if (!x_dev || !gamma_dev || !beta_dev || !y_dev) return fail(TFCB_INVALID_ARGUMENT, "null pointer");
  cudaStream_t s = as_stream(stream);
  bool handled = false;
  TFCB_TRY(gdn_tc_forward(io, x_dev, gamma_dev, beta_dev, y_dev, n_pix, C, flags, alpha, epsilon, s, &handled));
  if (handled) return TFCB_OK;
  if (io != 0)
    return fail(TFCB_INVALID_ARGUMENT, "GDN 16-bit: only C in {128, 192} with fixed alpha in {1, 2}, epsilon in {1, 1/2}, 16-byte "
                "aligned x / y / beta (and fewer than 2^31 pixels at C = 192) has a native 16-bit kernel; convert to float32 "
                "for this configuration");
  const float* x = static_cast<const float*>(x_dev);
  float* y = static_cast<float*>(y_dev);
  GdnFlags f;
  parse_flags(flags, alpha, epsilon, &f);
  if (fast_c(C)) {
    const size_t smem = fast_smem(C);
    const long long n_tiles = (n_pix + kTM - 1) / kTM;
    const int grid = (int)std::min<long long>(n_tiles, device_sm_count());
    DISPATCH_CPL(C, {
      TFCB_TRY(set_smem(gdn_fwd_kernel<CPL>, smem));
      gdn_fwd_kernel<CPL><<<grid, kThreads, smem, s>>>(x, gamma_dev, beta_dev, y, n_pix, f);
    });
  } else {
    const long long blocks = (n_pix + 3) / 4;
    gdn_fwd_generic_kernel<<<(unsigned)blocks, 128, 0, s>>>(x, gamma_dev, beta_dev, y, n_pix, C, f);
  }
  TFCB_LAUNCHED();
  TFCB_CUDA_TRY(cudaGetLastError());
  return TFCB_OK;
}

// One backward for every activation type io, on the same terms as gdn_forward.
int gdn_backward(int io, const void* x_dev, const float* gamma_dev, const float* beta_dev, const void* dy_dev,
                 void* dx_dev, float* dgamma_dev, float* dbeta_dev, void* workspace_dev, int64_t n_pix, int C, int flags,
                 float alpha, float epsilon, void* stream) {
  if (n_pix < 0 || C <= 0) return fail(TFCB_INVALID_ARGUMENT, "bad GDN shape: n_pix=%lld C=%d", (long long)n_pix, C);
  if (!x_dev || !gamma_dev || !beta_dev || !dy_dev || !dx_dev || !dgamma_dev || !dbeta_dev || !workspace_dev)
    return fail(TFCB_INVALID_ARGUMENT, "null pointer");
  cudaStream_t s = as_stream(stream);
  if (n_pix == 0) {
    TFCB_CUDA_TRY(cudaMemsetAsync(dgamma_dev, 0, (size_t)C * C * sizeof(float), s));
    TFCB_CUDA_TRY(cudaMemsetAsync(dbeta_dev, 0, (size_t)C * sizeof(float), s));
    return TFCB_OK;
  }
  // the workspace: q (the C = 192 tensor-core kernels: its bf16 operand planes), then the per-CTA partial sums
  float* q = reinterpret_cast<float*>(workspace_dev);
  float* part_g = q + (size_t)((n_pix + 127) / 128 * 128) * C;
  float* part_b = part_g + (size_t)kGdnPartSlots * C * C;
  bool handled = false;
  int n_parts = 0;
  TFCB_TRY(gdn_tc_backward(io, x_dev, gamma_dev, beta_dev, dy_dev, dx_dev, q, part_g, part_b, &n_parts, n_pix, C, flags,
                           alpha, epsilon, s, &handled));
  if (!handled) {
    if (io != 0)
      return fail(TFCB_INVALID_ARGUMENT, "GDN 16-bit backward: only C in {128, 192} with fixed alpha in {1, 2}, epsilon in "
                  "{1, 1/2}, 16-byte aligned x / dy / dx / workspace and fewer than 2^31 pixels has a native 16-bit kernel; "
                  "convert to float32 for this configuration");
    const float* x = static_cast<const float*>(x_dev);
    const float* dy = static_cast<const float*>(dy_dev);
    float* dx = static_cast<float*>(dx_dev);
    GdnFlags f;
    parse_flags(flags, alpha, epsilon, &f);
    if (!fast_c(C)) {
      const long long blocks = (n_pix + 3) / 4;
      gdn_bwd_generic_kernel<<<(unsigned)blocks, 128, 0, s>>>(x, gamma_dev, beta_dev, dy, q, dx, n_pix, C, f);
      const long long e = (long long)C * C + C;
      gdn_bwd_generic_dgamma_kernel<<<(unsigned)((e + 127) / 128), 128, 0, s>>>(x, q, dgamma_dev, dbeta_dev, n_pix, C, f);
      TFCB_LAUNCHED();
      TFCB_LAUNCHED();
      TFCB_CUDA_TRY(cudaGetLastError());
      return TFCB_OK;
    }
    const size_t smem = fast_smem(C);
    const long long n_tiles = (n_pix + kTM - 1) / kTM;
    const int grid = (int)std::min<long long>(n_tiles, device_sm_count());
    n_parts = (int)std::min<long long>((n_pix + 31) / 32, kGdnPartSlots);
    DISPATCH_CPL(C, {
      TFCB_TRY(set_smem(gdn_bwd_q_kernel<CPL>, smem));
      TFCB_TRY(set_smem(gdn_bwd_dx_kernel<CPL>, smem));
      gdn_bwd_q_kernel<CPL><<<grid, kThreads, smem, s>>>(x, gamma_dev, beta_dev, dy, q, dx, n_pix, f);
      gdn_bwd_dx_kernel<CPL><<<grid, kThreads, smem, s>>>(x, gamma_dev, q, dx, n_pix, f);
      gdn_bwd_dgamma_kernel<CPL><<<n_parts, 256, 0, s>>>(x, q, part_g, part_b, n_pix, f);
    });
    TFCB_LAUNCHED();
    TFCB_LAUNCHED();
    TFCB_LAUNCHED();
  }
  const long long ng = (long long)C * C;
  reduce_partials_kernel<<<(unsigned)((ng + 255) / 256), 256, 0, s>>>(part_g, n_parts, ng, dgamma_dev);
  reduce_partials_kernel<<<(unsigned)((C + 255) / 256), 256, 0, s>>>(part_b, n_parts, C, dbeta_dev);
  TFCB_LAUNCHED();
  TFCB_LAUNCHED();
  TFCB_CUDA_TRY(cudaGetLastError());
  return TFCB_OK;
}

}  // namespace

extern "C" {

int tfcb_gdn_forward(const float* x_dev, const float* gamma_dev, const float* beta_dev, float* y_dev,
                     int64_t n_pix, int C, int flags, float alpha, float epsilon, void* stream) {
  return gdn_forward(0, x_dev, gamma_dev, beta_dev, y_dev, n_pix, C, flags, alpha, epsilon, stream);
}

int tfcb_gdn_forward_16bit(const void* x_dev, const float* gamma_dev, const float* beta_dev, void* y_dev, int64_t n_pix,
                           int C, int dtype, int flags, float alpha, float epsilon, void* stream) {
  if (dtype != 1 && dtype != 2) return fail(TFCB_INVALID_ARGUMENT, "GDN 16-bit: dtype must be 1 (float16) or 2 (bfloat16)");
  return gdn_forward(dtype, x_dev, gamma_dev, beta_dev, y_dev, n_pix, C, flags, alpha, epsilon, stream);
}

int64_t tfcb_gdn_backward_workspace_bytes(int64_t n_pix, int C) {
  const int64_t q = ((n_pix + 127) / 128 * 128) * C * (int64_t)sizeof(float);  // whole 128-pixel tiles (the C = 192 tensor-core pair hands q over tile by tile)
  const int64_t parts = (int64_t)kGdnPartSlots * ((int64_t)C * C + C) * (int64_t)sizeof(float);
  return q + parts + 256;
}

int tfcb_gdn_backward(const float* x_dev, const float* gamma_dev, const float* beta_dev, const float* dy_dev,
                      float* dx_dev, float* dgamma_dev, float* dbeta_dev, void* workspace_dev, int64_t n_pix,
                      int C, int flags, float alpha, float epsilon, void* stream) {
  return gdn_backward(0, x_dev, gamma_dev, beta_dev, dy_dev, dx_dev, dgamma_dev, dbeta_dev, workspace_dev, n_pix, C,
                      flags, alpha, epsilon, stream);
}

int tfcb_gdn_backward_16bit(const void* x_dev, const float* gamma_dev, const float* beta_dev, const void* dy_dev,
                            void* dx_dev, float* dgamma_dev, float* dbeta_dev, void* workspace_dev, int64_t n_pix, int C,
                            int dtype, int flags, float alpha, float epsilon, void* stream) {
  if (dtype != 1 && dtype != 2) return fail(TFCB_INVALID_ARGUMENT, "GDN 16-bit: dtype must be 1 (float16) or 2 (bfloat16)");
  return gdn_backward(dtype, x_dev, gamma_dev, beta_dev, dy_dev, dx_dev, dgamma_dev, dbeta_dev, workspace_dev, n_pix, C,
                      flags, alpha, epsilon, stream);
}

int64_t tfcb_gdn_exponent_grads_workspace_bytes(void) { return (int64_t)kExpGrid * 2 * (int64_t)sizeof(float); }

int tfcb_gdn_exponent_grads(const float* x_dev, const float* gamma_dev, const float* beta_dev, const float* dy_dev,
                            float* dalpha_depsilon_dev, void* workspace_dev, int64_t n_pix, int C, int flags,
                            float alpha, float epsilon, void* stream) {
  if (n_pix < 0 || C <= 0) return fail(TFCB_INVALID_ARGUMENT, "bad GDN shape: n_pix=%lld C=%d", (long long)n_pix, C);
  if (!x_dev || !gamma_dev || !beta_dev || !dy_dev || !dalpha_depsilon_dev || !workspace_dev)
    return fail(TFCB_INVALID_ARGUMENT, "null pointer");
  if ((size_t)C * 4 * sizeof(float) > 48 * 1024) return fail(TFCB_INVALID_ARGUMENT, "GDN exponent gradients: C too large");
  cudaStream_t s = as_stream(stream);
  GdnFlags f;
  parse_flags(flags, alpha, epsilon, &f);
  if (n_pix == 0) {
    TFCB_CUDA_TRY(cudaMemsetAsync(dalpha_depsilon_dev, 0, 2 * sizeof(float), s));
    return TFCB_OK;
  }
  const int grid = (int)std::min<long long>((n_pix + 3) / 4, kExpGrid);
  float* part = reinterpret_cast<float*>(workspace_dev);
  gdn_bwd_exponents_kernel<<<grid, 128, (size_t)C * 4 * sizeof(float), s>>>(x_dev, gamma_dev, beta_dev, dy_dev, part, n_pix, C, f);
  reduce_partials_kernel<<<1, 32, 0, s>>>(part, grid, 2, dalpha_depsilon_dev);
  TFCB_LAUNCHED();
  TFCB_LAUNCHED();
  TFCB_CUDA_TRY(cudaGetLastError());
  return TFCB_OK;
}

}  // extern "C"
