// BatchNorm1d (chem/model.py:252,269; bio/model.py:24), the inter-layer ReLU (bio/model.py:281) and
// GraphSAGE's row L2-normalisation (chem/model.py:201-202), forward and backward.
//
// Column statistics are a grid-wide dependency.  Blocks of 32 columns x 8 row-lanes sweep a row chunk with
// coalesced 128-byte loads, accumulate in fp64, fold the 8 lanes in shared memory and add their partial to
// the [2, C] accumulators with fp64 atomics (order-dependent only at the 1e-16 level, i.e. invisible in the
// fp32 results); a finalize pass over the C columns derives mean / invstd / scale / shift.  fp64
// accumulation makes E[x^2]-E[x]^2 safe (relative error ~1e-16 * mean^2/var).
#include "common.cuh"

#include <cstdlib>

namespace {

// PGNN_BN_V4=0 falls back to the scalar sweeps (development switch)
inline bool bn_v4_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("PGNN_BN_V4");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

constexpr int kStatRows = 128;  // rows per block of the statistics sweeps

// sums of f0(row, col) and f1(row, col) over the rows, per column -> acc[0][C], acc[1][C] (fp64 atomics)
template <typename F>
__device__ __forceinline__ void column_pair_sums(int M, int C, double* __restrict__ acc, F f) {
  __shared__ double red[2][8][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  const int r0 = blockIdx.y * kStatRows, r1 = min(M, r0 + kStatRows);
  double s0 = 0.0, s1 = 0.0;
  if (c < C) {
#pragma unroll 4
    for (int r = r0 + w; r < r1; r += 8) {
      double a, b;
      f(r, c, a, b);
      s0 += a;
      s1 += b;
    }
  }
  red[0][w][lane] = s0;
  red[1][w][lane] = s1;
  __syncthreads();
  if (w < 2 && c < C) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[w][k][lane];
    atomicAdd(&acc[(int64_t)w * C + c], t);
  }
}

__global__ void __launch_bounds__(256)
k_bn_stats(const float* __restrict__ x, int64_t ldx, int M, int C, double* __restrict__ acc) {
  pdl_prologue();
  column_pair_sums(M, C, acc, [&](int r, int c, double& a, double& b) {
    const double v = (double)x[(int64_t)r * ldx + c];
    a = v;
    b = v * v;
  });
}

__global__ void __launch_bounds__(128)
k_bn_finalize(const double* __restrict__ acc, int M, int C, const float* __restrict__ gamma, const float* __restrict__ beta,
              float* __restrict__ running_mean, float* __restrict__ running_var, int64_t* __restrict__ nbt, float momentum,
              float eps, float* __restrict__ save_mean, float* __restrict__ save_invstd, float* __restrict__ scale,
              float* __restrict__ shift) {
  pdl_prologue();
  const int c = blockIdx.x * 128 + threadIdx.x;
  if (c == 0 && nbt) *nbt += 1;
  if (c >= C) return;
  const double s = acc[c], ss = acc[(int64_t)C + c];
  const double mean = s / M;
  double var = ss / M - mean * mean;
  var = var < 0.0 ? 0.0 : var;
  const float invstd = (float)(1.0 / sqrt(var + (double)eps));
  const float meanf = (float)mean;
  if (save_mean) save_mean[c] = meanf;
  if (save_invstd) save_invstd[c] = invstd;
  if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * meanf;
  if (running_var) {
    const double unbiased = var * ((double)M / (double)(M > 1 ? M - 1 : 1));
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
  if (scale) {
    const float sc = gamma[c] * invstd;
    scale[c] = sc;
    shift[c] = fmaf(-meanf, sc, beta[c]);
  }
}

__global__ void __launch_bounds__(256)
k_bn_apply(const float* __restrict__ x, int64_t ldx, int64_t M, int C, const float* __restrict__ mean,
           const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta, int relu,
           float* __restrict__ y, int64_t ldy) {
  pdl_prologue();
  const int64_t total = M * C;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C;
    const int c = (int)(idx - r * C);
    float v = fmaf((x[r * ldx + c] - mean[c]) * invstd[c], gamma[c], beta[c]);
    if (relu) v = fmaxf(v, 0.f);
    y[r * ldy + c] = v;
  }
}

// BatchNorm apply with the finalisation folded in (the last encoder layer materialises node_rep this way)
__global__ void __launch_bounds__(256)
k_bn_apply_fold(const float* __restrict__ x, int64_t ldx, int64_t M, int C, PgnnBnFold fold, int relu, float* __restrict__ y,
                int64_t ldy) {
  pdl_prologue();
  extern __shared__ __align__(16) float s_aff[];
  for (int c = threadIdx.x; c < C; c += blockDim.x) bn_fold_column(fold, C, c, blockIdx.x == 0, s_aff[c], s_aff[C + c]);
  __syncthreads();
  const int64_t total = M * C;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C;
    const int c = (int)(idx - r * C);
    float v = fmaf(x[r * ldx + c], s_aff[c], s_aff[C + c]);
    if (relu) v = fmaxf(v, 0.f);
    y[r * ldy + c] = v;
  }
}

__global__ void __launch_bounds__(256)
k_bn_eval(const float* __restrict__ x, int64_t ldx, int64_t M, int C, const float* __restrict__ gamma,
          const float* __restrict__ beta, const float* __restrict__ rm, const float* __restrict__ rv, float eps, int relu,
          float* __restrict__ y, int64_t ldy) {
  pdl_prologue();
  const int64_t total = M * C;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C;
    const int c = (int)(idx - r * C);
    const float invstd = __frcp_rn(__fsqrt_rn(rv[c] + eps));
    float v = fmaf((x[r * ldx + c] - rm[c]) * invstd, gamma[c], beta[c]);
    if (relu) v = fmaxf(v, 0.f);
    y[r * ldy + c] = v;
  }
}

__global__ void __launch_bounds__(256)
k_bn_bwd_stats(const float* __restrict__ gy, int64_t ldgy, const float* __restrict__ x, int64_t ldx, int M, int C,
               const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
               const float* __restrict__ invstd, int relu, double* __restrict__ acc) {
  pdl_prologue();
  column_pair_sums(M, C, acc, [&](int r, int c, double& a, double& b) {
    const float xhat = (x[(int64_t)r * ldx + c] - mean[c]) * invstd[c];
    float d = gy[(int64_t)r * ldgy + c];
    if (relu && !(fmaf(xhat, gamma[c], beta[c]) > 0.f)) d = 0.f;
    a = (double)d;
    b = (double)d * (double)xhat;  // exact product: small batches make the BN backward a difference of large terms
  });
}

__global__ void __launch_bounds__(128)
k_bn_bwd_finalize(const double* __restrict__ acc, int M, int C, float* __restrict__ ggamma, float* __restrict__ gbeta,
                  float* __restrict__ c1, float* __restrict__ c2) {
  pdl_prologue();
  const int c = blockIdx.x * 128 + threadIdx.x;
  if (c >= C) return;
  const double s = acc[c], sx = acc[(int64_t)C + c];
  if (gbeta) gbeta[c] = (float)s;
  if (ggamma) ggamma[c] = (float)sx;
  c1[c] = (float)(s / M);
  c2[c] = (float)(sx / M);
}

__global__ void __launch_bounds__(256)
k_bn_bwd_apply(const float* __restrict__ gy, int64_t ldgy, const float* __restrict__ x, int64_t ldx, int64_t M, int C,
               const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
               const float* __restrict__ invstd, int relu, const float* __restrict__ c1, const float* __restrict__ c2,
               float* __restrict__ gx, int64_t ldgx) {
  pdl_prologue();
  const int64_t total = M * C;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C;
    const int c = (int)(idx - r * C);
    const float xhat = (x[r * ldx + c] - mean[c]) * invstd[c];
    float d = gy[r * ldgy + c];
    if (relu && !(fmaf(xhat, gamma[c], beta[c]) > 0.f)) d = 0.f;
    gx[r * ldgx + c] = gamma[c] * invstd[c] * (d - c1[c] - xhat * c2[c]);
  }
}

// same arithmetic as k_bn_bwd_apply in the 32-column x 8-row-lane block shape of the statistics sweeps, so that the
// column sums of gx (= the bias gradient of the Linear that produced x, chem/model.py:29 mlp[2]) fall out of the same pass
__global__ void __launch_bounds__(256)
k_bn_bwd_apply_colsum(const float* __restrict__ gy, int64_t ldgy, const float* __restrict__ x, int64_t ldx, int M, int C,
                      const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                      const float* __restrict__ invstd, int relu, const double* __restrict__ sums, float* __restrict__ ggamma,
                      float* __restrict__ gbeta, float* __restrict__ gx, int64_t ldgx, float* __restrict__ colsum_part) {
  pdl_prologue();
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  const int r0 = blockIdx.y * kStatRows, r1 = min(M, r0 + kStatRows);
  float acc = 0.f;
  if (c < C) {
    // finalisation of the statistics pass folded in: sum(dy), sum(dy*xhat) -> the two BatchNorm-backward means
    const double sd = sums[c], sdx = sums[(int64_t)C + c];
    if (blockIdx.y == 0 && w == 0) {
      if (gbeta) gbeta[c] = (float)sd;
      if (ggamma) ggamma[c] = (float)sdx;
    }
    const float mu = mean[c], is = invstd[c], ga = gamma[c], be = beta[c], k1 = (float)(sd / M), k2 = (float)(sdx / M);
#pragma unroll 4
    for (int r = r0 + w; r < r1; r += 8) {
      const float xhat = (x[(int64_t)r * ldx + c] - mu) * is;
      float d = gy[(int64_t)r * ldgy + c];
      if (relu && !(fmaf(xhat, ga, be) > 0.f)) d = 0.f;
      const float v = ga * is * (d - k1 - xhat * k2);
      gx[(int64_t)r * ldgx + c] = v;
      acc += v;
    }
  }
  red[w][lane] = acc;
  __syncthreads();
  if (w == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][lane];
    colsum_part[(int64_t)blockIdx.y * C + c] = t;
  }
}

// ---- 16-byte versions of the two BatchNorm-backward sweeps (encoder path: C % 4 == 0, aligned rows) ----------------------
// Tile = 128 columns (one float4 per lane) x kVecRows rows; warp w walks rows r0 + w, r0 + w + 8, ...: every load is a
// 512-byte warp access, 4x fewer instructions than the scalar sweeps and 2 x 8 independent loads in flight per thread.
constexpr int kVecRows = 64;

__device__ __forceinline__ float4 ldg4(const float* p) { return *reinterpret_cast<const float4*>(p); }

__global__ void __launch_bounds__(256)
k_bn_bwd_stats_v4(const float* __restrict__ gy, int64_t ldgy, const float* __restrict__ x, int64_t ldx, int M, int C,
                  const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                  const float* __restrict__ invstd, int relu, double* __restrict__ acc) {
  pdl_prologue();
  __shared__ double red[2][8][128];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + lane * 4;
  const int r0 = blockIdx.y * kVecRows, r1 = min(M, r0 + kVecRows);
  double s0[4] = {0.0, 0.0, 0.0, 0.0}, s1[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < C) {
    const float4 mu = ldg4(mean + c), is = ldg4(invstd + c), ga = ldg4(gamma + c), be = ldg4(beta + c);
    const float muv[4] = {mu.x, mu.y, mu.z, mu.w}, isv[4] = {is.x, is.y, is.z, is.w}, gav[4] = {ga.x, ga.y, ga.z, ga.w},
                bev[4] = {be.x, be.y, be.z, be.w};
#pragma unroll 4
    for (int r = r0 + w; r < r1; r += 8) {
      const float4 xv = ldg4(x + (int64_t)r * ldx + c), gv = ldg4(gy + (int64_t)r * ldgy + c);
      const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float xhat = (xs[q] - muv[q]) * isv[q];
        float d = gs[q];
        if (relu && !(fmaf(xhat, gav[q], bev[q]) > 0.f)) d = 0.f;
        s0[q] += (double)d;
        s1[q] += (double)d * (double)xhat;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    red[0][w][lane * 4 + q] = s0[q];
    red[1][w][lane * 4 + q] = s1[q];
  }
  __syncthreads();
  const int which = threadIdx.x >> 7, col = threadIdx.x & 127;
  if (blockIdx.x * 128 + col < C) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[which][k][col];
    atomicAdd(&acc[(int64_t)which * C + blockIdx.x * 128 + col], t);
  }
}

__global__ void __launch_bounds__(256)
k_bn_bwd_apply_colsum_v4(const float* __restrict__ gy, int64_t ldgy, const float* __restrict__ x, int64_t ldx, int M, int C,
                         const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                         const float* __restrict__ invstd, int relu, const double* __restrict__ sums, float* __restrict__ ggamma,
                         float* __restrict__ gbeta, float* __restrict__ gx, int64_t ldgx, float* __restrict__ colsum_part) {
  pdl_prologue();
  __shared__ float red[8][128];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + lane * 4;
  const int r0 = blockIdx.y * kVecRows, r1 = min(M, r0 + kVecRows);
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  if (c < C) {
    const float4 mu = ldg4(mean + c), is = ldg4(invstd + c), ga = ldg4(gamma + c), be = ldg4(beta + c);
    const float muv[4] = {mu.x, mu.y, mu.z, mu.w}, isv[4] = {is.x, is.y, is.z, is.w}, gav[4] = {ga.x, ga.y, ga.z, ga.w},
                bev[4] = {be.x, be.y, be.z, be.w};
    float k1[4], k2[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const double sd = sums[c + q], sdx = sums[(int64_t)C + c + q];
      k1[q] = (float)(sd / M);
      k2[q] = (float)(sdx / M);
      if (blockIdx.y == 0 && w == 0) {  // finalisation of the statistics pass folded in
        if (gbeta) gbeta[c + q] = (float)sd;
        if (ggamma) ggamma[c + q] = (float)sdx;
      }
    }
#pragma unroll 4
    for (int r = r0 + w; r < r1; r += 8) {
      const float4 xv = ldg4(x + (int64_t)r * ldx + c), gv = ldg4(gy + (int64_t)r * ldgy + c);
      const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
      float o[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float xhat = (xs[q] - muv[q]) * isv[q];
        float d = gs[q];
        if (relu && !(fmaf(xhat, gav[q], bev[q]) > 0.f)) d = 0.f;
        o[q] = gav[q] * isv[q] * (d - k1[q] - xhat * k2[q]);
        acc[q] += o[q];
      }
      *reinterpret_cast<float4*>(gx + (int64_t)r * ldgx + c) = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) red[w][lane * 4 + q] = acc[q];
  __syncthreads();
  if (colsum_part && threadIdx.x < 128 && blockIdx.x * 128 + threadIdx.x < C) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
    colsum_part[(int64_t)blockIdx.y * C + blockIdx.x * 128 + threadIdx.x] = t;
  }
}

// forward statistics and apply in the same 16-byte tiling
__global__ void __launch_bounds__(256)
k_bn_stats_v4(const float* __restrict__ x, int64_t ldx, int M, int C, double* __restrict__ acc) {
  pdl_prologue();
  __shared__ double red[2][8][128];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + lane * 4;
  const int r0 = blockIdx.y * kVecRows, r1 = min(M, r0 + kVecRows);
  double s0[4] = {0.0, 0.0, 0.0, 0.0}, s1[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < C) {
#pragma unroll 8
    for (int r = r0 + w; r < r1; r += 8) {
      const float4 xv = ldg4(x + (int64_t)r * ldx + c);
      const double v[4] = {(double)xv.x, (double)xv.y, (double)xv.z, (double)xv.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        s0[q] += v[q];
        s1[q] += v[q] * v[q];
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    red[0][w][lane * 4 + q] = s0[q];
    red[1][w][lane * 4 + q] = s1[q];
  }
  __syncthreads();
  const int which = threadIdx.x >> 7, col = threadIdx.x & 127;
  if (blockIdx.x * 128 + col < C) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[which][k][col];
    atomicAdd(&acc[(int64_t)which * C + blockIdx.x * 128 + col], t);
  }
}

__global__ void __launch_bounds__(256)
k_bn_apply_v4(const float* __restrict__ x, int64_t ldx, int64_t M, int C4, const float* __restrict__ mean,
              const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta, int relu,
              float* __restrict__ y, int64_t ldy) {
  pdl_prologue();
  const int64_t total = M * C4;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C4;
    const int c = (int)(idx - r * C4) * 4;
    const float4 xv = ldg4(x + r * ldx + c), mu = ldg4(mean + c), is = ldg4(invstd + c), ga = ldg4(gamma + c), be = ldg4(beta + c);
    float4 o;
    o.x = fmaf((xv.x - mu.x) * is.x, ga.x, be.x);
    o.y = fmaf((xv.y - mu.y) * is.y, ga.y, be.y);
    o.z = fmaf((xv.z - mu.z) * is.z, ga.z, be.z);
    o.w = fmaf((xv.w - mu.w) * is.w, ga.w, be.w);
    if (relu) {
      o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
    }
    *reinterpret_cast<float4*>(y + r * ldy + c) = o;
  }
}

__global__ void __launch_bounds__(256)
k_relu_fwd(const float* __restrict__ x, int64_t ldx, int64_t M, int C, float* __restrict__ y, int64_t ldy) {
  pdl_prologue();
  const int64_t total = M * C;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C;
    const int c = (int)(idx - r * C);
    y[r * ldy + c] = fmaxf(x[r * ldx + c], 0.f);
  }
}
__global__ void __launch_bounds__(256)
k_relu_bwd(const float* __restrict__ gy, int64_t ldgy, const float* __restrict__ y, int64_t ldy, int64_t M, int C,
           float* __restrict__ gx, int64_t ldgx) {
  pdl_prologue();
  const int64_t total = M * C;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C;
    const int c = (int)(idx - r * C);
    gx[r * ldgx + c] = y[r * ldy + c] > 0.f ? gy[r * ldgy + c] : 0.f;
  }
}

// float4 variants (rows 16-byte aligned, C % 4 == 0): one 64-bit division per FOUR elements instead of one per element, 16-byte
// accesses.  The scalar kernels ran at ~2.5 TB/s on the bio step's [32 k, 300] activations (180 us per step for four ReLU backward sweeps).
__global__ void __launch_bounds__(256)
k_relu_fwd_v4(const float* __restrict__ x, int64_t ldx, int64_t M, int C4, float* __restrict__ y, int64_t ldy) {
  pdl_prologue();
  const int64_t total = M * C4;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C4;
    const int c = (int)(idx - r * C4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(x + r * ldx + c);
    *reinterpret_cast<float4*>(y + r * ldy + c) = make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
  }
}
__global__ void __launch_bounds__(256)
k_relu_bwd_v4(const float* __restrict__ gy, int64_t ldgy, const float* __restrict__ y, int64_t ldy, int64_t M, int C4,
              float* __restrict__ gx, int64_t ldgx) {
  pdl_prologue();
  const int64_t total = M * C4;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / C4;
    const int c = (int)(idx - r * C4) * 4;
    const float4 g = *reinterpret_cast<const float4*>(gy + r * ldgy + c);
    const float4 v = *reinterpret_cast<const float4*>(y + r * ldy + c);
    *reinterpret_cast<float4*>(gx + r * ldgx + c) =
        make_float4(v.x > 0.f ? g.x : 0.f, v.y > 0.f ? g.y : 0.f, v.z > 0.f ? g.z : 0.f, v.w > 0.f ? g.w : 0.f);
  }
}

// one warp per row
__global__ void __launch_bounds__(256)
k_l2norm_fwd(const float* __restrict__ x, int64_t ldx, int64_t M, int C, float* __restrict__ y, int64_t ldy,
             float* __restrict__ norm) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  for (int64_t r = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); r < M; r += (int64_t)gridDim.x * (blockDim.x >> 5)) {
    float ss = 0.f;
    for (int c = lane; c < C; c += 32) { const float v = x[r * ldx + c]; ss = fmaf(v, v, ss); }
    ss = warp_sum(ss);
    const float nrm = fmaxf(sqrtf(ss), 1e-12f);  // F.normalize: x / max(||x||, eps)
    if (lane == 0) norm[r] = nrm;
    for (int c = lane; c < C; c += 32) y[r * ldy + c] = x[r * ldx + c] / nrm;
  }
}
__global__ void __launch_bounds__(256)
k_l2norm_bwd(const float* __restrict__ gy, int64_t ldgy, const float* __restrict__ y, int64_t ldy, const float* __restrict__ norm,
             int64_t M, int C, float* __restrict__ gx, int64_t ldgx) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  for (int64_t r = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); r < M; r += (int64_t)gridDim.x * (blockDim.x >> 5)) {
    float dot = 0.f;
    for (int c = lane; c < C; c += 32) dot = fmaf(gy[r * ldgy + c], y[r * ldy + c], dot);
    dot = warp_sum(dot);
    const float nrm = norm[r];
    // y = x / n with n = max(||x||, eps); for ||x|| > eps: gx = (gy - y * <gy, y>) / n; below eps n is constant
    const bool clamped = nrm <= 1e-12f;
    for (int c = lane; c < C; c += 32) {
      const float g = gy[r * ldgy + c];
      gx[r * ldgx + c] = clamped ? g / nrm : (g - y[r * ldy + c] * dot) / nrm;
    }
  }
}

inline int grid_items(int64_t items, int threads) {
  int64_t b = ceil_div(items, threads);
  const int64_t cap = (int64_t)kNumSMs * 16;
  if (b > cap) b = cap;
  return (int)(b < 1 ? 1 : b);
}

}  // namespace

// encoder.cu: BatchNorm forward when the column sums / sums of squares were already accumulated (fp64, [2][C]) by the
// epilogue of the GEMM that produced x (PgnnGemmHooks::stats)
int pgnn_internal_bn_apply_fold(const float* x, int64_t ldx, int64_t M, int64_t C, const PgnnBnFold& fold, int relu, float* y,
                                int64_t ldy, cudaStream_t st) {
  PGNN_CUDA(pgnn_launch(k_bn_apply_fold, dim3(grid_items(M * C, 256)), dim3(256), sizeof(float) * 2 * C, st, x, ldx, M, (int)C, fold, relu, y, ldy));
  PGNN_LAUNCH_CHECK();
  return PGNN_OK;
}

// Row blocks of the BatchNorm-backward sweeps below (either variant) for M rows: the size of colsum_part is this x C floats.
int64_t pgnn_internal_bn_colsum_parts(int64_t M) { return ceil_div(M > 0 ? M : 1, (int64_t)(kVecRows < kStatRows ? kVecRows : kStatRows)); }

// encoder.cu: pgnn_bn_bwd that also leaves the column sums of gx, per row block, in colsum_part[*parts][C]; the caller folds
// them in block order (pgnn_internal_fold_colsums).  The column sum is the gradient of the bias in front of the BatchNorm:
// zero in exact arithmetic, so what is computed is cancellation noise, which a fixed summation order keeps the same from run
// to run (atomics in arrival order did not).
int pgnn_internal_bn_bwd_colsum(const float* gy, int64_t ldgy, const float* x, int64_t ldx, int64_t M, int64_t C, const float* gamma,
                                const float* beta, const float* save_mean, const float* save_invstd, int relu, float* gx,
                                int64_t ldgx, float* ggamma, float* gbeta, float* colsum_part, int* parts, void* workspace, cudaStream_t st) {
  double* acc = reinterpret_cast<double*>(workspace);
  PGNN_CUDA(cudaMemsetAsync(acc, 0, sizeof(double) * 2 * C, st));
  auto a16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  if (bn_v4_enabled() && C % 4 == 0 && ldgy % 4 == 0 && ldx % 4 == 0 && ldgx % 4 == 0 && a16(gy) && a16(x) && a16(gx) && a16(gamma) && a16(beta) &&
      a16(save_mean) && a16(save_invstd)) {
    dim3 gv((unsigned)ceil_div(C, 128), (unsigned)ceil_div(M, kVecRows));
    PGNN_CUDA(pgnn_launch(k_bn_bwd_stats_v4, dim3(gv), dim3(256), 0, st, gy, ldgy, x, ldx, (int)M, (int)C, gamma, beta, save_mean, save_invstd, relu, acc));
    PGNN_LAUNCH_CHECK();
    PGNN_CUDA(pgnn_launch(k_bn_bwd_apply_colsum_v4, dim3(gv), dim3(256), 0, st, gy, ldgy, x, ldx, (int)M, (int)C, gamma, beta, save_mean, save_invstd,
                          relu, (const double*)acc, ggamma, gbeta, gx, ldgx, colsum_part));
    PGNN_LAUNCH_CHECK();
    *parts = (int)gv.y;
    return PGNN_OK;
  }
  dim3 g1((unsigned)ceil_div(C, 32), (unsigned)ceil_div(M, kStatRows));
  PGNN_CUDA(pgnn_launch(k_bn_bwd_stats, dim3(g1), dim3(256), 0, st, gy, ldgy, x, ldx, (int)M, (int)C, gamma, beta, save_mean, save_invstd, relu, acc));
  PGNN_LAUNCH_CHECK();
  PGNN_CUDA(pgnn_launch(k_bn_bwd_apply_colsum, dim3(g1), dim3(256), 0, st, gy, ldgy, x, ldx, (int)M, (int)C, gamma, beta, save_mean, save_invstd, relu,
                        (const double*)acc, ggamma, gbeta, gx, ldgx, colsum_part));
  PGNN_LAUNCH_CHECK();
  *parts = (int)g1.y;
  return PGNN_OK;
}

namespace {
constexpr int kMaxFoldJobs = 16;
struct ColsumFolds {
  const float* part[kMaxFoldJobs];
  float* out[kMaxFoldJobs];
  int parts[kMaxFoldJobs];
};
// out[j][c] = sum over b = 0, 1, ... of part[j][b][c]; blockIdx.y = job
__global__ void __launch_bounds__(256) k_fold_colsums(ColsumFolds f, int C) {
  pdl_prologue();
  const int j = blockIdx.y;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    float a = 0.f;
    for (int b = 0; b < f.parts[j]; ++b) a += f.part[j][(int64_t)b * C + c];
    f.out[j][c] = a;
  }
}
}  // namespace

// folds the row-block partials of `count` pgnn_internal_bn_bwd_colsum calls (all with C columns), one launch per 16
int pgnn_internal_fold_colsums(const float* const* part, const int* parts, float* const* out, int count, int64_t C, cudaStream_t st) {
  for (int first = 0; first < count; first += kMaxFoldJobs) {
    ColsumFolds f;
    const int k = count - first < kMaxFoldJobs ? count - first : kMaxFoldJobs;
    for (int i = 0; i < k; ++i) {
      f.part[i] = part[first + i];
      f.out[i] = out[first + i];
      f.parts[i] = parts[first + i];
    }
    PGNN_CUDA(pgnn_launch(k_fold_colsums, dim3((unsigned)ceil_div(C, 256), (unsigned)k), dim3(256), 0, st, f, (int)C));
    PGNN_LAUNCH_CHECK();
  }
  return PGNN_OK;
}

extern "C" {

int64_t pgnn_bn_workspace_bytes(int64_t M, int64_t C) {
  if (M < 0 || C <= 0) return PGNN_EINVAL;
  return align_up(2 * C * 8, 256) + align_up(2 * C * 4, 256);
}

int pgnn_bn_fwd_train(const float* x, int64_t ldx, int64_t M, int64_t C, const float* gamma, const float* beta,
                      float* running_mean, float* running_var, int64_t* num_batches_tracked, float momentum, float eps, int relu,
                      float* y, int64_t ldy, float* save_mean, float* save_invstd, float* scale, float* shift, void* workspace,
                      int64_t workspace_bytes, void* stream) {
  PGNN_CHECK_ARG(M > 0 && C > 0 && M < (1ll << 31) && x && gamma && beta && save_mean && save_invstd && workspace);
  PGNN_CHECK_ARG((scale == nullptr) == (shift == nullptr));
  if (workspace_bytes < pgnn_bn_workspace_bytes(M, C)) return PGNN_EWORKSPACE;
  cudaStream_t st = as_stream(stream);
  double* acc = reinterpret_cast<double*>(workspace);
  PGNN_CUDA(cudaMemsetAsync(acc, 0, sizeof(double) * 2 * C, st));
  auto a16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const bool v4 = bn_v4_enabled() && C % 4 == 0 && ldx % 4 == 0 && a16(x) && a16(gamma) && a16(beta) && a16(save_mean) && a16(save_invstd) &&
                  (!y || (ldy % 4 == 0 && a16(y)));
  if (v4) {
    dim3 gv((unsigned)ceil_div(C, 128), (unsigned)ceil_div(M, kVecRows));
    PGNN_CUDA(pgnn_launch(k_bn_stats_v4, dim3(gv), dim3(256), 0, st, x, ldx, (int)M, (int)C, acc));
  } else {
    dim3 g1((unsigned)ceil_div(C, 32), (unsigned)ceil_div(M, kStatRows));
    PGNN_CUDA(pgnn_launch(k_bn_stats, dim3(g1), dim3(256), 0, st, x, ldx, (int)M, (int)C, acc));
  }
  PGNN_LAUNCH_CHECK();
  PGNN_CUDA(pgnn_launch(k_bn_finalize, dim3((unsigned)ceil_div(C, 128)), dim3(128), 0, st, acc, (int)M, (int)C, gamma, beta, running_mean, running_var,
                                                           num_batches_tracked, momentum, eps, save_mean, save_invstd, scale,
                                                           shift));
  PGNN_LAUNCH_CHECK();
  if (y) {
    if (v4) PGNN_CUDA(pgnn_launch(k_bn_apply_v4, dim3(grid_items(M * (C / 4), 256)), dim3(256), 0, st, x, ldx, M, (int)(C / 4), save_mean, save_invstd, gamma, beta, relu, y, ldy));
    else PGNN_CUDA(pgnn_launch(k_bn_apply, dim3(grid_items(M * C, 256)), dim3(256), 0, st, x, ldx, M, (int)C, save_mean, save_invstd, gamma, beta, relu, y, ldy));
    PGNN_LAUNCH_CHECK();
  }
  return PGNN_OK;
}

int pgnn_bn_fwd_eval(const float* x, int64_t ldx, int64_t M, int64_t C, const float* gamma, const float* beta,
                     const float* running_mean, const float* running_var, float eps, int relu, float* y, int64_t ldy,
                     void* stream) {
  PGNN_CHECK_ARG(M >= 0 && C > 0);
  if (M == 0) return PGNN_OK;
  PGNN_CHECK_ARG(x && gamma && beta && running_mean && running_var && y);
  PGNN_CUDA(pgnn_launch(k_bn_eval, dim3(grid_items(M * C, 256)), dim3(256), 0, as_stream(stream), x, ldx, M, (int)C, gamma, beta, running_mean, running_var, eps,
                                                                    relu, y, ldy));
  PGNN_LAUNCH_CHECK();
  return PGNN_OK;
}

int pgnn_bn_bwd(const float* gy, int64_t ldgy, const float* x, int64_t ldx, int64_t M, int64_t C, const float* gamma,
                const float* beta, const float* save_mean, const float* save_invstd, int relu, float* gx, int64_t ldgx,
                float* ggamma, float* gbeta, void* workspace, int64_t workspace_bytes, void* stream) {
  PGNN_CHECK_ARG(M > 0 && C > 0 && M < (1ll << 31) && gy && x && gamma && beta && save_mean && save_invstd && gx && workspace);
  if (workspace_bytes < pgnn_bn_workspace_bytes(M, C)) return PGNN_EWORKSPACE;
  cudaStream_t st = as_stream(stream);
  double* acc = reinterpret_cast<double*>(workspace);
  float* c1 = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + align_up(2 * C * 8, 256));
  float* c2 = c1 + C;
  PGNN_CUDA(cudaMemsetAsync(acc, 0, sizeof(double) * 2 * C, st));
  {
    auto a16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    if (bn_v4_enabled() && C % 4 == 0 && ldgy % 4 == 0 && ldx % 4 == 0 && ldgx % 4 == 0 && a16(gy) && a16(x) && a16(gx) && a16(gamma) && a16(beta) &&
        a16(save_mean) && a16(save_invstd)) {
      dim3 gv((unsigned)ceil_div(C, 128), (unsigned)ceil_div(M, kVecRows));
      PGNN_CUDA(pgnn_launch(k_bn_bwd_stats_v4, dim3(gv), dim3(256), 0, st, gy, ldgy, x, ldx, (int)M, (int)C, gamma, beta, save_mean, save_invstd, relu, acc));
      PGNN_LAUNCH_CHECK();
      PGNN_CUDA(pgnn_launch(k_bn_bwd_apply_colsum_v4, dim3(gv), dim3(256), 0, st, gy, ldgy, x, ldx, (int)M, (int)C, gamma, beta, save_mean, save_invstd,
                            relu, (const double*)acc, ggamma, gbeta, gx, ldgx, (float*)nullptr));
      PGNN_LAUNCH_CHECK();
      return PGNN_OK;
    }
  }
  dim3 g1((unsigned)ceil_div(C, 32), (unsigned)ceil_div(M, kStatRows));
  PGNN_CUDA(pgnn_launch(k_bn_bwd_stats, dim3(g1), dim3(256), 0, st, gy, ldgy, x, ldx, (int)M, (int)C, gamma, beta, save_mean, save_invstd, relu, acc));
  PGNN_LAUNCH_CHECK();
  PGNN_CUDA(pgnn_launch(k_bn_bwd_finalize, dim3((unsigned)ceil_div(C, 128)), dim3(128), 0, st, acc, (int)M, (int)C, ggamma, gbeta, c1, c2));
  PGNN_LAUNCH_CHECK();
  PGNN_CUDA(pgnn_launch(k_bn_bwd_apply, dim3(grid_items(M * C, 256)), dim3(256), 0, st, gy, ldgy, x, ldx, M, (int)C, gamma, beta, save_mean, save_invstd, relu,
                                                        c1, c2, gx, ldgx));
  PGNN_LAUNCH_CHECK();
  return PGNN_OK;
}

int pgnn_relu_fwd(const float* x, int64_t ldx, int64_t M, int64_t C, float* y, int64_t ldy, void* stream) {
  PGNN_CHECK_ARG(M >= 0 && C > 0);
  if (M == 0) return PGNN_OK;
  PGNN_CHECK_ARG(x && y);
  if (C % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0) {
    PGNN_CUDA(pgnn_launch(k_relu_fwd_v4, dim3(grid_items(M * (C / 4), 256)), dim3(256), 0, as_stream(stream), x, ldx, M, (int)(C / 4), y, ldy));
    PGNN_LAUNCH_CHECK();
    return PGNN_OK;
  }
  PGNN_CUDA(pgnn_launch(k_relu_fwd, dim3(grid_items(M * C, 256)), dim3(256), 0, as_stream(stream), x, ldx, M, (int)C, y, ldy));
  PGNN_LAUNCH_CHECK();
  return PGNN_OK;
}

int pgnn_relu_bwd(const float* gy, int64_t ldgy, const float* y, int64_t ldy_, int64_t M, int64_t C, float* gx, int64_t ldgx,
                  void* stream) {
  PGNN_CHECK_ARG(M >= 0 && C > 0);
  if (M == 0) return PGNN_OK;
  PGNN_CHECK_ARG(gy && y && gx);
  if (C % 4 == 0 && ldgy % 4 == 0 && ldy_ % 4 == 0 && ldgx % 4 == 0 &&
      ((reinterpret_cast<uintptr_t>(gy) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gx)) & 15) == 0) {
    PGNN_CUDA(pgnn_launch(k_relu_bwd_v4, dim3(grid_items(M * (C / 4), 256)), dim3(256), 0, as_stream(stream), gy, ldgy, y, ldy_, M, (int)(C / 4), gx, ldgx));
    PGNN_LAUNCH_CHECK();
    return PGNN_OK;
  }
  PGNN_CUDA(pgnn_launch(k_relu_bwd, dim3(grid_items(M * C, 256)), dim3(256), 0, as_stream(stream), gy, ldgy, y, ldy_, M, (int)C, gx, ldgx));
  PGNN_LAUNCH_CHECK();
  return PGNN_OK;
}

int pgnn_l2norm_fwd(const float* x, int64_t ldx, int64_t M, int64_t C, float* y, int64_t ldy, float* norm, void* stream) {
  PGNN_CHECK_ARG(M >= 0 && C > 0);
  if (M == 0) return PGNN_OK;
  PGNN_CHECK_ARG(x && y && norm);
  PGNN_CUDA(pgnn_launch(k_l2norm_fwd, dim3(grid_items(M * 32, 256)), dim3(256), 0, as_stream(stream), x, ldx, M, (int)C, y, ldy, norm));
  PGNN_LAUNCH_CHECK();
  return PGNN_OK;
}

int pgnn_l2norm_bwd(const float* gy, int64_t ldgy, const float* y, int64_t ldy_, const float* norm, int64_t M, int64_t C,
                    float* gx, int64_t ldgx, void* stream) {
  PGNN_CHECK_ARG(M >= 0 && C > 0);
  if (M == 0) return PGNN_OK;
  PGNN_CHECK_ARG(gy && y && norm && gx);
  PGNN_CUDA(pgnn_launch(k_l2norm_bwd, dim3(grid_items(M * 32, 256)), dim3(256), 0, as_stream(stream), gy, ldgy, y, ldy_, norm, M, (int)C, gx, ldgx));
  PGNN_LAUNCH_CHECK();
  return PGNN_OK;
}

}  // extern "C"
