// norm.cu -- LayerNorm forward/backward, column sums, and small elementwise helpers (sm_100a).
// All HBM-bound: one pass over the data, 16-byte accesses, fixed-order two-stage reductions
// (deterministic, no float atomics).
//
// LayerNorm: nn.LayerNorm(eps=1e-6) of the reference (dinov2/models/vision_transformer.py:89;
// backbones/adapter_blocks.py:114).  Column sums: bias gradients of nn.Linear and the LayerScale
// gamma gradient (dinov2/layers/layer_scale.py:26-27).
#include "common.cuh"

namespace asis {

constexpr int kLnWarps = 8;  // rows in flight per block

// one warp per row; lane owns float4 vectors v = lane + 32*j, j < NV (C <= 128*NV)
template <typename XT, typename YT, int NV>
__global__ void __launch_bounds__(kLnWarps * 32) ln_fwd_kernel(const XT *__restrict__ x, const float *__restrict__ gamma,
                                                                const float *__restrict__ beta, YT *__restrict__ y,
                                                                float *__restrict__ mean, float *__restrict__ rstd,
                                                                int R, int C, float eps) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * kLnWarps + (threadIdx.x >> 5);
  if (row >= R) return;
  const XT *xr = x + (size_t)row * C;
  float v[NV][4];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int c = 4 * (lane + 32 * j);
    if (c < C) {
      load4(xr + c, v[j]);
      s += v[j][0] + v[j][1] + v[j][2] + v[j][3];
    } else {
      v[j][0] = v[j][1] = v[j][2] = v[j][3] = 0.f;
    }
  }
  const float mu = warp_sum(s) / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int c = 4 * (lane + 32 * j);
    if (c < C) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float d = v[j][i] - mu;
        sq += d * d;
      }
    }
  }
  const float rs = rsqrtf(warp_sum(sq) / (float)C + eps);
  if (lane == 0) {
    if (mean) mean[row] = mu;
    if (rstd) rstd[row] = rs;
  }
  YT *yr = y + (size_t)row * C;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int c = 4 * (lane + 32 * j);
    if (c < C) {
      float g[4], b[4], o[4];
      load4(gamma + c, g);
      load4(beta + c, b);
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = (v[j][i] - mu) * rs * g[i] + b[i];
      store4(yr + c, o);
    }
  }
}

// backward: a block owns kLn2Rows rows per iteration and a thread owns 4 columns (C <= 1024 = 256 x 4), so
// the column partials d gamma / d beta are 8 registers per thread, every element is read once
// (row data stays in registers between the row reduction and the dx pass), and the loads of all
// kLn2Rows rows are in flight together.  Row sums: warp shuffles, then one shared-memory exchange per
// iteration (double buffered: one __syncthreads per kLn2Rows rows).  Each block writes one partial
// row -> workspace[block][2][C].
// Tuning knobs (A/B builds, tools/ln_variants.sh, profiles/r2y_ln_variants.md): rows per block iteration and resident
// blocks per SM (= grid / 148).  4 rows x 3 blocks (80 registers, 28-40 bytes of spills) was the first setting: 78.9 us
// for [21168 x 1024] with the fused residual gradient; 2 rows x 4 blocks (59 registers, no spills): 68.6 us = 4.4 TB/s,
// [83388 x 1024] 253 -> 218 us = 5.5 TB/s; 2 x 5 the same, 2 x 6 / 4 x 4 spill 100+ bytes and are slower, 1 x 8 no gain.
#ifndef ASIS_LN_BWD_ROWS
#define ASIS_LN_BWD_ROWS 2
#endif
#ifndef ASIS_LN_BWD_MINB
#define ASIS_LN_BWD_MINB 4
#endif
constexpr int kLn2Rows = ASIS_LN_BWD_ROWS;
constexpr int kLn2Blocks = ASIS_LN_BWD_MINB * 148;

template <typename DT, typename XT>
__global__ void __launch_bounds__(256, ASIS_LN_BWD_MINB) ln_bwd2_kernel(const DT *__restrict__ dy, const XT *__restrict__ x,
                                                      const float *__restrict__ gamma, const float *__restrict__ mean,
                                                      const float *__restrict__ rstd, const float *__restrict__ dres,
                                                      float *__restrict__ dx, float *__restrict__ partial, int R, int C) {
  __shared__ __align__(16) float red[2][kLn2Rows][2][8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int c = 4 * threadIdx.x;
  const bool on = c < C;
  float g[4] = {0.f, 0.f, 0.f, 0.f}, dg[4] = {0.f, 0.f, 0.f, 0.f}, db[4] = {0.f, 0.f, 0.f, 0.f};
  if (on) load4(gamma + c, g);
  const float invC = 1.f / (float)C;
  int buf = 0;
  for (int row0 = blockIdx.x * kLn2Rows; row0 < R; row0 += gridDim.x * kLn2Rows, buf ^= 1) {
    float d[kLn2Rows][4], xh[kLn2Rows][4], rr[kLn2Rows][4], rs[kLn2Rows], mu[kLn2Rows];
#pragma unroll
    for (int r = 0; r < kLn2Rows; ++r) {
      const int row = row0 + r;
      const bool live = on && row < R;
#pragma unroll
      for (int i = 0; i < 4; ++i) d[r][i] = xh[r][i] = rr[r][i] = 0.f;
      mu[r] = 0.f;
      rs[r] = 0.f;
      if (row < R) {
        mu[r] = __ldg(mean + row);
        rs[r] = __ldg(rstd + row);
      }
      if (live) {
        load4(dy + (size_t)row * C + c, d[r]);
        load4(x + (size_t)row * C + c, xh[r]);
        if (dres) load4(dres + (size_t)row * C + c, rr[r]);
      }
    }
    float s1[kLn2Rows], s2[kLn2Rows];
#pragma unroll
    for (int r = 0; r < kLn2Rows; ++r) {
      s1[r] = s2[r] = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        xh[r][i] = on ? (xh[r][i] - mu[r]) * rs[r] : 0.f;
        const float t = d[r][i] * g[i];
        s1[r] += t;
        s2[r] += t * xh[r][i];
      }
      s1[r] = warp_sum(s1[r]);
      s2[r] = warp_sum(s2[r]);
      if (lane == 0) {
        red[buf][r][0][wid] = s1[r];
        red[buf][r][1][wid] = s2[r];
      }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kLn2Rows; ++r) {
      const float4 a0 = *reinterpret_cast<const float4 *>(&red[buf][r][0][0]);
      const float4 a1 = *reinterpret_cast<const float4 *>(&red[buf][r][0][4]);
      const float4 b0 = *reinterpret_cast<const float4 *>(&red[buf][r][1][0]);
      const float4 b1 = *reinterpret_cast<const float4 *>(&red[buf][r][1][4]);
      const float m1 = (((a0.x + a0.y) + (a0.z + a0.w)) + ((a1.x + a1.y) + (a1.z + a1.w))) * invC;
      const float m2 = (((b0.x + b0.y) + (b0.z + b0.w)) + ((b1.x + b1.y) + (b1.z + b1.w))) * invC;
      const int row = row0 + r;
      if (on && row < R) {
        float o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          dg[i] += d[r][i] * xh[r][i];
          db[i] += d[r][i];
          o[i] = rs[r] * (d[r][i] * g[i] - m1 - xh[r][i] * m2) + rr[r][i];
        }
        store4(dx + (size_t)row * C + c, o);
      }
    }
  }
  if (on) {
    float *pg = partial + (size_t)blockIdx.x * 2 * C;
    store4(pg + c, dg);
    store4(pg + C + c, db);
  }
}

// out[c] (+)= sum over nparts of partial[p][c], fixed order
// (columns [n, 2n) go to out2 when it is given: dgamma and dbeta of LayerNorm in one launch)
// block = 32 columns x PL part-lanes: part-lane y sums parts y, y+PL, ... (coalesced 128-byte rows, four loads in
// flight), the PL part sums are combined through shared memory in a fixed order.  PL = 32 for long part lists (the
// 444-592 block partials of the LayerNorm backward: with 8 lanes each thread walked 55 parts, ~14 dependent load rounds
// = 9.6 us for 3.6 MB; 113 launches per step), 8 otherwise.
template <int PL>
__global__ void __launch_bounds__(32 * PL) reduce_partials_kernel(const float *__restrict__ partial, int nparts, int stride,
                                                                  float *__restrict__ out, float *__restrict__ out2, int n,
                                                                  int accumulate) {
  __shared__ float red[PL][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  const int ncols = out2 ? 2 * n : n;
  float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
  if (c < ncols) {
    int p = ty;
    for (; p + 3 * PL < nparts; p += 4 * PL) {
      t0 += partial[(size_t)p * stride + c];
      t1 += partial[(size_t)(p + PL) * stride + c];
      t2 += partial[(size_t)(p + 2 * PL) * stride + c];
      t3 += partial[(size_t)(p + 3 * PL) * stride + c];
    }
    for (; p < nparts; p += PL) t0 += partial[(size_t)p * stride + c];
  }
  red[ty][tx] = (t0 + t1) + (t2 + t3);
  __syncthreads();
  if (ty == 0 && c < ncols) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < PL; ++w) t += red[w][tx];
    float *dst = c < n ? out + c : out2 + (c - n);
    *dst = accumulate ? *dst + t : t;
  }
}

static void launch_reduce_partials(const float *partial, int nparts, int stride, float *out, float *out2, int n, int accumulate,
                                   cudaStream_t st) {
  const int ncols = out2 ? 2 * n : n;
  if (nparts >= 96) reduce_partials_kernel<32><<<(ncols + 31) / 32, 1024, 0, st>>>(partial, nparts, stride, out, out2, n, accumulate);
  else reduce_partials_kernel<8><<<(ncols + 31) / 32, 256, 0, st>>>(partial, nparts, stride, out, out2, n, accumulate);
}

// column sums of X (optionally X*Y): block = 32 lanes x 8 row-lanes, lane owns 4 columns
template <typename XT, typename YT, bool kMul>
__global__ void __launch_bounds__(256) colsum_kernel(const XT *__restrict__ X, const YT *__restrict__ Y, int64_t ld,
                                                     float *__restrict__ partial, int M, int N) {
  __shared__ float red[8][132];
  const int lane = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + lane * 4;
  float acc[4] = {0, 0, 0, 0};
  if (c < N) {
    // four rows per iteration: four independent loads in flight per lane (one load at a time was latency bound:
    // 88 us for a [83388 x 64] matrix, 46 us = 60 % of the copy roofline for [21180 x 4096])
    const int stride = gridDim.y * 8;
    int r = blockIdx.y * 8 + ty;
    for (; r + 3 * stride < M; r += 4 * stride) {
      float a[4][4], b[4][4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        load4(X + (size_t)(r + u * stride) * ld + c, a[u]);
        if (kMul) load4(Y + (size_t)(r + u * stride) * ld + c, b[u]);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] += kMul ? a[u][i] * b[u][i] : a[u][i];
    }
    for (; r < M; r += stride) {
      float a[4];
      load4(X + (size_t)r * ld + c, a);
      if (kMul) {
        float b[4];
        load4(Y + (size_t)r * ld + c, b);
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] += a[i] * b[i];
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] += a[i];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) red[ty][lane * 4 + i] = acc[i];
  __syncthreads();
  if (threadIdx.x < 128) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
    const int cc = blockIdx.x * 128 + threadIdx.x;
    if (cc < N) partial[(size_t)blockIdx.y * N + cc] = t;
  }
}

// LayerScale backward in one pass over the incoming gradient d [M, N] (f32):
//   du = d * gamma (compute dtype: the gradient of the branch output, next GEMM's operand),
//   partial column sums of d * u (-> d gamma) and of du as stored (-> bias gradient of the branch's last Linear).
// Replaces scale_cols + colsum(d, u) + colsum(du): d is read once instead of twice, du is not re-read.
// block = 32 lanes x 8 row-lanes, lane owns 4 columns; partial[blockIdx.y][2][N].
template <typename UT>
__global__ void __launch_bounds__(256) layerscale_bwd_kernel(const float *__restrict__ d, const UT *__restrict__ u,
                                                             const float *__restrict__ gamma, UT *__restrict__ du,
                                                             float *__restrict__ partial, int M, int N) {
  __shared__ float red[8][132];
  const int lane = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + lane * 4;
  float ag[4] = {0, 0, 0, 0}, ab[4] = {0, 0, 0, 0};
  if (c < N) {
    float g[4];
    load4(gamma + c, g);
    for (int r = blockIdx.y * 8 + ty; r < M; r += gridDim.y * 8) {
      float dv[4], o[4];
      load4(d + (size_t)r * N + c, dv);
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = to_f(from_f<UT>(dv[i] * g[i]));    // as the next GEMM will see it
      store4(du + (size_t)r * N + c, o);
#pragma unroll
      for (int i = 0; i < 4; ++i) ab[i] += o[i];
      if (u) {
        float uv[4];
        load4(u + (size_t)r * N + c, uv);
#pragma unroll
        for (int i = 0; i < 4; ++i) ag[i] += dv[i] * uv[i];
      }
    }
  }
  float *pg = partial + (size_t)blockIdx.y * 2 * N;
  for (int pass = 0; pass < 2; ++pass) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) red[ty][lane * 4 + i] = pass == 0 ? ag[i] : ab[i];
    __syncthreads();
    if (threadIdx.x < 128) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
      const int cc = blockIdx.x * 128 + threadIdx.x;
      if (cc < N) pg[pass * N + cc] = t;
    }
  }
}

template <typename AT, typename OT>
__global__ void __launch_bounds__(256) scale_cols_kernel(const AT *__restrict__ a, const float *__restrict__ gamma,
                                                         OT *__restrict__ out, int64_t M, int N) {
  const int64_t nv = (int64_t)N / 4;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * nv) return;
  const int c = (int)(i % nv) * 4;
  float v[4], g[4];
  load4(a + i * 4, v);
  load4(gamma + c, g);
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] *= g[k];
  store4(out + i * 4, v);
}

template <typename AT, typename BT, typename OT, bool kAdd>
__global__ void __launch_bounds__(256) add_cast_kernel(const AT *__restrict__ a, const BT *__restrict__ b,
                                                       OT *__restrict__ out, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    float v[4];
    load4(a + i, v);
    if (kAdd) {
      float w[4];
      load4(b + i, w);
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] += w[k];
    }
    store4(out + i, v);
  } else {
    for (int64_t k = i; k < n; ++k) out[k] = from_f<OT>(to_f(a[k]) + (kAdd ? to_f(b[k]) : 0.f));
  }
}

static int ln_nv(int C) {
  const int nv = (C + 127) / 128;
  if (nv <= 1) return 1;
  if (nv <= 2) return 2;
  if (nv <= 3) return 3;
  if (nv <= 4) return 4;
  if (nv <= 6) return 6;
  if (nv <= 8) return 8;
  return 0;
}

// ---- SGD with momentum and weight decay over a LIST of tensors (train.py:178-189: torch.optim.SGD(momentum=0.99,
// weight_decay=3e-5)): g' = g + wd p;  buf = momentum buf + g';  p -= lr buf  -- up to kSgdMax tensors per launch, the
// pointer table travels in the kernel parameters (no device-side table: the launch is CUDA-graph capturable as is).
constexpr int kSgdMax = 48;
constexpr int kSgdChunk = 8192;          // elements per block
struct SgdTable {
  float *p[kSgdMax];
  const float *g[kSgdMax];
  float *m[kSgdMax];
  int first_block[kSgdMax + 1];          // blocks [first_block[i], first_block[i+1]) work on tensor i
  long long n[kSgdMax];
  int count;
};
__global__ void __launch_bounds__(256) sgd_kernel(const __grid_constant__ SgdTable t, float lr, float momentum, float wd) {
  int i = 0;
  while (i + 1 < t.count && (int)blockIdx.x >= t.first_block[i + 1]) ++i;          // (<= 48 entries: a short scan)
  const long long base = (long long)((int)blockIdx.x - t.first_block[i]) * kSgdChunk;
  const long long n = t.n[i];
  float *__restrict__ p = t.p[i];
  const float *__restrict__ g = t.g[i];
  float *__restrict__ m = t.m[i];
  const long long end = base + kSgdChunk < n ? base + kSgdChunk : n;
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m)) & 15) == 0;
  if (vec) {
    for (long long e = base + 4 * threadIdx.x; e + 3 < end; e += 4 * 256) {
      float pv[4], gv[4], mv[4];
      load4(p + e, pv);
      load4(g + e, gv);
      load4(m + e, mv);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float gg = gv[k] + wd * pv[k];
        mv[k] = momentum * mv[k] + gg;
        pv[k] = pv[k] - lr * mv[k];
      }
      store4(m + e, mv);
      store4(p + e, pv);
    }
    const long long tail = base + ((end - base) & ~3ll);
    for (long long e = tail + threadIdx.x; e < end; e += 256) {
      const float gg = g[e] + wd * p[e];
      const float mm = momentum * m[e] + gg;
      m[e] = mm;
      p[e] = p[e] - lr * mm;
    }
  } else {
    for (long long e = base + threadIdx.x; e < end; e += 256) {
      const float gg = g[e] + wd * p[e];
      const float mm = momentum * m[e] + gg;
      m[e] = mm;
      p[e] = p[e] - lr * mm;
    }
  }
}

static int ln_bwd_blocks(int R) {
  const int want = (R + kLn2Rows - 1) / kLn2Rows;
  return want < kLn2Blocks ? want : kLn2Blocks;  // resident blocks x 148 SMs (persistent)
}

}  // namespace asis

using namespace asis;

#define LN_NV_SWITCH(nv, ...)                    \
  switch (nv) {                                  \
    case 1: { constexpr int NV = 1; __VA_ARGS__; } break; \
    case 2: { constexpr int NV = 2; __VA_ARGS__; } break; \
    case 3: { constexpr int NV = 3; __VA_ARGS__; } break; \
    case 4: { constexpr int NV = 4; __VA_ARGS__; } break; \
    case 6: { constexpr int NV = 6; __VA_ARGS__; } break; \
    default: { constexpr int NV = 8; __VA_ARGS__; } break; \
  }

extern "C" int asis_layernorm_forward(const void *x, int x_dtype, const float *gamma, const float *beta, void *y,
                                      int y_dtype, float *mean, float *rstd, int R, int C, float eps, void *stream) {
  ASIS_REQUIRE(x && gamma && beta && y, "layernorm_forward: null pointer");
  ASIS_REQUIRE(dtype_ok(x_dtype) && dtype_ok(y_dtype), "layernorm_forward: bad dtype");
  ASIS_REQUIRE(R > 0 && C > 0 && C % 4 == 0, "layernorm_forward: C=%d must be a positive multiple of 4", C);
  const int nv = ln_nv(C);
  if (!nv) ASIS_FAIL(ASIS_ERR_UNSUPPORTED, "layernorm_forward: C=%d > 1024 not supported", C);
  ASIS_REQUIRE(aligned16(x) && aligned16(y) && aligned16(gamma) && aligned16(beta), "layernorm_forward: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (R + kLnWarps - 1) / kLnWarps;
  ASIS_DISPATCH_DTYPE(x_dtype, XT, ASIS_DISPATCH_DTYPE(y_dtype, YT, LN_NV_SWITCH(nv, (ln_fwd_kernel<XT, YT, NV><<<blocks, kLnWarps * 32, 0, st>>>((const XT *)x, gamma, beta, (YT *)y, mean, rstd, R, C, eps)))));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" size_t asis_layernorm_backward_workspace_bytes(int R, int C) {
  return (size_t)ln_bwd_blocks(R) * 2 * C * sizeof(float);
}

extern "C" int asis_layernorm_backward(const void *dy, int dy_dtype, const void *x, int x_dtype, const float *gamma,
                                       const float *mean, const float *rstd, const float *dres, float *dx,
                                       float *dgamma, float *dbeta, int accumulate, int R, int C, void *workspace,
                                       size_t workspace_bytes, void *stream) {
  ASIS_REQUIRE(dy && x && gamma && mean && rstd && dx && workspace, "layernorm_backward: null pointer");
  ASIS_REQUIRE(dtype_ok(dy_dtype) && dtype_ok(x_dtype), "layernorm_backward: bad dtype");
  ASIS_REQUIRE(R > 0 && C > 0 && C % 4 == 0, "layernorm_backward: C=%d must be a positive multiple of 4", C);
  if (C > 1024) ASIS_FAIL(ASIS_ERR_UNSUPPORTED, "layernorm_backward: C=%d > 1024 not supported", C);   // 256 threads x 4 columns
  const size_t need = asis_layernorm_backward_workspace_bytes(R, C);
  if (workspace_bytes < need) ASIS_FAIL(ASIS_ERR_WORKSPACE, "layernorm_backward: workspace %zu < %zu bytes", workspace_bytes, need);
  ASIS_REQUIRE(aligned16(dy) && aligned16(x) && aligned16(dx) && aligned16(gamma) && aligned16(workspace) && (!dres || aligned16(dres)), "layernorm_backward: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = ln_bwd_blocks(R);
  float *partial = (float *)workspace;
  ASIS_DISPATCH_DTYPE(dy_dtype, DT, ASIS_DISPATCH_DTYPE(x_dtype, XT, (ln_bwd2_kernel<DT, XT><<<blocks, 256, 0, st>>>((const DT *)dy, (const XT *)x, gamma, mean, rstd, dres, dx, partial, R, C))));
  ASIS_LAUNCHED();
  if (dgamma && dbeta) {
    launch_reduce_partials(partial, blocks, 2 * C, dgamma, dbeta, C, accumulate, st);
    ASIS_LAUNCHED();
  } else if (dgamma) {
    launch_reduce_partials(partial, blocks, 2 * C, dgamma, nullptr, C, accumulate, st);
    ASIS_LAUNCHED();
  } else if (dbeta) {
    launch_reduce_partials(partial + C, blocks, 2 * C, dbeta, nullptr, C, accumulate, st);
    ASIS_LAUNCHED();
  }
  return ASIS_OK;
}

// row blocks of the column-sum kernels: 128 for wide matrices; narrow ones (few column blocks) get more, so that the
// grid still fills the GPU (a [83388 x 64] sum ran on 128 blocks)
static int colsum_rb(int M, int N = 1 << 30) {
  const int cb = (N + 127) / 128;
  int want = 128;
  if (cb < 8) want = 1024 / cb;
  int rb = (M + 63) / 64;
  if (rb > want) rb = want;
  if (rb < 1) rb = 1;
  return rb;
}

extern "C" size_t asis_colsum_workspace_bytes(int M, int N) { return (size_t)colsum_rb(M, N) * N * sizeof(float); }

extern "C" int asis_colsum(const void *X, int x_dtype, const void *Y, int y_dtype, int64_t ld, float *out,
                           int accumulate, int M, int N, void *workspace, size_t workspace_bytes, void *stream) {
  ASIS_REQUIRE(X && out && workspace, "colsum: null pointer");
  ASIS_REQUIRE(dtype_ok(x_dtype) && (!Y || dtype_ok(y_dtype)), "colsum: bad dtype");
  ASIS_REQUIRE(M > 0 && N > 0 && N % 4 == 0 && ld % 4 == 0 && ld >= N, "colsum: N=%d and ld must be multiples of 4", N);
  const size_t need = asis_colsum_workspace_bytes(M, N);
  if (workspace_bytes < need) ASIS_FAIL(ASIS_ERR_WORKSPACE, "colsum: workspace %zu < %zu bytes", workspace_bytes, need);
  ASIS_REQUIRE(aligned16(X) && (!Y || aligned16(Y)), "colsum: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int rb = colsum_rb(M, N);
  dim3 grid((N + 127) / 128, rb);
  float *partial = (float *)workspace;
  if (Y) {
    ASIS_DISPATCH_DTYPE(x_dtype, XT, ASIS_DISPATCH_DTYPE(y_dtype, YT, (colsum_kernel<XT, YT, true><<<grid, 256, 0, st>>>((const XT *)X, (const YT *)Y, ld, partial, M, N))));
  } else {
    ASIS_DISPATCH_DTYPE(x_dtype, XT, (colsum_kernel<XT, float, false><<<grid, 256, 0, st>>>((const XT *)X, nullptr, ld, partial, M, N)));
  }
  ASIS_LAUNCHED();
  launch_reduce_partials(partial, rb, N, out, nullptr, N, accumulate, st);
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" size_t asis_layerscale_backward_workspace_bytes(int M, int N) { return (size_t)colsum_rb(M) * 2 * N * sizeof(float); }

extern "C" int asis_layerscale_backward(const float *d, const void *u, const float *gamma, void *du, int dtype,
                                        float *dgamma, float *dbias, int M, int N, void *workspace,
                                        size_t workspace_bytes, void *stream) {
  ASIS_REQUIRE(d && gamma && du && workspace, "layerscale_backward: null pointer");
  ASIS_REQUIRE(dtype_ok(dtype), "layerscale_backward: bad dtype");
  ASIS_REQUIRE(!dgamma || u, "layerscale_backward: d gamma needs the saved branch output u");
  ASIS_REQUIRE(M > 0 && N > 0 && N % 4 == 0, "layerscale_backward: N=%d must be a multiple of 4", N);
  const size_t need = asis_layerscale_backward_workspace_bytes(M, N);
  if (workspace_bytes < need) ASIS_FAIL(ASIS_ERR_WORKSPACE, "layerscale_backward: workspace %zu < %zu bytes", workspace_bytes, need);
  ASIS_REQUIRE(aligned16(d) && aligned16(du) && aligned16(gamma) && (!u || aligned16(u)), "layerscale_backward: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int rb = colsum_rb(M);
  dim3 grid((N + 127) / 128, rb);
  float *partial = (float *)workspace;
  ASIS_DISPATCH_DTYPE(dtype, UT, (layerscale_bwd_kernel<UT><<<grid, 256, 0, st>>>(d, dgamma ? (const UT *)u : nullptr, gamma, (UT *)du, partial, M, N)));
  ASIS_LAUNCHED();
  if (dgamma && dbias) {
    launch_reduce_partials(partial, rb, 2 * N, dgamma, dbias, N, 0, st);
    ASIS_LAUNCHED();
  } else if (dgamma) {
    launch_reduce_partials(partial, rb, 2 * N, dgamma, nullptr, N, 0, st);
    ASIS_LAUNCHED();
  } else if (dbias) {
    launch_reduce_partials(partial + N, rb, 2 * N, dbias, nullptr, N, 0, st);
    ASIS_LAUNCHED();
  }
  return ASIS_OK;
}

extern "C" int asis_scale_cols(const void *a, int a_dtype, const float *gamma, void *out, int out_dtype, int64_t M,
                               int N, void *stream) {
  ASIS_REQUIRE(a && gamma && out, "scale_cols: null pointer");
  ASIS_REQUIRE(dtype_ok(a_dtype) && dtype_ok(out_dtype), "scale_cols: bad dtype");
  ASIS_REQUIRE(M > 0 && N > 0 && N % 4 == 0, "scale_cols: N=%d must be a multiple of 4", N);
  ASIS_REQUIRE(aligned16(a) && aligned16(out) && aligned16(gamma), "scale_cols: pointers must be 16-byte aligned");
  const int64_t total = M * (N / 4);
  const unsigned blocks = (unsigned)((total + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  ASIS_DISPATCH_DTYPE(a_dtype, AT, ASIS_DISPATCH_DTYPE(out_dtype, OT, (scale_cols_kernel<AT, OT><<<blocks, 256, 0, st>>>((const AT *)a, gamma, (OT *)out, M, N))));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" int asis_add(const void *a, int a_dtype, const void *b, int b_dtype, void *out, int out_dtype, int64_t n,
                        void *stream) {
  ASIS_REQUIRE(a && b && out && n > 0, "add: null pointer or empty");
  ASIS_REQUIRE(dtype_ok(a_dtype) && dtype_ok(b_dtype) && dtype_ok(out_dtype), "add: bad dtype");
  ASIS_REQUIRE(aligned16(a) && aligned16(b) && aligned16(out), "add: pointers must be 16-byte aligned");
  const unsigned blocks = (unsigned)(((n + 3) / 4 + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  ASIS_DISPATCH_DTYPE(a_dtype, AT, ASIS_DISPATCH_DTYPE(b_dtype, BT, ASIS_DISPATCH_DTYPE(out_dtype, OT, (add_cast_kernel<AT, BT, OT, true><<<blocks, 256, 0, st>>>((const AT *)a, (const BT *)b, (OT *)out, n)))));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" int asis_cast(const void *a, int a_dtype, void *out, int out_dtype, int64_t n, void *stream) {
  ASIS_REQUIRE(a && out && n > 0, "cast: null pointer or empty");
  ASIS_REQUIRE(dtype_ok(a_dtype) && dtype_ok(out_dtype), "cast: bad dtype");
  ASIS_REQUIRE(aligned16(a) && aligned16(out), "cast: pointers must be 16-byte aligned");
  const unsigned blocks = (unsigned)(((n + 3) / 4 + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  ASIS_DISPATCH_DTYPE(a_dtype, AT, ASIS_DISPATCH_DTYPE(out_dtype, OT, (add_cast_kernel<AT, AT, OT, false><<<blocks, 256, 0, st>>>((const AT *)a, nullptr, (OT *)out, n))));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" int asis_sgd_step(int n_tensors, void *const *params, const void *const *grads, void *const *bufs, const int64_t *numels,
                             float lr, float momentum, float weight_decay, void *stream) {
  ASIS_REQUIRE(n_tensors >= 0 && (n_tensors == 0 || (params && grads && bufs && numels)), "sgd_step: null table");
  cudaStream_t st = (cudaStream_t)stream;
  int i = 0;
  while (i < n_tensors) {
    SgdTable t{};
    int blocks = 0, c = 0;
    for (; i < n_tensors && c < kSgdMax; ++i) {
      ASIS_REQUIRE(params[i] && grads[i] && bufs[i] && numels[i] >= 0, "sgd_step: bad entry %d", i);
      if (numels[i] == 0) continue;
      t.p[c] = (float *)params[i];
      t.g[c] = (const float *)grads[i];
      t.m[c] = (float *)bufs[i];
      t.n[c] = numels[i];
      t.first_block[c] = blocks;
      blocks += (int)((numels[i] + kSgdChunk - 1) / kSgdChunk);
      ++c;
    }
    t.first_block[c] = blocks;
    t.count = c;
    if (c == 0) break;
    sgd_kernel<<<blocks, 256, 0, st>>>(t, lr, momentum, weight_decay);
    ASIS_LAUNCHED();
  }
  return ASIS_OK;
}
