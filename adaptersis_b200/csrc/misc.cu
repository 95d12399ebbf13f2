// misc.cu -- patch gather for the patch-embedding GEMM and the token-major depth-wise 3x3
// convolution of the extractor's ConvFFN (sm_100a; HBM-bound, 16-byte channel vectors).
//   patchify <- PatchEmbed.forward (dinov2/layers/patch_embed.py:65-81): stride-p conv == GEMM
//   dwconv   <- DWConv.forward (backbones/adapter_blocks.py:62-80): the reference transposes each
//               pyramid level to NCHW, runs cuDNN, transposes back; here the conv runs directly
//               on the [B, tokens, C] layout (channels are the contiguous dimension).
#include <algorithm>

#include "common.cuh"

namespace asis {

template <typename OT>
__global__ void __launch_bounds__(256) patchify_kernel(const float *__restrict__ img, OT *__restrict__ cols, int B, int Cin,
                                                       int Himg, int Wimg, int patch, int64_t ldk) {
  const int gh = Himg / patch, gw = Wimg / patch;
  const int K = Cin * patch * patch;
  const int64_t total = (int64_t)B * gh * gw * ldk;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int k = (int)(i % ldk);
  const int64_t row = i / ldk;
  float v = 0.f;
  if (k < K) {
    const int dx = k % patch, dy = (k / patch) % patch, c = k / (patch * patch);
    const int px = (int)(row % gw), py = (int)((row / gw) % gh), b = (int)(row / ((int64_t)gw * gh));
    v = img[(((int64_t)b * Cin + c) * Himg + py * patch + dy) * Wimg + px * patch + dx];
  }
  cols[i] = from_f<OT>(v);
}

constexpr int kMaxMaps = 4;
struct Maps {
  int n;
  int h[kMaxMaps], w[kMaxMaps], start[kMaxMaps + 1];
};

__device__ __forceinline__ int find_map(const Maps &mp, int tok) {
  int i = 0;
#pragma unroll
  for (int k = 1; k < kMaxMaps; ++k)
    if (k < mp.n && tok >= mp.start[k]) i = k;
  return i;
}

// one thread per (b, token, 4 channels), kDwIter such items per thread.
// The nine taps of all channels sit transposed in shared memory ([9][C], filled with coalesced loads): read from the
// [C][9] parameter directly, a warp's tap load touches 32 different 128-byte lines (stride 36 bytes x 4 channels), 36 such
// loads per thread -- the first version spent its time there (210 us per [12, 6949, 256] bf16 call, 14x the copy
// roofline).  The nine neighbour loads are unconditional (clamped coordinates, the tap zeroed outside the map), so they
// are all in flight together instead of one per resolved branch.
constexpr int kDwIter = 4;
template <typename T>
__global__ void __launch_bounds__(256) dwconv_fwd_kernel(const T *__restrict__ x, const float *__restrict__ weight,
                                                         const float *__restrict__ bias, T *__restrict__ pre,
                                                         T *__restrict__ y, int B, int C, int ntok, Maps mp,
                                                         int fuse_gelu) {
  extern __shared__ __align__(16) float dw_taps[];     // [9][C]
  for (int i = threadIdx.x; i < 9 * C; i += blockDim.x) dw_taps[(i % 9) * C + i / 9] = __ldg(weight + i);
  __syncthreads();
  const int cv = C / 4;
  const int64_t total = (int64_t)B * ntok * cv;
  for (int it = 0; it < kDwIter; ++it) {
    const int64_t i = ((int64_t)blockIdx.x * kDwIter + it) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = (int)(i % cv) * 4;
    const int tok = (int)((i / cv) % ntok);
    const int b = (int)(i / ((int64_t)cv * ntok));
    const int mi = find_map(mp, tok);
    const int W = mp.w[mi], H = mp.h[mi], t0 = mp.start[mi];
    const int py = (tok - t0) / W, px = (tok - t0) % W;
    float acc[4];
    load4(bias + c, acc);
    const T *xb = x + ((int64_t)b * ntok + t0) * C + c;
    float v[9][4];
    bool ok[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      const int yy = py + j / 3 - 1, xx = px + j % 3 - 1;
      ok[j] = yy >= 0 && yy < H && xx >= 0 && xx < W;
      const int yc = min(max(yy, 0), H - 1), xc = min(max(xx, 0), W - 1);
      load4(xb + (int64_t)(yc * W + xc) * C, v[j]);
    }
#pragma unroll
    for (int j = 0; j < 9; ++j) {      // same order and the same fused multiply-adds as a loop that skips the outside taps
      const float4 w4 = *reinterpret_cast<const float4 *>(dw_taps + j * C + c);
      if (ok[j]) {
        acc[0] += v[j][0] * w4.x;
        acc[1] += v[j][1] * w4.y;
        acc[2] += v[j][2] * w4.z;
        acc[3] += v[j][3] * w4.w;
      }
    }
    const int64_t o = ((int64_t)b * ntok + tok) * C + c;
    if (fuse_gelu) {
      if (pre) store4(pre + o, acc);
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[k] = gelu_erf(acc[k]);
    }
    store4(y + o, acc);
  }
}

// g = dy * GELU'(pre), once per element: the 3x3 backward below reads the gradient at 9 neighbours, and
// recomputing erf-GELU' for each of them made it 680 us per [12, 6949, 256] call (instruction bound)
template <typename T>
__global__ void __launch_bounds__(256) dwconv_gelu_grad_kernel(const T *__restrict__ dy, const T *__restrict__ pre,
                                                               T *__restrict__ g, int64_t n4) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float d[4], h[4];
  load4(dy + 4 * i, d);
  load4(pre + 4 * i, h);
#pragma unroll
  for (int k = 0; k < 4; ++k) d[k] *= dgelu_erf(h[k]);
  store4(g + 4 * i, d);
}

// backward: block = 32 channel-lanes (128 channels) x 8 token-lanes; grid (C/128, token blocks).
// dx per element; per-block partial dweight/dbias -> workspace[block_y][10][C].  `g` is the gradient w.r.t. the
// convolution output (the host multiplies by GELU' first when the activation was fused).  The 18 neighbour loads of a
// token (x and g at the nine clamped positions) are unconditional and issued together; positions outside the map are
// skipped in the arithmetic only (the first version loaded under the bounds branches, one load in flight at a time:
// 318 us per [12, 6949, 256] bf16 call).
template <typename T>
__global__ void __launch_bounds__(256) dwconv_bwd_kernel(const T *__restrict__ g_, const T *__restrict__ x,
                                                         const float *__restrict__ weight, T *__restrict__ dx_,
                                                         float *__restrict__ partial, int B, int C, int ntok, Maps mp) {
  __shared__ float red[8][132];
  const int lane = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + lane * 4;
  const bool on = c < C;
  float dw[10][4];
#pragma unroll
  for (int j = 0; j < 10; ++j)
#pragma unroll
    for (int k = 0; k < 4; ++k) dw[j][k] = 0.f;
  float wv[9][4];
#pragma unroll
  for (int j = 0; j < 9; ++j)
#pragma unroll
    for (int k = 0; k < 4; ++k) wv[j][k] = on ? __ldg(weight + (c + k) * 9 + j) : 0.f;

  const int64_t rows = (int64_t)B * ntok;
  for (int64_t r = (int64_t)blockIdx.y * 8 + ty; r < rows && on; r += (int64_t)gridDim.y * 8) {
    const int tok = (int)(r % ntok);
    const int b = (int)(r / ntok);
    const int mi = find_map(mp, tok);
    const int W = mp.w[mi], H = mp.h[mi], t0 = mp.start[mi];
    const int py = (tok - t0) / W, px = (tok - t0) % W;
    const int64_t base = ((int64_t)b * ntok + t0) * C + c;
    float g[4];
    load4(g_ + r * C + c, g);
    // position j = (py + j/3 - 1, px + j%3 - 1): the input neighbour of tap j, and the output pixel that used this
    // token with tap 8 - j
    float xv[9][4], gv[9][4];
    bool ok[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      const int yy = py + j / 3 - 1, xx = px + j % 3 - 1;
      ok[j] = yy >= 0 && yy < H && xx >= 0 && xx < W;
      const int64_t off = base + (int64_t)(min(max(yy, 0), H - 1) * W + min(max(xx, 0), W - 1)) * C;
      load4(x + off, xv[j]);
      load4(g_ + off, gv[j]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) dw[9][k] += g[k];
    float dxv[4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 9; ++j) {      // (same order of accumulation as the branchy version: tap j, then input tap j)
      if (ok[j]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) dw[j][k] += g[k] * xv[j][k];
      }
      if (ok[8 - j]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) dxv[k] += gv[8 - j][k] * wv[j][k];
      }
    }
    store4(dx_ + r * C + c, dxv);
  }
  float *pp = partial + (size_t)blockIdx.y * 10 * C;
  for (int j = 0; j < 10; ++j) {
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) red[ty][lane * 4 + k] = dw[j][k];
    __syncthreads();
    if (threadIdx.x < 128) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
      const int cc = blockIdx.x * 128 + threadIdx.x;
      if (cc < C) pp[(size_t)j * C + cc] = t;
    }
  }
}

// dweight[c*9+j] / dbias[c] (+)= sum over blocks of partial[p][j][c], fixed order
__global__ void __launch_bounds__(256) dwconv_reduce_kernel(const float *__restrict__ partial, int nparts, int C,
                                                            float *__restrict__ dweight, float *__restrict__ dbias,
                                                            int accumulate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 10 * C) return;
  const int j = i / C, c = i % C;
  float t = 0.f;
  for (int p = 0; p < nparts; ++p) t += partial[((size_t)p * 10 + j) * C + c];
  float *dst = j < 9 ? dweight + c * 9 + j : dbias + c;
  if (!dst) return;
  *dst = accumulate ? *dst + t : t;
}

static int make_maps(Maps &mp, int n_maps, const int *hs, const int *ws) {
  ASIS_REQUIRE(n_maps >= 1 && n_maps <= kMaxMaps && hs && ws, "dwconv: 1..%d maps required", kMaxMaps);
  mp.n = n_maps;
  int s = 0;
  for (int i = 0; i < kMaxMaps; ++i) {
    mp.h[i] = i < n_maps ? hs[i] : 1;
    mp.w[i] = i < n_maps ? ws[i] : 1;
    mp.start[i] = s;
    if (i < n_maps) {
      ASIS_REQUIRE(hs[i] > 0 && ws[i] > 0, "dwconv: empty map");
      s += hs[i] * ws[i];
    }
  }
  mp.start[kMaxMaps] = s;
  return ASIS_OK;
}

// token blocks of the backward: one wave of 2 resident blocks (128 registers) on each of the 148 SMs over all channel blocks
static int dwconv_row_blocks(int64_t rows, int C) {
  int64_t rb = (rows + 63) / 64;
  const int cap = std::max(1, 296 / ((C + 127) / 128));
  if (rb > cap) rb = cap;
  if (rb < 1) rb = 1;
  return (int)rb;
}


// ---------------------------------------------------------------------------------------------
// Bilinear 2x upsampling, align_corners=True, channels-last (the four nn.Upsample layers of
// FeatureDecoder, backbones/decoders.py:104-127).  HBM-bound: one thread per (output pixel, 16-byte
// channel vector) forward; the backward is a gather per INPUT pixel over the few output pixels whose
// footprint contains it (no atomics, fixed order).  Source index = dst * (in-1)/(out-1), as ATen's
// area_pixel_compute_source_index(align_corners=True).
// ---------------------------------------------------------------------------------------------
template <typename T> struct Up2Vec;
template <> struct Up2Vec<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void load(const float *p, float (&v)[4]) { load4(p, v); }
  static __device__ __forceinline__ void store(float *p, const float (&v)[4]) { store4(p, v); }
};
template <> struct Up2Vec<bf16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void load(const bf16 *p, float (&v)[8]) {
    const uint4 t = __ldg(reinterpret_cast<const uint4 *>(p));
    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  static __device__ __forceinline__ void store(bf16 *p, const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t *>(&h);
    }
    *reinterpret_cast<uint4 *>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};

struct Up2Src {
  int i0, i1;
  float l;   // weight of i1; 1 - l of i0
};
__device__ __forceinline__ Up2Src up2_src(int o, float scale, int in) {
  const float s = scale * (float)o;
  Up2Src r;
  r.i0 = min((int)s, in - 1);
  r.i1 = r.i0 + (r.i0 < in - 1 ? 1 : 0);
  r.l = s - (float)r.i0;
  return r;
}

// pi / po: storage padding of the input / output maps ([B, H + 2p, W + 2p, C], zeros in the border; 0 = plain)
template <typename T>
__global__ void __launch_bounds__(256) upsample2x_fwd_kernel(const T *__restrict__ x, T *__restrict__ y, int B, int H,
                                                             int W, int C, float sy, float sx, int pi, int po) {
  constexpr int N = Up2Vec<T>::N;
  const int CV = C / N, OH = 2 * H, OW = 2 * W;
  const int Hi = H + 2 * pi, Wi = W + 2 * pi, Hs = OH + 2 * po, Ws = OW + 2 * po;
  const size_t total = (size_t)B * Hs * Ws * CV;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int cv = (int)(t % CV);
    size_t r = t / CV;
    const int ox = (int)(r % Ws) - po;
    r /= Ws;
    const int oy = (int)(r % Hs) - po;
    const int b = (int)(r / Hs);
    float o[N];
#pragma unroll
    for (int i = 0; i < N; ++i) o[i] = 0.f;
    if (oy >= 0 && oy < OH && ox >= 0 && ox < OW) {
      const Up2Src ys = up2_src(oy, sy, H), xs = up2_src(ox, sx, W);
      const T *xb = x + ((size_t)b * Hi * Wi + (size_t)pi * Wi + pi) * C + (size_t)cv * N;
      float v00[N], v01[N], v10[N], v11[N];
      Up2Vec<T>::load(xb + ((size_t)ys.i0 * Wi + xs.i0) * C, v00);
      Up2Vec<T>::load(xb + ((size_t)ys.i0 * Wi + xs.i1) * C, v01);
      Up2Vec<T>::load(xb + ((size_t)ys.i1 * Wi + xs.i0) * C, v10);
      Up2Vec<T>::load(xb + ((size_t)ys.i1 * Wi + xs.i1) * C, v11);
      const float w00 = (1.f - ys.l) * (1.f - xs.l), w01 = (1.f - ys.l) * xs.l, w10 = ys.l * (1.f - xs.l), w11 = ys.l * xs.l;
#pragma unroll
      for (int i = 0; i < N; ++i) o[i] = w00 * v00[i] + w01 * v01[i] + w10 * v10[i] + w11 * v11[i];
    }
    Up2Vec<T>::store(y + t * N, o);
  }
}

// weights with which output index o reads input index i (0 if it does not)
__device__ __forceinline__ float up2_weight(int o, int i, float scale, int in) {
  const Up2Src s = up2_src(o, scale, in);
  return (s.i0 == i ? 1.f - s.l : 0.f) + (s.i1 == i ? s.l : 0.f);
}

template <typename T>
__global__ void __launch_bounds__(256) upsample2x_bwd_kernel(const T *__restrict__ gy, T *__restrict__ gx, int B, int H,
                                                             int W, int C, float sy, float sx, int pi, int po) {
  constexpr int N = Up2Vec<T>::N;
  const int CV = C / N, OH = 2 * H, OW = 2 * W;
  const int Hi = H + 2 * pi, Wi = W + 2 * pi, Hs = OH + 2 * po, Ws = OW + 2 * po;
  const size_t total = (size_t)B * Hi * Wi * CV;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int cv = (int)(t % CV);
    size_t r = t / CV;
    const int ix = (int)(r % Wi) - pi;
    r /= Wi;
    const int iy = (int)(r % Hi) - pi;
    const int b = (int)(r / Hi);
    float acc[N];
#pragma unroll
    for (int i = 0; i < N; ++i) acc[i] = 0.f;
    if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
      // output rows / columns that can touch this input pixel: src in (i - 1, i + 1)  ->  a window of at
      // most 6 around 2 i (scale is just below 1/2); exact membership is decided by up2_weight
      const int oy_lo = max(0, 2 * iy - 3), oy_hi = min(OH - 1, 2 * iy + 4);
      const int ox_lo = max(0, 2 * ix - 3), ox_hi = min(OW - 1, 2 * ix + 4);
      const T *gb = gy + ((size_t)b * Hs * Ws + (size_t)po * Ws + po) * C + (size_t)cv * N;
      for (int oy = oy_lo; oy <= oy_hi; ++oy) {
        const float wy = up2_weight(oy, iy, sy, H);
        if (wy == 0.f) continue;
        for (int ox = ox_lo; ox <= ox_hi; ++ox) {
          const float w = wy * up2_weight(ox, ix, sx, W);
          if (w == 0.f) continue;
          float v[N];
          Up2Vec<T>::load(gb + ((size_t)oy * Ws + ox) * C, v);
#pragma unroll
          for (int i = 0; i < N; ++i) acc[i] = fmaf(w, v[i], acc[i]);
        }
      }
    }
    Up2Vec<T>::store(gx + t * N, acc);
  }
}

}  // namespace asis

using namespace asis;

// ---- input ingest (tools/dataset.py:111-118): uint8 HWC frames -> float CHW / 255, uint8 masks -> int64 ---------------
// one thread per pixel: three coalesced-enough byte reads, three plane-strided float writes (each plane coalesced);
// IEEE division (torch computes uint8 / 255.0 in fp32), so the batch is bit-identical to the host pipeline's tensor
__global__ void __launch_bounds__(256) frames_to_batch_kernel(const uint8_t *__restrict__ frames, float *__restrict__ img,
                                                              const uint8_t *__restrict__ masks, int64_t *__restrict__ target,
                                                              int B, int HW) {
  const size_t total = (size_t)B * HW;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t b = t / HW, p = t - b * HW;
    const uint8_t *src = frames + t * 3;
    float *dst = img + b * 3 * (size_t)HW + p;
#pragma unroll
    for (int c = 0; c < 3; ++c) dst[(size_t)c * HW] = __fdiv_rn((float)src[c], 255.0f);
    if (masks) target[t] = (int64_t)masks[t];
  }
}

extern "C" int asis_frames_to_batch(const uint8_t *frames, float *img, const uint8_t *masks, int64_t *target, int B, int H,
                                    int W, void *stream) {
  ASIS_REQUIRE(frames && img, "frames_to_batch: null pointer");
  ASIS_REQUIRE((masks == nullptr) == (target == nullptr), "frames_to_batch: masks and target go together");
  ASIS_REQUIRE(B > 0 && H > 0 && W > 0, "frames_to_batch: non-positive dimension");
  const size_t total = (size_t)B * H * W;
  const unsigned blocks = (unsigned)std::min<size_t>((total + 255) / 256, (size_t)148 * 16);
  frames_to_batch_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(frames, img, masks, target, B, H * W);
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" int asis_patchify(const float *img, void *cols, int out_dtype, int B, int Cin, int Himg, int Wimg,
                             int patch, int64_t ldk, void *stream) {
  ASIS_REQUIRE(img && cols, "patchify: null pointer");
  ASIS_REQUIRE(dtype_ok(out_dtype), "patchify: bad dtype");
  ASIS_REQUIRE(B > 0 && Cin > 0 && patch > 0, "patchify: non-positive dimension");
  ASIS_REQUIRE(Himg % patch == 0, "Input image height %d is not a multiple of patch height %d", Himg, patch);
  ASIS_REQUIRE(Wimg % patch == 0, "Input image width %d is not a multiple of patch width: %d", Wimg, patch);
  ASIS_REQUIRE(ldk >= (int64_t)Cin * patch * patch, "patchify: ldk too small");
  const int64_t total = (int64_t)B * (Himg / patch) * (Wimg / patch) * ldk;
  const unsigned blocks = (unsigned)((total + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  ASIS_DISPATCH_DTYPE(out_dtype, OT, (patchify_kernel<OT><<<blocks, 256, 0, st>>>(img, (OT *)cols, B, Cin, Himg, Wimg, patch, ldk)));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" int asis_dwconv3x3_forward(const void *x, int dtype, const float *weight, const float *bias, void *pre,
                                      void *y, int B, int C, int n_maps, const int *hs_host, const int *ws_host,
                                      int fuse_gelu, void *stream) {
  ASIS_REQUIRE(x && weight && bias && y, "dwconv_forward: null pointer");
  ASIS_REQUIRE(dtype_ok(dtype), "dwconv_forward: bad dtype");
  ASIS_REQUIRE(B > 0 && C > 0 && C % 4 == 0, "dwconv_forward: C=%d must be a positive multiple of 4", C);
  ASIS_REQUIRE(aligned16(x) && aligned16(y) && aligned16(bias) && (!pre || aligned16(pre)), "dwconv_forward: pointers must be 16-byte aligned");
  Maps mp;
  if (int rc = make_maps(mp, n_maps, hs_host, ws_host)) return rc;
  const int ntok = mp.start[kMaxMaps];
  const int64_t total = (int64_t)B * ntok * (C / 4);
  ASIS_REQUIRE(C <= 1280, "dwconv_forward: C=%d > 1280 (the taps of all channels are staged in 36 C bytes of shared memory)", C);
  const unsigned blocks = (unsigned)((total + 256 * kDwIter - 1) / (256 * kDwIter));
  const size_t smem = (size_t)9 * C * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  ASIS_DISPATCH_DTYPE(dtype, T, (dwconv_fwd_kernel<T><<<blocks, 256, smem, st>>>((const T *)x, weight, bias, (T *)pre, (T *)y, B, C, ntok, mp, fuse_gelu)));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

static size_t dwconv_partial_bytes(int B, int C, int n_tok) {
  return align_up((size_t)dwconv_row_blocks((int64_t)B * n_tok, C) * 10 * C * sizeof(float), 256);
}

// column partials + one [B, n_tok, C] buffer for dy * GELU'(pre) (sized for f32)
extern "C" size_t asis_dwconv3x3_backward_workspace_bytes(int B, int C, int n_tok) {
  return dwconv_partial_bytes(B, C, n_tok) + (size_t)B * n_tok * C * sizeof(float);
}

extern "C" int asis_dwconv3x3_backward(const void *dy, const void *pre, const void *x, int dtype, const float *weight,
                                       void *dx, float *dweight, float *dbias, int accumulate, int B, int C,
                                       int n_maps, const int *hs_host, const int *ws_host, int fuse_gelu,
                                       void *workspace, size_t workspace_bytes, void *stream) {
  ASIS_REQUIRE(dy && x && weight && dx && dweight && dbias && workspace, "dwconv_backward: null pointer");
  ASIS_REQUIRE(!fuse_gelu || pre, "dwconv_backward: fused GELU needs the saved pre-activation");
  ASIS_REQUIRE(dtype_ok(dtype), "dwconv_backward: bad dtype");
  ASIS_REQUIRE(B > 0 && C > 0 && C % 4 == 0, "dwconv_backward: C=%d must be a positive multiple of 4", C);
  // 4-channel vector loads and stores of dy, pre, x, dx and of the GELU' buffer inside the workspace
  ASIS_REQUIRE(aligned16(dy) && aligned16(x) && aligned16(dx) && aligned16(workspace) && (!pre || aligned16(pre)),
               "dwconv_backward: pointers must be 16-byte aligned");
  Maps mp;
  if (int rc = make_maps(mp, n_maps, hs_host, ws_host)) return rc;
  const int ntok = mp.start[kMaxMaps];
  const size_t need = asis_dwconv3x3_backward_workspace_bytes(B, C, ntok);
  if (workspace_bytes < need) ASIS_FAIL(ASIS_ERR_WORKSPACE, "dwconv_backward: workspace %zu < %zu bytes", workspace_bytes, need);
  const int rb = dwconv_row_blocks((int64_t)B * ntok, C);
  dim3 grid((C + 127) / 128, rb);
  cudaStream_t st = (cudaStream_t)stream;
  float *partial = (float *)workspace;
  if (fuse_gelu) {
    void *gbuf = (char *)workspace + dwconv_partial_bytes(B, C, ntok);
    const int64_t n4 = (int64_t)B * ntok * C / 4;
    ASIS_DISPATCH_DTYPE(dtype, T, (dwconv_gelu_grad_kernel<T><<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>((const T *)dy, (const T *)pre, (T *)gbuf, n4)));
    ASIS_LAUNCHED();
    dy = gbuf;
  }
  ASIS_DISPATCH_DTYPE(dtype, T, (dwconv_bwd_kernel<T><<<grid, 256, 0, st>>>((const T *)dy, (const T *)x, weight, (T *)dx, partial, B, C, ntok, mp)));
  ASIS_LAUNCHED();
  dwconv_reduce_kernel<<<(10 * C + 255) / 256, 256, 0, st>>>(partial, rb, C, dweight, dbias, accumulate);
  ASIS_LAUNCHED();
  return ASIS_OK;
}

static int up2_check(const void *a, const void *b, int dtype, int B, int H, int W, int C) {
  ASIS_REQUIRE(a && b, "upsample2x: null pointer");
  ASIS_REQUIRE(dtype_ok(dtype), "upsample2x: bad dtype");
  ASIS_REQUIRE(B > 0 && H > 1 && W > 1 && C > 0, "upsample2x: need B > 0, H > 1, W > 1, C > 0");
  ASIS_REQUIRE(C % (dtype == ASIS_BF16 ? 8 : 4) == 0, "upsample2x: C=%d must be a multiple of %d", C, dtype == ASIS_BF16 ? 8 : 4);
  ASIS_REQUIRE(aligned16(a) && aligned16(b), "upsample2x: pointers must be 16-byte aligned");
  return ASIS_OK;
}

extern "C" int asis_upsample2x_bilinear_forward_padded(const void *x, void *y, int dtype, int B, int H, int W, int C, int pad_in,
                                                       int pad_out, void *stream) {
  if (int rc = up2_check(x, y, dtype, B, H, W, C)) return rc;
  ASIS_REQUIRE(pad_in >= 0 && pad_out >= 0, "upsample2x: negative storage padding");
  const float sy = (float)(H - 1) / (float)(2 * H - 1), sx = (float)(W - 1) / (float)(2 * W - 1);
  const size_t total = (size_t)B * (2 * H + 2 * pad_out) * (2 * W + 2 * pad_out) * (C / (dtype == ASIS_BF16 ? 8 : 4));
  const unsigned blocks = (unsigned)std::min<size_t>((total + 255) / 256, (size_t)148 * 32);
  cudaStream_t st = (cudaStream_t)stream;
  ASIS_DISPATCH_DTYPE(dtype, T, (upsample2x_fwd_kernel<T><<<blocks, 256, 0, st>>>((const T *)x, (T *)y, B, H, W, C, sy, sx, pad_in, pad_out)));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" int asis_upsample2x_bilinear_backward_padded(const void *gy, void *gx, int dtype, int B, int H, int W, int C, int pad_in,
                                                        int pad_out, void *stream) {
  if (int rc = up2_check(gy, gx, dtype, B, H, W, C)) return rc;
  ASIS_REQUIRE(pad_in >= 0 && pad_out >= 0, "upsample2x: negative storage padding");
  const float sy = (float)(H - 1) / (float)(2 * H - 1), sx = (float)(W - 1) / (float)(2 * W - 1);
  const size_t total = (size_t)B * (H + 2 * pad_in) * (W + 2 * pad_in) * (C / (dtype == ASIS_BF16 ? 8 : 4));
  const unsigned blocks = (unsigned)std::min<size_t>((total + 255) / 256, (size_t)148 * 32);
  cudaStream_t st = (cudaStream_t)stream;
  ASIS_DISPATCH_DTYPE(dtype, T, (upsample2x_bwd_kernel<T><<<blocks, 256, 0, st>>>((const T *)gy, (T *)gx, B, H, W, C, sy, sx, pad_in, pad_out)));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

extern "C" int asis_upsample2x_bilinear_forward(const void *x, void *y, int dtype, int B, int H, int W, int C, void *stream) {
  return asis_upsample2x_bilinear_forward_padded(x, y, dtype, B, H, W, C, 0, 0, stream);
}

extern "C" int asis_upsample2x_bilinear_backward(const void *gy, void *gx, int dtype, int B, int H, int W, int C, void *stream) {
  return asis_upsample2x_bilinear_backward_padded(gy, gx, dtype, B, H, W, C, 0, 0, stream);
}
