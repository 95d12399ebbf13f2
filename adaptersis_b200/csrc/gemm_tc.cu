// gemm_tc.cu -- bf16 tensor-core GEMM for sm_100a: C[M,N] = epilogue(sum_k A[m,k] * B[n,k]).
//
// Persistent, warp-specialised kernels; roles by warp id (the SMSP arbiter favours the highest id, so the two
// latency-critical single-warp roles get the top ids):
//   warps 0..7  epilogue       tcgen05.ld -> registers -> per-warp smem transposition -> fused epilogue
//                              (bias / exact GELU (+ derivative) / LayerScale + residual / x aux / accumulate) with
//                              row-contiguous (coalesced) global loads and stores
//   warp 8      TMA producer   cp.async.bulk.tensor -> 128B-swizzled smem ring
//   warp 9      MMA issuer     tcgen05.mma.kind::f16, fp32 accumulators in TMEM (2 x 256 columns, double buffered)
// Three mbarrier pipelines: smem full/empty (TMA <-> MMA), TMEM full/empty (MMA <-> epilogue).
//
// gemm_tc_pair_kernel (every GEMM with M > 128): the two CTAs of a cluster form ONE 256 x 256 tcgen05.mma.cta_group::2
//   tile (6 x 32 KB ring per CTA: its 128 rows of A + half of the B tile); one instantiation per hot
//   (A-major, B-major, epilogue kind, output dtype, saved-branch flag) combination plus an all-in-one fallback;
//   also runs the implicit 3x3 convolutions (gemm_tc_conv3x3: taps as TMA row shifts over zero-padded maps).
// gemm_tc_kernel<A_MN, B_MN> (M <= 128: one M tile): 128 x 256 cta_group::1 tiles, one CTA each (4 x 48 KB ring).
// Tails in M, N and K come for free from TMA zero fill; stores are masked.
//
// Both operands may be K-major (nn.Linear forward: x[R,K], W[N,K]) or MN-major (input gradient:
// W as [K=N_out rows, K_in]; weight gradient: dy[R,N_out] and x[R,K_in], reduction over the rows),
// so no operand is ever transposed in memory.  Weight gradients (few output tiles, very long K)
// are split along K across CTAs and combined with fp32 red.global.add.
#include <mutex>

#define ASIS_WATCHDOG 1   // barrier waits of the GEMM kernels trap after ~2 s instead of spinning forever
#include "epilogue.cuh"
#include "tc_common.cuh"

namespace asis {

using namespace tc;

constexpr int BM = 128, BN = 256, BK = 64, STAGES = 4;
constexpr int A_BYTES = BM * BK * 2;           // 16 KB
constexpr int B_BYTES = BN * BK * 2;           // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES; // 48 KB
constexpr int BOX_BYTES = 64 * BK * 2;         // one 64 x 64 MN-major TMA box: 8 KB
constexpr int NUM_EPI_WARPS = 8;   // (16 epilogue warps measured slower: 96-register cap, spills)
constexpr int GEMM_THREADS = 64 + NUM_EPI_WARPS * 32;
constexpr int EPI_STAGE_BYTES = NUM_EPI_WARPS * 32 * 32 * 4;   // 4 KB transposition buffer per epilogue warp
constexpr int GEMM_SMEM = STAGES * STAGE_BYTES + EPI_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;

struct GemmTcParams {
  int M, N, K;
  int m_tiles, m_groups, n_tiles, splits, kb_per_split, kb_total;
  int atomic_out;  // split-K: combine with red.global.add.f32
  int n_mma;       // pair kernel: N of the MMA instruction (256; 128 / 64 for narrow outputs -- each CTA stages n_mma / 2 rows of B)
  // 3x3 / stride-1 convolution as an implicit GEMM over a zero-padded channels-last map (pair kernel only): the K loop
  // runs over (tap, channel block); tap t reads the A rows shifted by conv_a_row_off[t] (TMA zero-fills rows outside
  // the tensor) -- "im2col by TMA coordinates", no column matrix in memory.
  int conv_taps;           // 0: plain GEMM
  int conv_kpt;            // k-blocks per tap
  int conv_b_k_tap;        // B's K coordinate of (tap, kk) = tap * conv_b_k_tap + kk * BK
  int conv_b_n_tap;        // B's N coordinate shift of tap t = t * conv_b_n_tap
  int conv_wp, conv_sign;  // row shift of tap t = conv_sign * ((t / 3 - 1) * conv_wp + t % 3 - 1)   (conv_wp = W + 2)
  int conv_wg_cin;         // weight gradient of the implicit convolution (MN-major B = x_p, N = 9 Cin): the 64-column box
                           // at N coordinate n belongs to tap n / Cin: it reads channels n % Cin of the rows shifted by that tap
  EpiArgs epi;
};

// ---- epilogue -------------------------------------------------------------------------------------
// tcgen05.ld hands every thread one accumulator ROW (TMEM lane); storing from that layout makes each
// warp store touch 32 different rows with 16 bytes each (32 partial-sector requests per instruction:
// the first version's epilogue was bound by exactly that -- an fp32 output or a second (aux) output
// cost as much as the whole MMA main loop).  So every epilogue warp transposes its 32 x 32 fp32 chunk
// through a private, XOR-swizzled 4 KB smem buffer and then works in a COALESCED layout: lane ->
// (row it*4 + lane/8, 4 columns (lane%8)*4..+3), i.e. 128 contiguous bytes (fp32) / 64 (bf16) per row
// for every global load (residual, aux, C) and store (C, aux).
constexpr int EPI_STAGE_FLOATS = 32 * 32;   // per warp

__device__ __forceinline__ void load4_any(const void *base, int dtype, size_t idx, float (&v)[4]) {
  if (dtype == ASIS_F32) {
    const float4 t = *reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(base) + idx);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
    const uint2 t = *reinterpret_cast<const uint2 *>(reinterpret_cast<const bf16 *>(base) + idx);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162 *>(&t.x);
    const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162 *>(&t.y);
    v[0] = __low2float(a); v[1] = __high2float(a); v[2] = __low2float(b); v[3] = __high2float(b);
  }
}
__device__ __forceinline__ void store4_any(void *base, int dtype, size_t idx, const float (&v)[4]) {
  if (dtype == ASIS_F32) store4(reinterpret_cast<float *>(base) + idx, v);
  else store4(reinterpret_cast<bf16 *>(base) + idx, v);
}

// raw 16-byte (fp32 x4) or 8-byte (bf16 x4) global load kept undecoded, so that nothing depends on
// the load until the values are used one chunk later
__device__ __forceinline__ uint4 ldraw4(const void *base, int dtype, size_t idx) {
  if (dtype == ASIS_F32) return *reinterpret_cast<const uint4 *>(reinterpret_cast<const float *>(base) + idx);
  const uint2 t = *reinterpret_cast<const uint2 *>(reinterpret_cast<const bf16 *>(base) + idx);
  return make_uint4(t.x, t.y, 0u, 0u);
}
__device__ __forceinline__ void decode4(const uint4 &r, int dtype, float (&v)[4]) {
  if (dtype == ASIS_F32) {
    v[0] = __uint_as_float(r.x); v[1] = __uint_as_float(r.y); v[2] = __uint_as_float(r.z); v[3] = __uint_as_float(r.w);
  } else {
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162 *>(&r.x);
    const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162 *>(&r.y);
    v[0] = __low2float(a); v[1] = __high2float(a); v[2] = __low2float(b); v[3] = __high2float(b);
  }
}

// which epilogues read a second [M, N] operand (the residual, the saved pre-activation, or C itself)
template <int KIND> struct EpiReads { static constexpr bool value = KIND == ASIS_EPI_SCALE_RESIDUAL || KIND == ASIS_EPI_DGELU || KIND == ASIS_EPI_ACCUMULATE || KIND == ASIS_EPI_MUL_AUX; };

// the 4-column group of one row in the coalesced layout, vector path (col + 4 <= N, 16-byte aligned
// pitches, no split-K); KIND is a compile-time constant; `pre` is the prefetched second operand
template <int KIND>
__device__ __forceinline__ void epi_group4(const EpiArgs &e, int row, int col, float (&v)[4], const float (&b4)[4],
                                           const float (&g4)[4], const uint4 &pre) {
  const size_t ci = (size_t)row * e.ldc + col;
  const size_t ai = (size_t)row * e.ldaux + col;
  if (KIND != ASIS_EPI_DGELU && KIND != ASIS_EPI_ACCUMULATE && KIND != ASIS_EPI_MUL_AUX) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] += b4[i];
  }
  if (KIND == ASIS_EPI_GELU_GRAD) {
    float d[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = gelu_and_grad_fast(v[i], d[i]);
    store4_any(e.aux, e.aux_dtype, ai, d);
  } else if (KIND == ASIS_EPI_MUL_AUX) {
    float h[4];
    decode4(pre, e.aux_dtype, h);
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] *= h[i];
  } else if (KIND == ASIS_EPI_GELU) {
    if (e.aux) store4_any(e.aux, e.aux_dtype, ai, v);
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = gelu_fast(v[i]);
  } else if (KIND == ASIS_EPI_SCALE_RESIDUAL) {
    if (e.aux) store4_any(e.aux, e.aux_dtype, ai, v);
    float r[4];
    decode4(pre, ASIS_F32, r);
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = fmaf(g4[i], v[i], r[i]);
  } else if (KIND == ASIS_EPI_DGELU) {
    float h[4];
    decode4(pre, e.aux_dtype, h);
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] *= dgelu_fast(h[i]);
  } else if (KIND == ASIS_EPI_ACCUMULATE) {
    float c[4];
    decode4(pre, ASIS_F32, c);
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] += c[i];
  }
  store4_any(e.C, e.c_dtype, ci, v);
}

// everything else (N tails, unaligned pitches, split-K reduction): rolled loops, so that the hot
// path above stays small (fully unrolled and inlined 32x, the generic path quadrupled the code size
// and the epilogue warps stalled on instruction fetch)
__device__ __forceinline__ void epi_group4_slow(const GemmTcParams &p, int row, int col, const float4 &t, bool vec_ok) {
  const EpiArgs &e = p.epi;
  if (p.atomic_out && vec_ok && col + 4 <= p.N) {
    atomicAdd(reinterpret_cast<float4 *>(reinterpret_cast<float *>(e.C) + (size_t)row * e.ldc + col), t);
    return;
  }
#pragma unroll 1
  for (int j = 0; j < 4; ++j) {
    const float vj = j == 0 ? t.x : j == 1 ? t.y : j == 2 ? t.z : t.w;
    if (col + j < p.N) {
      if (p.atomic_out) atomicAdd(reinterpret_cast<float *>(e.C) + (size_t)row * e.ldc + col + j, vj);
      else epi_scalar(e, row, col + j, vj);
    }
  }
}

// prefetch the 8 row groups of chunk c (this lane's 4 columns) of the epilogue's second operand.
// The compiler may not hoist these loads above earlier stores (possible aliasing), so without the
// explicit software pipeline every one of the 32 (chunk, row group) steps of a tile waited a full
// global-memory round trip: the residual / GELU' epilogues cost 2-3x the MMA main loop.
template <int KIND>
__device__ __forceinline__ void epi_prefetch(const GemmTcParams &p, int row0, int col, int r, bool vec_ok, uint4 (&pre)[8]) {
  if (!EpiReads<KIND>::value) return;
  const EpiArgs &e = p.epi;
  if (!vec_ok || p.atomic_out || col + 4 > p.N) return;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int row = row0 + it * 4 + r;
    if (row < p.M) {
      if (KIND == ASIS_EPI_SCALE_RESIDUAL) pre[it] = ldraw4(e.residual, ASIS_F32, (size_t)row * e.ldc + col);
      else if (KIND == ASIS_EPI_DGELU || KIND == ASIS_EPI_MUL_AUX) pre[it] = ldraw4(e.aux, e.aux_dtype, (size_t)row * e.ldaux + col);
      else pre[it] = ldraw4(e.C, ASIS_F32, (size_t)row * e.ldc + col);
    }
  }
}

#ifdef ASIS_TRACE
__device__ unsigned long long *g_gemm_trace = nullptr;     // [9 slots][256 tiles] clock64 stamps of cluster 0's leader CTA
#define GEMM_TRACE(slot, idx)                                                                          \
  do {                                                                                                 \
    if (g_gemm_trace && blockIdx.x == 0 && lane == 0 && (idx) < 256) g_gemm_trace[(slot) * 256 + (idx)] = clock64(); \
  } while (0)
#else
#define GEMM_TRACE(slot, idx) do { } while (0)
#endif

// the epilogue of one 32-row x 128-column slab owned by one warp
template <int KIND>
__device__ __forceinline__ void epi_slab(const GemmTcParams &p, uint32_t taddr, float *stage, int row0, int col_base,
                                         bool vec_ok, int lane, uint64_t *tfull, uint32_t tfull_phase, int tr_idx = -1) {
  const EpiArgs &e = p.epi;
  const int cg = lane & 7, r = lane >> 3;
  (void)tr_idx;
  uint4 pre[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) pre[i] = make_uint4(0u, 0u, 0u, 0u);
  epi_prefetch<KIND>(p, row0, col_base + cg * 4, r, vec_ok, pre);   // in flight while the MMAs of this tile finish
  if (tr_idx >= 0) GEMM_TRACE(3, tr_idx);
  mbar_wait(tfull, tfull_phase);
  tc_fence_after();
  if (tr_idx >= 0) GEMM_TRACE(4, tr_idx);
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    float v[32];
    tmem_ld32_issue(taddr + c * 32, v);
    tmem_ld_wait();
    // thread = row  ->  smem, 16-byte groups XOR-swizzled by the row (conflict-free both ways)
#pragma unroll
    for (int g = 0; g < 8; ++g)
      *reinterpret_cast<float4 *>(stage + lane * 32 + ((g ^ (lane & 7)) << 2)) = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
    __syncwarp();
    const int col = col_base + c * 32 + cg * 4;
    uint4 cur[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) cur[i] = pre[i];
    if (c + 1 < 4) epi_prefetch<KIND>(p, row0, col + 32, r, vec_ok, pre);
    if (col < p.N) {
      float b4[4] = {0.f, 0.f, 0.f, 0.f}, g4[4] = {0.f, 0.f, 0.f, 0.f};
      if (KIND != ASIS_EPI_DGELU && KIND != ASIS_EPI_ACCUMULATE && KIND != ASIS_EPI_MUL_AUX && e.bias) {
#pragma unroll
        for (int i = 0; i < 4; ++i) b4[i] = (col + i < p.N) ? __ldg(e.bias + col + i) : 0.f;
      }
      if (KIND == ASIS_EPI_SCALE_RESIDUAL) {
#pragma unroll
        for (int i = 0; i < 4; ++i) g4[i] = (col + i < p.N) ? __ldg(e.gamma + col + i) : 0.f;
      }
      const bool fast = vec_ok && !p.atomic_out && col + 4 <= p.N;
      if (fast) {
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int rl = it * 4 + r;
          const float4 t = *reinterpret_cast<const float4 *>(stage + rl * 32 + ((cg ^ (rl & 7)) << 2));
          float w[4] = {t.x, t.y, t.z, t.w};
          if (row0 + rl < p.M) epi_group4<KIND>(e, row0 + rl, col, w, b4, g4, cur[it]);
        }
      } else {
#pragma unroll 1
        for (int it = 0; it < 8; ++it) {
          const int rl = it * 4 + r;
          const float4 t = *reinterpret_cast<const float4 *>(stage + rl * 32 + ((cg ^ (rl & 7)) << 2));
          if (row0 + rl < p.M) epi_group4_slow(p, row0 + rl, col, t, vec_ok);
        }
      }
    }
    __syncwarp();
  }
}

// ---- lean slab epilogue (CTA-pair kernel) ------------------------------------------------------------
// A timeline of the first pair kernel (tools/gemm_trace.py, profiles/r2_gemm_trace.md) showed the epilogue, not the
// MMA main loop, setting the tile period: 8.0 k clk per 128 x 256 tile for the plain bias epilogue, 12.4 k / 13.9 k for
// GELU without / with the saved pre-activation, against 8.3-9.6 k clk of MMAs.  Software-pipelining the chunks (TMEM
// load of chunk c+1 under chunk c, alternating transposition buffers) changed nothing, and the SASS said why: ~25
// instructions per output element, most of them 64-bit address arithmetic ((size_t)row * ld + col redone for every
// 4-element group of every operand), run-time dtype selects, per-element bounds predicates and generic-space LD/ST
// for the transposition buffer -- the epilogue warps were ISSUE bound.  This version keeps the pipelining and
//   * takes the output dtype as a template parameter and assumes bf16 for the optional aux operand,
//   * handles only slabs that lie inside N with 16-byte-aligned pitches (everything else, and split-K, goes to
//     the generic epi_slab), so no column predicates,
//   * carries one byte pointer per operand per lane and reaches row group `it` with one IMAD.WIDE,
//   * replaces the per-row M predicate by a per-lane count of valid row groups,
//   * uses 32-bit shared-window addresses (ld/st.shared) whose swizzle is folded into two per-lane bases.
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ uint2 pack_bf16x4(const float (&v)[4]) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
  __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
  return make_uint2(*reinterpret_cast<uint32_t *>(&a), *reinterpret_cast<uint32_t *>(&b));
}

template <int KIND> struct EpiHasBias { static constexpr bool value = KIND != ASIS_EPI_DGELU && KIND != ASIS_EPI_ACCUMULATE && KIND != ASIS_EPI_MUL_AUX; };

// state of one lane for one slab: byte pointers at (its first row, its 4 columns of the current chunk)
struct EpiLane {
  char *c;               // output
  char *aux;             // GELU / SCALE_RESIDUAL: optional bf16 output (null: none)
  const char *in2;       // SCALE_RESIDUAL: residual f32; DGELU: saved pre-activation bf16; ACCUMULATE: C f32
  uint32_t cstep, astep, istep;   // bytes between row groups (4 rows)
  int nit;               // valid row groups of this lane (rows < M)
};

template <int KIND>
__device__ __forceinline__ void epi3_prefetch(const EpiLane &L, uint4 (&pre)[8]) {
  if (!EpiReads<KIND>::value) return;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    if (it < L.nit) {
      const char *q = L.in2 + (size_t)((uint32_t)it * L.istep);
      if (KIND == ASIS_EPI_DGELU || KIND == ASIS_EPI_MUL_AUX) {
        const uint2 t = *reinterpret_cast<const uint2 *>(q);
        pre[it] = make_uint4(t.x, t.y, 0u, 0u);
      } else {
        pre[it] = *reinterpret_cast<const uint4 *>(q);
      }
    }
  }
}

template <int KIND>
__device__ __forceinline__ void epi3_colvec(const GemmTcParams &p, int col, float4 &b4, float4 &g4) {
  const EpiArgs &e = p.epi;
  b4 = g4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (EpiHasBias<KIND>::value && e.bias) b4 = __ldg(reinterpret_cast<const float4 *>(e.bias + col));
  if (KIND == ASIS_EPI_SCALE_RESIDUAL) g4 = __ldg(reinterpret_cast<const float4 *>(e.gamma + col));
}

// one transposed 32 x 32 chunk read back as lane -> (row it*4 + lane/8, 4 columns): fused math, coalesced stores
// SAUX (SCALE_RESIDUAL only): the branch output is saved as well -- a compile-time flag, each variant in its own kernel
template <int KIND, bool CBF16, bool SAUX>
__device__ __forceinline__ void epi3_chunk(const EpiLane &L, uint32_t rd0, uint32_t rd1, const float4 &b4, const float4 &g4,
                                           const uint4 (&cur)[8]) {
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    if (it < L.nit) {
      const float4 t = lds128(((it & 1) ? rd1 : rd0) + it * 512);
      float w[4] = {t.x, t.y, t.z, t.w};
      if (EpiHasBias<KIND>::value) { w[0] += b4.x; w[1] += b4.y; w[2] += b4.z; w[3] += b4.w; }
      if (KIND == ASIS_EPI_SCALE_RESIDUAL && SAUX)
        *reinterpret_cast<uint2 *>(L.aux + (size_t)((uint32_t)it * L.astep)) = pack_bf16x4(w);
      if (KIND == ASIS_EPI_GELU) {
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = gelu_fast(w[i]);
      } else if (KIND == ASIS_EPI_GELU_GRAD) {
        float d[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = gelu_and_grad_fast(w[i], d[i]);
        *reinterpret_cast<uint2 *>(L.aux + (size_t)((uint32_t)it * L.astep)) = pack_bf16x4(d);
      } else if (KIND == ASIS_EPI_MUL_AUX) {
        const __nv_bfloat162 ha = *reinterpret_cast<const __nv_bfloat162 *>(&cur[it].x);
        const __nv_bfloat162 hb = *reinterpret_cast<const __nv_bfloat162 *>(&cur[it].y);
        w[0] *= __low2float(ha); w[1] *= __high2float(ha); w[2] *= __low2float(hb); w[3] *= __high2float(hb);
      } else if (KIND == ASIS_EPI_SCALE_RESIDUAL) {
        w[0] = fmaf(g4.x, w[0], __uint_as_float(cur[it].x)); w[1] = fmaf(g4.y, w[1], __uint_as_float(cur[it].y));
        w[2] = fmaf(g4.z, w[2], __uint_as_float(cur[it].z)); w[3] = fmaf(g4.w, w[3], __uint_as_float(cur[it].w));
      } else if (KIND == ASIS_EPI_DGELU) {
        const __nv_bfloat162 ha = *reinterpret_cast<const __nv_bfloat162 *>(&cur[it].x);
        const __nv_bfloat162 hb = *reinterpret_cast<const __nv_bfloat162 *>(&cur[it].y);
        w[0] *= dgelu_fast(__low2float(ha)); w[1] *= dgelu_fast(__high2float(ha));
        w[2] *= dgelu_fast(__low2float(hb)); w[3] *= dgelu_fast(__high2float(hb));
      } else if (KIND == ASIS_EPI_ACCUMULATE) {
        w[0] += __uint_as_float(cur[it].x); w[1] += __uint_as_float(cur[it].y);
        w[2] += __uint_as_float(cur[it].z); w[3] += __uint_as_float(cur[it].w);
      }
      char *q = L.c + (size_t)((uint32_t)it * L.cstep);
      if (CBF16) *reinterpret_cast<uint2 *>(q) = pack_bf16x4(w);
      else *reinterpret_cast<float4 *>(q) = make_float4(w[0], w[1], w[2], w[3]);
    }
  }
}

// the epilogue of one 32-row x 128-column slab (entirely inside N) owned by one warp; `stage_u32`: its 4 KB buffer
// `nch`: how many of the slab's four 32-column chunks lie inside N (a narrow GEMM -- N = 64 convolutions -- uses 2 or 0)
// FULL: all four chunks, known at compile time (the hot instantiation: every loop bound and `last` are constants)
template <int KIND, bool CBF16, bool FULL, bool SAUX = false>
__device__ __forceinline__ void epi_slab3(const GemmTcParams &p, uint32_t taddr, uint32_t stage_u32, int row0, int col_base,
                                          int lane, uint64_t *tfull, uint32_t tfull_phase, int tr_idx, int nch_rt) {
  const int nch = FULL ? 4 : nch_rt;
  const EpiArgs &e = p.epi;
  const int cg = lane & 7, r = lane >> 3;
  (void)tr_idx;
  constexpr uint32_t CE = CBF16 ? 2 : 4;
  int col = col_base + cg * 4;
  EpiLane L;
  {
    const size_t eoff = (size_t)(row0 + r) * e.ldc + col;
    L.c = reinterpret_cast<char *>(e.C) + eoff * CE;
    L.cstep = (uint32_t)(4 * e.ldc) * CE;
    const int left = p.M - row0 - r;
    L.nit = left <= 0 ? 0 : (left + 3 >= 32 ? 8 : (left + 3) >> 2);
    L.aux = nullptr;
    L.astep = (uint32_t)(4 * e.ldaux) * 2u;
    L.in2 = nullptr;
    L.istep = 0;
    if (((KIND == ASIS_EPI_SCALE_RESIDUAL && SAUX) || KIND == ASIS_EPI_GELU_GRAD) && e.aux)      // (GELU + saved pre-activation: generic path)
      L.aux = reinterpret_cast<char *>(e.aux) + ((size_t)(row0 + r) * e.ldaux + col) * 2;
    if (KIND == ASIS_EPI_SCALE_RESIDUAL) {
      L.in2 = reinterpret_cast<const char *>(e.residual) + eoff * 4;
      L.istep = (uint32_t)(4 * e.ldc) * 4u;
    } else if (KIND == ASIS_EPI_ACCUMULATE) {
      L.in2 = reinterpret_cast<const char *>(e.C) + eoff * 4;
      L.istep = (uint32_t)(4 * e.ldc) * 4u;
    } else if (KIND == ASIS_EPI_DGELU || KIND == ASIS_EPI_MUL_AUX) {
      L.in2 = reinterpret_cast<const char *>(e.aux) + ((size_t)(row0 + r) * e.ldaux + col) * 2;
      L.istep = L.astep;
    }
  }
  constexpr uint32_t I2E = (KIND == ASIS_EPI_DGELU || KIND == ASIS_EPI_MUL_AUX) ? 2 : 4;       // element size of the second operand
  // transposition buffers: write side (thread = row `lane`), read side (row it*4 + r, 16-byte group cg)
  const uint32_t wrA = stage_u32 + lane * 128 + ((lane & 7) << 4);
  const uint32_t rdA0 = stage_u32 + r * 128 + ((cg ^ r) << 4), rdA1 = stage_u32 + r * 128 + ((cg ^ (r + 4)) << 4);
  uint4 pre[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) pre[i] = make_uint4(0u, 0u, 0u, 0u);
  float4 b4n = make_float4(0.f, 0.f, 0.f, 0.f), g4n = b4n;
  if (nch > 0) {
    epi3_colvec<KIND>(p, col, b4n, g4n);                  // chunk 0's columns
    epi3_prefetch<KIND>(L, pre);                          // in flight while the MMAs of this tile finish
    // chunks 1..3 of the second operand (residual / saved derivative): pulled into L2 now, while this warp only waits
    // for the MMAs -- their register loads are issued one chunk (~300 clk) ahead, far less than a DRAM round trip, and
    // with K = 1024 the epilogue, not the MMA loop, sets the tile period.  One lane per 128-byte line.
    if (EpiReads<KIND>::value && KIND != ASIS_EPI_ACCUMULATE) {
      constexpr uint32_t I2Ep = (KIND == ASIS_EPI_DGELU || KIND == ASIS_EPI_MUL_AUX) ? 2 : 4;
      if (I2Ep == 4 || (cg & 1) == 0) {                   // f32: 8 lanes = one 128 B line per chunk; bf16: 64 B per chunk
#pragma unroll
        for (int c = 1; c < 4; ++c) {
          if (I2Ep == 4 && cg != 0) break;
          if (I2Ep == 2 && (cg != 0 || (c & 1) == 0)) continue;       // bf16: chunks 2c, 2c+1 share a line: prefetch once
#pragma unroll
          for (int it = 0; it < 8; ++it)
            if (it < L.nit)
              asm volatile("prefetch.global.L2 [%0];" ::"l"(L.in2 + (size_t)((uint32_t)it * L.istep) + c * 32 * I2Ep));
        }
      }
    }
  }
  if (tr_idx >= 0) GEMM_TRACE(3, tr_idx);
  mbar_wait(tfull, tfull_phase);
  tc_fence_after();
  if (tr_idx >= 0) GEMM_TRACE(4, tr_idx);
  if (nch <= 0) return;                     // (the wait above keeps this warp in step with the accumulator phases)
  float va[32], vb[32];
  tmem_ld32_issue(taddr, va);
#pragma unroll 1
  for (int c2 = 0; c2 < 2; ++c2) {
    if (2 * c2 >= nch) break;
#pragma unroll
    for (int h = 0; h < 2; ++h) {           // h = 0: registers va;  h = 1: registers vb
      if (2 * c2 + h >= nch) break;
      const bool last = (2 * c2 + h + 1 >= nch);
      tmem_ld_wait();
      if (!last) {
        if (h == 0) tmem_ld32_issue(taddr + (2 * c2 + 1) * 32, vb);
        else tmem_ld32_issue(taddr + 2 * 32, va);
      }
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const float *v = h == 0 ? va : vb;
        sts128(wrA ^ (g << 4), v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
      }
      __syncwarp();
      const float4 b4 = b4n, g4 = g4n;
      uint4 cur[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) cur[i] = pre[i];
      if (!last) {                          // next chunk's column vectors and second operand, under this chunk's math
        epi3_colvec<KIND>(p, col + 32, b4n, g4n);
        L.in2 += EpiReads<KIND>::value ? 32 * I2E : 0;
        epi3_prefetch<KIND>(L, pre);
      }
      epi3_chunk<KIND, CBF16, SAUX>(L, rdA0, rdA1, b4, g4, cur);
      __syncwarp();                         // the buffer is rewritten by the next chunk
      L.c += 32 * CE;
      if (KIND == ASIS_EPI_GELU_GRAD || SAUX) L.aux += 32 * 2;
      col += 32;
    }
  }
}

// ---- 1-CTA kernel (tcgen05.mma.cta_group::1), GEMMs with M <= 128 -------------------------------------------
// One 128 x 256 tile per CTA (4 x 48 KB ring).  With a single M tile the pair kernel would spend its second CTA on zero
// rows: on the step's M <= 128 weight gradients it measured 0-8 % slower than this kernel (DESIGN.md section 5.2).
template <int A_MN, int B_MN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float *epi_stage = reinterpret_cast<float *>(smem + STAGES * STAGE_BYTES);
  uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + STAGES * STAGE_BYTES + EPI_STAGE_BYTES);
  uint64_t *empty_bar = full_bar + STAGES;
  uint64_t *tfull_bar = empty_bar + STAGES;
  uint64_t *tempty_bar = tfull_bar + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int TMA_WARP = NUM_EPI_WARPS, MMA_WARP = NUM_EPI_WARPS + 1;

  if (warp == TMA_WARP && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar + a, 1);
      mbar_init(tempty_bar + a, NUM_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int total_tiles = p.m_groups * p.n_tiles * p.splits;

  // (warp-uniform producer and MMA roles: see the pair kernel)
  if (warp == TMA_WARP) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int m_blk = tile % p.m_groups;
      const int rest = tile / p.m_groups;
      const int n_blk = rest % p.n_tiles;
      const int split = rest / p.n_tiles;
      const int kb0 = split * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty_bar + stage, phase ^ 1);
        if (lane == 0) {
          uint8_t *sa = smem + stage * STAGE_BYTES;
          uint8_t *sb = sa + A_BYTES;
          mbar_arrive_expect_tx(full_bar + stage, STAGE_BYTES);
          if (A_MN == 0) {
            tma_load_2d(&tmA, full_bar + stage, sa, kb * BK, m_blk * BM);
          } else {
#pragma unroll
            for (int j = 0; j < BM / 64; ++j)
              tma_load_2d(&tmA, full_bar + stage, sa + j * BOX_BYTES, m_blk * BM + j * 64, kb * BK);
          }
          if (B_MN == 0) {
            tma_load_2d(&tmB, full_bar + stage, sb, kb * BK, n_blk * BN);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 64; ++j)
              tma_load_2d(&tmB, full_bar + stage, sb + j * BOX_BYTES, n_blk * BN + j * 64, kb * BK);
          }
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == MMA_WARP) {
    constexpr uint32_t idesc = make_idesc(BM, BN, A_MN, B_MN);
    const uint32_t smem_base = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int split = (tile / p.m_groups) / p.n_tiles;
      const int kb0 = split * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      mbar_wait(tempty_bar + acc, acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(full_bar + stage, phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint32_t sb = sa + A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t da = A_MN == 0 ? smem_desc(sa + k * 32, 16, 1024) : smem_desc(sa + k * 2048, BOX_BYTES, 1024);
            const uint64_t db = B_MN == 0 ? smem_desc(sb + k * 32, 16, 1024) : smem_desc(sb + k * 2048, BOX_BYTES, 1024);
            umma_bf16(d_tmem, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(empty_bar + stage);                    // frees the smem stage when the MMAs above have read it
          if (kb == kb1 - 1) umma_commit(tfull_bar + acc);  // accumulator complete
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else {
    const int ew = warp;               // 0..7
    const int quarter = warp & 3;      // TMEM lane quarter this warp may access
    const int half = ew >> 2;          // column half: [half*128, half*128+128)
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool vec_ok = (p.epi.ldc % 4 == 0) && (!p.epi.aux || p.epi.ldaux % 4 == 0);
    float *stage = epi_stage + ew * EPI_STAGE_FLOATS;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int m_blk = tile % p.m_groups;
      const int n_blk = (tile / p.m_groups) % p.n_tiles;
      const int row0 = m_blk * BM + quarter * 32;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + half * 128;
      const int col_base = n_blk * BN + half * 128;
      switch (p.epi.kind) {
        case ASIS_EPI_GELU: epi_slab<ASIS_EPI_GELU>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase); break;
        case ASIS_EPI_SCALE_RESIDUAL: epi_slab<ASIS_EPI_SCALE_RESIDUAL>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase); break;
        case ASIS_EPI_DGELU: epi_slab<ASIS_EPI_DGELU>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase); break;
        case ASIS_EPI_ACCUMULATE: epi_slab<ASIS_EPI_ACCUMULATE>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase); break;
        case ASIS_EPI_GELU_GRAD: epi_slab<ASIS_EPI_GELU_GRAD>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase); break;
        case ASIS_EPI_MUL_AUX: epi_slab<ASIS_EPI_MUL_AUX>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase); break;
        default: epi_slab<ASIS_EPI_NONE>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase); break;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar + acc);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---- CTA-pair kernel (tcgen05.mma.cta_group::2) ----------------------------------------------------
// The two CTAs of a cluster form ONE 256 x 256 MMA: each CTA stages its own 128 rows of A and HALF of the B tile (128 of
// the 256 n-rows); the leader (cluster rank 0) issues every instruction for both tensor cores, which read the other half
// of B from the peer's shared memory.  Per CTA and k-block that is 32 KB filled + 32 KB read instead of the 48 + 48 of a
// 128 x 256 cta_group::1 tile (whose tensor core reads the whole B tile even when clusters share it by TMA multicast):
// the 128 B/clk shared-memory port is what this relieves (TMA fill 96 B/clk + operand reads 96 B/clk at full MMA rate
// with 1-CTA tiles).  With M <= 128 the peer's A rows are TMA zero fill.  Ring: 6 x 32 KB (the timeline showed the
// producer only ~2 k clk ahead of the MMAs with 5 stages, about one L2 round trip: the first k-block of a tile arrived
// late).
// Protocol (as in DeepGEMM's sm_100 kernels): both producers report their TMA bytes to the LEADER's full barrier
// (cp.async.bulk.tensor.cta_group::2 with a shared::cluster barrier address; arrival count 2 = leader's
// arrive.expect_tx + the peer's plain arrive); tcgen05.commit.cta_group::2 multicasts "stage free" / "accumulator
// complete" to both CTAs; the epilogue warps of both CTAs release the accumulator on the leader's barrier.
constexpr int STAGES2 = 6;
constexpr int B2_BYTES = (BN / 2) * BK * 2;           // 16 KB: this CTA's half of the B tile
constexpr int STAGE2_BYTES = A_BYTES + B2_BYTES;      // 32 KB
constexpr int GEMM2_SMEM = STAGES2 * STAGE2_BYTES + EPI_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
static_assert(GEMM2_SMEM <= 227 * 1024, "pair kernel: shared memory over the 227 KB limit");

// EPI: -1 = every epilogue kind behind a run-time switch (any combination the C ABI allows); >= 0 = the kernel is compiled
// for that ONE kind (the switch collapses): the hot (majors, kind) pairs of the step each get their own kernel.  With all
// fourteen epilogue bodies (7 lean + 7 generic) in one kernel the code was ~23 k SASS lines and the register allocation
// the union of all of them -- removing one `if (aux)` store from the lean GELU body alone made that call 20 % faster.
// CDT: output dtype fixed at compile time (0 f32, 1 bf16, -1 run time); AUX: SCALE_RESIDUAL's saved branch output
// (1 present, 0 absent, -1 run time).
template <int A_MN, int B_MN, int EPI, int CDT, int AUX>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float *epi_stage = reinterpret_cast<float *>(smem + STAGES2 * STAGE2_BYTES);
  uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + STAGES2 * STAGE2_BYTES + EPI_STAGE_BYTES);
  uint64_t *empty_bar = full_bar + STAGES2;
  uint64_t *tfull_bar = empty_bar + STAGES2;
  uint64_t *tempty_bar = tfull_bar + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int TMA_WARP = NUM_EPI_WARPS, MMA_WARP = NUM_EPI_WARPS + 1;
  const int crank = (int)cluster_ctarank();
  const bool leader = crank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (warp == TMA_WARP && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES2; ++s) {
      mbar_init(full_bar + s, 2);       // (used in the leader) its own arrive.expect_tx + the peer's arrive
      mbar_init(empty_bar + s, 1);      // one multicast commit per use
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar + a, 1);                    // one multicast commit per tile
      mbar_init(tempty_bar + a, 2 * NUM_EPI_WARPS);   // (used in the leader) the epilogue warps of both CTAs
    }
    fence_barrier_init();
  }
  // Each CTA allocates ALL 512 columns of its own tensor memory (cta_group::1): the base
  // address is then 0 in both CTAs of the pair, which is the symmetric layout cta_group::2 MMAs address.
  if (warp == MMA_WARP) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int total_tiles = p.m_groups * p.n_tiles * p.splits;   // per pair: two adjacent m-tiles, one n-tile

  // Producer and MMA roles run WARP-UNIFORMLY (all 32 lanes execute the loops and the barrier waits;
  // only the TMA / tcgen05 instructions themselves sit under elect_one).  With the whole role under
  // `if (lane == 0)` the loop state lives in per-thread registers and every TMA / MMA operand has
  // to be moved to uniform registers through an ELECT / R2UR.BROADCAST waterfall loop: the MMA
  // thread then needs ~100 issue cycles per 128-cycle MMA and the tensor pipe starves.
  if (warp == TMA_WARP) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = cluster_id; tile < total_tiles; tile += num_clusters) {
      // N fastest: the n-tiles of one pair of m-tiles run on neighbouring clusters at the same time, so an A tile
      // (activations, streamed once) is fetched from HBM once and hit in L2 by the others; the B operand (weights,
      // a few MB) is L2-resident anyway.  With M fastest a K = 4096, N = 1024 GEMM re-read its 173 MB A operand from
      // HBM once per n-tile.
      const int n_blk = tile % p.n_tiles;
      const int rest = tile / p.n_tiles;
      const int m_blk = (rest % p.m_groups) * 2 + crank;
      const int split = rest / p.m_groups;
      const int kb0 = split * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      const int n0 = n_blk * BN + crank * (p.n_mma / 2);       // this CTA's half of the B tile
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty_bar + stage, phase ^ 1);
        if (kb == kb0) GEMM_TRACE(5, tile / num_clusters);
        if (kb == kb1 - 1) GEMM_TRACE(6, tile / num_clusters);
        if (lane == 0) {
          uint8_t *sa = smem + stage * STAGE2_BYTES;
          uint8_t *sb = sa + A_BYTES;
          const uint32_t lfull = mapa_u32(full_bar + stage, 0);   // the leader's barrier for this stage
          // both CTAs' A tile + their B slices: n_mma / 2 rows (K-major box) or n_mma / 128 64-column boxes (MN-major) --
          // a narrow output loads (and zero-fills) only the B rows its MMA reads
          if (leader) mbar_arrive_expect_tx_cluster(lfull, 2 * (A_BYTES + (p.n_mma / 2) * BK * 2));
          else mbar_arrive_cluster(lfull);
          int a_k = kb * BK, a_row = m_blk * BM, b_k = kb * BK, b_n = n0;
          if (p.conv_taps) {                 // implicit 3x3 convolution: (tap, channel block) of this k-block
            const int tap = kb / p.conv_kpt, kk = kb - tap * p.conv_kpt;
            a_k = kk * BK;
            a_row += p.conv_sign * ((tap / 3 - 1) * p.conv_wp + (tap % 3 - 1));
            b_k = tap * p.conv_b_k_tap + kk * BK;
            b_n += tap * p.conv_b_n_tap;
          }
          if (A_MN == 0) {
            tma_load_2d_pair(&tmA, lfull, sa, a_k, a_row);
          } else {
#pragma unroll
            for (int j = 0; j < BM / 64; ++j) tma_load_2d_pair(&tmA, lfull, sa + j * BOX_BYTES, m_blk * BM + j * 64, kb * BK);
          }
          if (B_MN == 0) {
            tma_load_2d_pair(&tmB, lfull, sb, b_k, b_n);
          } else {
#pragma unroll
            for (int j = 0; j < p.n_mma / 2 / 64; ++j) {
              int bn = b_n + j * 64, bk = b_k;
              if (p.conv_wg_cin) {
                const int tap = bn / p.conv_wg_cin;
                bn -= tap * p.conv_wg_cin;
                bk += (tap / 3 - 1) * p.conv_wp + (tap % 3 - 1);      // (taps >= 9: columns beyond N, never stored)
              }
              tma_load_2d_pair(&tmB, lfull, sb + j * BOX_BYTES, bn, bk);
            }
          }
        }
        __syncwarp();
        if (++stage == STAGES2) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == MMA_WARP) {
    if (leader) {
      const uint32_t idesc = make_idesc(2 * BM, p.n_mma, A_MN, B_MN);
      const uint32_t smem_base = smem_u32(smem);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = cluster_id; tile < total_tiles; tile += num_clusters) {
        const int split = (tile / p.n_tiles) / p.m_groups;
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        GEMM_TRACE(7, tile / num_clusters);
        mbar_wait(tempty_bar + acc, acc_phase ^ 1);
        tc_fence_after();
        GEMM_TRACE(0, tile / num_clusters);
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar + stage, phase);
          tc_fence_after();
          if (kb == kb0) GEMM_TRACE(1, tile / num_clusters);
          if (kb == kb1 - 1) GEMM_TRACE(2, tile / num_clusters);
          if (elect_one()) {
            const uint32_t sa = smem_base + stage * STAGE2_BYTES;
            const uint32_t sb = sa + A_BYTES;
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              const uint64_t da = A_MN == 0 ? smem_desc(sa + k * 32, 16, 1024) : smem_desc(sa + k * 2048, BOX_BYTES, 1024);
              const uint64_t db = B_MN == 0 ? smem_desc(sb + k * 32, 16, 1024) : smem_desc(sb + k * 2048, BOX_BYTES, 1024);
              umma_bf16_pair(d_tmem, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            }
            umma_commit_pair(empty_bar + stage, 3);                      // the stage is free in both CTAs
            if (kb == kb1 - 1) umma_commit_pair(tfull_bar + acc, 3);     // both halves of the accumulator are complete
          }
          __syncwarp();
          if (++stage == STAGES2) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    const int ew = warp;               // 0..7
    const int quarter = warp & 3;      // TMEM lane quarter this warp may access
    const int half = ew >> 2;          // column half: [half*128, half*128+128)
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool vec_ok = (p.epi.ldc % 4 == 0) && (!p.epi.aux || p.epi.ldaux % 4 == 0);
    float *stage = epi_stage + ew * EPI_STAGE_FLOATS;
    const uint32_t ltempty0 = mapa_u32(tempty_bar, 0);     // the leader's accumulator-free barriers
    for (int tile = cluster_id; tile < total_tiles; tile += num_clusters) {
      const int n_blk = tile % p.n_tiles;
      const int m_blk = ((tile / p.n_tiles) % p.m_groups) * 2 + crank;
      const int row0 = m_blk * BM + quarter * 32;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + half * 128;
      const int col_base = n_blk * BN + half * 128;
      const int tr = ew == 0 ? tile / num_clusters : -1;     // (trace builds: stamps of epilogue warp 0)
      // slabs inside N with vectorisable pitches and a bf16 (or no) aux operand take the lean epilogue
      // (GELU with a saved pre-activation -- round 1's backward, tests and tools only -- takes the generic path: the lean GELU
      //  instantiation, the taps pass's fc1, carries no aux code at all)
      const bool lean_ok = vec_ok && !p.atomic_out && (!p.epi.aux || p.epi.aux_dtype == ASIS_BF16) &&
                           !(p.epi.kind == ASIS_EPI_GELU && p.epi.aux);
      const bool lean = lean_ok && col_base + 128 <= p.N;
      if (lean) {
        const uint32_t st32 = smem_u32(stage);
        const bool cb = CDT >= 0 ? CDT == 1 : p.epi.c_dtype == ASIS_BF16;
#define ASIS_EPI3(K)                                                                                                   \
  do {                                                                                                                 \
    if (cb) epi_slab3<K, true, true>(p, taddr, st32, row0, col_base, lane, tfull_bar + acc, acc_phase, tr, 4);         \
    else epi_slab3<K, false, true>(p, taddr, st32, row0, col_base, lane, tfull_bar + acc, acc_phase, tr, 4);           \
  } while (0)
        switch (EPI >= 0 ? EPI : p.epi.kind) {
          case ASIS_EPI_GELU: ASIS_EPI3(ASIS_EPI_GELU); break;
          case ASIS_EPI_SCALE_RESIDUAL:
            if (AUX >= 0 ? AUX == 1 : p.epi.aux != nullptr)
              epi_slab3<ASIS_EPI_SCALE_RESIDUAL, false, true, true>(p, taddr, st32, row0, col_base, lane, tfull_bar + acc, acc_phase, tr, 4);
            else
              epi_slab3<ASIS_EPI_SCALE_RESIDUAL, false, true, false>(p, taddr, st32, row0, col_base, lane, tfull_bar + acc, acc_phase, tr, 4);
            break;
          case ASIS_EPI_DGELU: ASIS_EPI3(ASIS_EPI_DGELU); break;
          case ASIS_EPI_ACCUMULATE: epi_slab3<ASIS_EPI_ACCUMULATE, false, true>(p, taddr, st32, row0, col_base, lane, tfull_bar + acc, acc_phase, tr, 4); break;
          case ASIS_EPI_GELU_GRAD: ASIS_EPI3(ASIS_EPI_GELU_GRAD); break;
          case ASIS_EPI_MUL_AUX: ASIS_EPI3(ASIS_EPI_MUL_AUX); break;
          default: ASIS_EPI3(ASIS_EPI_NONE); break;
        }
#undef ASIS_EPI3
      } else {
        switch (EPI >= 0 ? EPI : p.epi.kind) {
          case ASIS_EPI_GELU: epi_slab<ASIS_EPI_GELU>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase, tr); break;
          case ASIS_EPI_SCALE_RESIDUAL: epi_slab<ASIS_EPI_SCALE_RESIDUAL>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase, tr); break;
          case ASIS_EPI_DGELU: epi_slab<ASIS_EPI_DGELU>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase, tr); break;
          case ASIS_EPI_ACCUMULATE: epi_slab<ASIS_EPI_ACCUMULATE>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase, tr); break;
          case ASIS_EPI_GELU_GRAD: epi_slab<ASIS_EPI_GELU_GRAD>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase, tr); break;
          case ASIS_EPI_MUL_AUX: epi_slab<ASIS_EPI_MUL_AUX>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase, tr); break;
          default: epi_slab<ASIS_EPI_NONE>(p, taddr, stage, row0, col_base, vec_ok, lane, tfull_bar + acc, acc_phase, tr); break;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (tr >= 0) GEMM_TRACE(8, tr);
      if (lane == 0) mbar_arrive_cluster(ltempty0 + acc * 8);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();     // nobody leaves (or frees TMEM) while the peer may still read this CTA's smem / arrive here
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

#ifdef ASIS_TRACE
extern "C" int asis_debug_set_gemm_trace(void *dev_buf) {
  unsigned long long *ptr = (unsigned long long *)dev_buf;
  return cudaMemcpyToSymbol(g_gemm_trace, &ptr, sizeof(ptr)) == cudaSuccess ? 0 : -1;
}
#endif

// ---- host ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void *f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)f;
  });
  return fn;
}

int make_tmap_2d(CUtensorMap *map, const void *base, uint64_t inner, uint64_t outer, uint64_t pitch_elems,
                 uint32_t box_inner, uint32_t box_outer) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) ASIS_FAIL(ASIS_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {pitch_elems * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) ASIS_FAIL(ASIS_ERR_CUDA, "cuTensorMapEncodeTiled failed with %d (inner=%llu outer=%llu pitch=%llu)", (int)r, (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)pitch_elems);
  return ASIS_OK;
}

int make_tmap_3d(CUtensorMap *map, const void *base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t pitch1_elems,
                 uint64_t pitch2_elems, uint32_t b0, uint32_t b1, uint32_t b2) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) ASIS_FAIL(ASIS_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {pitch1_elems * 2, pitch2_elems * 2};
  cuuint32_t box[3] = {b0, b1, b2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) ASIS_FAIL(ASIS_ERR_CUDA, "cuTensorMapEncodeTiled(3d) failed with %d", (int)r);
  return ASIS_OK;
}

int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int A_MN, int B_MN>
static int launch_variant(const CUtensorMap &ta, const CUtensorMap &tb, const GemmTcParams &p, int grid, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    ASIS_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
    configured = true;
  }
  gemm_tc_kernel<A_MN, B_MN><<<grid, GEMM_THREADS, GEMM_SMEM, st>>>(ta, tb, p);
  ASIS_LAUNCHED();
  return ASIS_OK;
}

static int launch_single(int a_major, int b_major, const CUtensorMap &ta, const CUtensorMap &tb, const GemmTcParams &p,
                         int grid, cudaStream_t st) {
  if (a_major == ASIS_MAJOR_K && b_major == ASIS_MAJOR_K) return launch_variant<0, 0>(ta, tb, p, grid, st);
  if (a_major == ASIS_MAJOR_K && b_major == ASIS_MAJOR_MN) return launch_variant<0, 1>(ta, tb, p, grid, st);
  if (a_major == ASIS_MAJOR_MN && b_major == ASIS_MAJOR_MN) return launch_variant<1, 1>(ta, tb, p, grid, st);
  return launch_variant<1, 0>(ta, tb, p, grid, st);
}

template <int A_MN, int B_MN, int EPI, int CDT, int AUX>
static int launch_pair_variant(const CUtensorMap &ta, const CUtensorMap &tb, const GemmTcParams &p, int grid, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    ASIS_CUDA(cudaFuncSetAttribute(gemm_tc_pair_kernel<A_MN, B_MN, EPI, CDT, AUX>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM));
    configured = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = GEMM2_SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ASIS_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_pair_kernel<A_MN, B_MN, EPI, CDT, AUX>, ta, tb, p));
  ASIS_LAUNCHED();
  return ASIS_OK;
}

static int launch_pair(int a_major, int b_major, const CUtensorMap &ta, const CUtensorMap &tb, const GemmTcParams &p,
                       int grid, cudaStream_t st) {
  const int kind = p.epi.kind;
  const bool bf = p.epi.c_dtype == ASIS_BF16;
  // the (majors, epilogue, output dtype) combinations of the training step: one specialised kernel each
  if (a_major == ASIS_MAJOR_K && b_major == ASIS_MAJOR_K) {          // nn.Linear forward, implicit convolution forward
    if (kind == ASIS_EPI_NONE) return bf ? launch_pair_variant<0, 0, ASIS_EPI_NONE, 1, -1>(ta, tb, p, grid, st)
                                         : launch_pair_variant<0, 0, ASIS_EPI_NONE, 0, -1>(ta, tb, p, grid, st);
    if (kind == ASIS_EPI_GELU && bf) return launch_pair_variant<0, 0, ASIS_EPI_GELU, 1, -1>(ta, tb, p, grid, st);
    if (kind == ASIS_EPI_SCALE_RESIDUAL && !bf)
      return p.epi.aux ? launch_pair_variant<0, 0, ASIS_EPI_SCALE_RESIDUAL, 0, 1>(ta, tb, p, grid, st)
                       : launch_pair_variant<0, 0, ASIS_EPI_SCALE_RESIDUAL, 0, 0>(ta, tb, p, grid, st);
    if (kind == ASIS_EPI_GELU_GRAD && bf) return launch_pair_variant<0, 0, ASIS_EPI_GELU_GRAD, 1, -1>(ta, tb, p, grid, st);
    return launch_pair_variant<0, 0, -1, -1, -1>(ta, tb, p, grid, st);
  }
  if (a_major == ASIS_MAJOR_K && b_major == ASIS_MAJOR_MN) {         // input gradients
    if (kind == ASIS_EPI_NONE && bf) return launch_pair_variant<0, 1, ASIS_EPI_NONE, 1, -1>(ta, tb, p, grid, st);
    if (kind == ASIS_EPI_MUL_AUX && bf) return launch_pair_variant<0, 1, ASIS_EPI_MUL_AUX, 1, -1>(ta, tb, p, grid, st);
    return launch_pair_variant<0, 1, -1, -1, -1>(ta, tb, p, grid, st);
  }
  if (a_major == ASIS_MAJOR_MN && b_major == ASIS_MAJOR_MN) {        // weight gradients
    if (kind == ASIS_EPI_NONE && !bf) return launch_pair_variant<1, 1, ASIS_EPI_NONE, 0, -1>(ta, tb, p, grid, st);
    return launch_pair_variant<1, 1, -1, -1, -1>(ta, tb, p, grid, st);
  }
  return launch_pair_variant<1, 0, -1, -1, -1>(ta, tb, p, grid, st);
}

// narrow outputs (the N = 64 / 128 convolutions and adapter projections): a 256-wide MMA would spend 4x / 2x the tensor
// time on columns nobody stores.  MN-major B comes in 64-column boxes, one per CTA at least: 128 is its minimum.
static int pick_n_mma(int N, int b_major) {
  if (N <= 64 && b_major == ASIS_MAJOR_K) return 64;
  if (N <= 128) return 128;
  return BN;
}

// 3x3 / stride 1 / pad 1 convolution pieces as implicit GEMMs over zero-padded channels-last maps
//   op 0 forward: y_p[R, Cout] = sum_t x_p[R + off_t, Cin] . W_t^T      A = x_p, B = w2 [Cout, 9 Cin] (K-major)
//   op 1 dgrad:   dx_p[R, Cin] = sum_t dy_p[R - off_t, Cout] . W_t      A = dy_p, B = w2 read MN-major (rows = Cout)
//   op 2 wgrad:   dW_t[Cout, Cin] = dy_p^T . x_p[. + off_t]  one split-K GEMM with N = 9 Cin: the 64-column boxes of B
//                 carry their tap's row shift (conv_wg_cin)
// R = B (H+2) (W+2) rows, off_t = (ky-1)(W+2) + (kx-1).  Border rows of the outputs of op 0 / 1 hold values of
// positions outside the image: consumers read the logical pixels only.
int gemm_tc_conv3x3(int op, const void *a, const void *b, void *c, int c_dtype, const float *bias, int B, int H, int W, int Cin,
                    int Cout, cudaStream_t st) {
  ASIS_REQUIRE(op >= 0 && op <= 2, "conv3x3_gemm: op must be 0 (forward), 1 (input gradient) or 2 (weight gradient)");
  ASIS_REQUIRE(aligned16(a) && aligned16(b) && aligned16(c), "conv3x3_gemm: pointers must be 16-byte aligned");
  ASIS_REQUIRE(Cin % 64 == 0 && Cout % 64 == 0, "conv3x3_gemm: Cin=%d and Cout=%d must be multiples of 64", Cin, Cout);
  const int64_t R64 = (int64_t)B * (H + 2) * (W + 2);
  ASIS_REQUIRE(R64 < (1ll << 31) - 4096, "conv3x3_gemm: map too large");
  const int R = (int)R64, Wp = W + 2;
  const int sms = sm_count();
  if (op == 2) {
    ASIS_REQUIRE(c_dtype == ASIS_F32, "conv3x3_gemm: the weight gradient is f32");
    GemmTcParams p{};
    p.M = Cout; p.N = 9 * Cin; p.K = R;
    p.n_mma = BN;
    p.m_tiles = (Cout + BM - 1) / BM;
    p.n_tiles = (p.N + BN - 1) / BN;
    p.kb_total = (R + BK - 1) / BK;
    p.m_groups = (p.m_tiles + 1) / 2;
    p.conv_wg_cin = Cin;
    p.conv_wp = Wp;
    p.conv_sign = 1;
    p.epi = EpiArgs{ASIS_EPI_NONE, nullptr, nullptr, nullptr, nullptr, 0, 0, c, ASIS_F32, (int64_t)9 * Cin};
    const int tiles = p.m_groups * p.n_tiles;       // cluster tiles
    int splits = (sms / 2) / tiles;
    if (splits > p.kb_total / 8) splits = p.kb_total / 8;
    if (splits > 64) splits = 64;
    if (splits < 1) splits = 1;
    p.kb_per_split = (p.kb_total + splits - 1) / splits;
    p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
    p.atomic_out = p.splits > 1;
    if (p.atomic_out) ASIS_CUDA(cudaMemsetAsync(c, 0, (size_t)Cout * 9 * Cin * sizeof(float), st));
    CUtensorMap ta, tb;
    if (int rc = make_tmap_2d(&ta, a, Cout, R, Cout, 64, BK)) return rc;      // dy_p read MN-major: inner = Cout (M), rows = pixels (K)
    if (int rc = make_tmap_2d(&tb, b, Cin, R, Cin, 64, BK)) return rc;        // x_p  read MN-major: inner = Cin, rows = pixels (K)
    const int cluster_tiles = tiles * p.splits;
    int clusters = sms / 2;
    if (cluster_tiles < clusters) clusters = cluster_tiles;
    return launch_pair(ASIS_MAJOR_MN, ASIS_MAJOR_MN, ta, tb, p, clusters * 2, st);
  }
  const int Ck = op == 0 ? Cin : Cout;          // channels contracted per tap
  const int Nn = op == 0 ? Cout : Cin;
  GemmTcParams p{};
  p.M = R; p.N = Nn; p.K = 9 * Ck;
  p.n_mma = pick_n_mma(Nn, op == 0 ? ASIS_MAJOR_K : ASIS_MAJOR_MN);
  p.m_tiles = (R + BM - 1) / BM;
  p.n_tiles = (Nn + BN - 1) / BN;
  p.kb_total = 9 * (Ck / BK);
  p.m_groups = (p.m_tiles + 1) / 2;
  p.splits = 1;
  p.kb_per_split = p.kb_total;
  p.conv_taps = 9;
  p.conv_kpt = Ck / BK;
  p.conv_b_k_tap = op == 0 ? Cin : 0;
  p.conv_b_n_tap = op == 0 ? 0 : Cin;
  p.conv_wp = Wp;
  p.conv_sign = op == 0 ? 1 : -1;
  p.epi = EpiArgs{ASIS_EPI_NONE, op == 0 ? bias : nullptr, nullptr, nullptr, nullptr, 0, 0, c, c_dtype, (int64_t)Nn};
  CUtensorMap ta, tb;
  if (int rc = make_tmap_2d(&ta, a, Ck, R, Ck, BK, BM)) return rc;                    // K-major A: inner = channels of one tap
  if (op == 0) {
    if (int rc = make_tmap_2d(&tb, b, (uint64_t)9 * Cin, Cout, (uint64_t)9 * Cin, BK, p.n_mma / 2)) return rc;      // w2 K-major
  } else {
    if (int rc = make_tmap_2d(&tb, b, (uint64_t)9 * Cin, Cout, (uint64_t)9 * Cin, 64, BK)) return rc;          // w2 MN-major: rows = Cout (K)
  }
  const int cluster_tiles = p.m_groups * p.n_tiles;
  int clusters = sms / 2;
  if (cluster_tiles < clusters) clusters = cluster_tiles;
  return launch_pair(ASIS_MAJOR_K, op == 0 ? ASIS_MAJOR_K : ASIS_MAJOR_MN, ta, tb, p, clusters * 2, st);
}

int gemm_tc_launch(const void *A, int a_major, int64_t lda, const void *B, int b_major, int64_t ldb, int M, int N,
                   int K, const EpiArgs &epi, cudaStream_t st) {
  ASIS_REQUIRE(aligned16(A) && aligned16(B) && aligned16(epi.C), "gemm(bf16): A, B, C must be 16-byte aligned");
  ASIS_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, "gemm(bf16): lda=%lld, ldb=%lld must be multiples of 8 elements (TMA 16-byte pitch)", (long long)lda, (long long)ldb);
  GemmTcParams p{};
  p.M = M; p.N = N; p.K = K;
  p.n_mma = pick_n_mma(N, b_major);
  p.m_tiles = (M + BM - 1) / BM;
  p.n_tiles = (N + BN - 1) / BN;
  p.kb_total = (K + BK - 1) / BK;
  p.epi = epi;
  const int CL = p.m_tiles == 1 ? 1 : 2;        // CTAs per cluster: M <= 128 runs the 1-CTA kernel, the rest the pair kernel
  p.m_groups = (p.m_tiles + CL - 1) / CL;
  const int sms = sm_count();
  const int tiles = p.m_groups * CL * p.n_tiles;
  int splits = 1;
  const bool can_split = epi.c_dtype == ASIS_F32 && (epi.kind == ASIS_EPI_ACCUMULATE || (epi.kind == ASIS_EPI_NONE && !epi.bias));
  if (can_split && tiles * 2 <= sms && p.kb_total >= 16) {
    splits = sms / tiles;                        // (one or two output tiles and a 10^6-row reduction -- the stem's weight
    if (splits > p.kb_total / 8) splits = p.kb_total / 8;      //  gradients -- used to stop at 16 CTAs: 370 us for 200 MB)
    if (splits < 1) splits = 1;
  }
  p.kb_per_split = (p.kb_total + splits - 1) / splits;
  splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  p.splits = splits;
  p.atomic_out = splits > 1;
  if (p.atomic_out && epi.kind == ASIS_EPI_NONE) {
    if (epi.ldc == N)
      ASIS_CUDA(cudaMemsetAsync(epi.C, 0, (size_t)M * N * sizeof(float), st));
    else
      ASIS_CUDA(cudaMemset2DAsync(epi.C, epi.ldc * sizeof(float), 0, (size_t)N * sizeof(float), M, st));
  }
  CUtensorMap ta, tb;
  int rc;
  if (a_major == ASIS_MAJOR_K) rc = make_tmap_2d(&ta, A, K, M, lda, BK, BM);
  else rc = make_tmap_2d(&ta, A, M, K, lda, 64, BK);
  if (rc) return rc;
  if (b_major == ASIS_MAJOR_K) rc = make_tmap_2d(&tb, B, K, N, ldb, BK, CL == 1 ? BN : p.n_mma / 2);   // a pair CTA loads half of the B tile
  else rc = make_tmap_2d(&tb, B, N, K, ldb, 64, BK);
  if (rc) return rc;
  const int cluster_tiles = p.m_groups * p.n_tiles * splits;
  int clusters = sms / CL;
  if (cluster_tiles < clusters) clusters = cluster_tiles;
  if (CL == 1) return launch_single(a_major, b_major, ta, tb, p, clusters, st);
  return launch_pair(a_major, b_major, ta, tb, p, clusters * 2, st);
}

}  // namespace asis
