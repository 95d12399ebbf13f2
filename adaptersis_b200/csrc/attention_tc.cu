// attention_tc.cu -- flash-style self-attention on tcgen05 for sm_100a, head_dim 64, bf16 operands,
// fp32 softmax statistics and accumulation.  softmax((q * hd^-0.5) k^T) v over the packed qkv tensor
// [B, T, 3, H, 64] exactly as dinov2/layers/attention.py:56-69 / :73-89 compute it (no mask, no
// dropout); T = 1765 is not a multiple of the 128-row tiles: TMA zero-fills rows >= T and the
// softmax masks key columns >= T.
//
// Forward (attn_fwd8_kernel): persistent CTAs walk
//   items = PAIRS of 128-query tiles of one (image, head).  Warps 0-3 / 4-7 are two softmax warpgroups (1 thread = 1 TMEM
//   lane = 1 query row), warpgroup w owns query tile 2*pair + w over all key tiles; warp 8 = TMA producer (K and V rings,
//   double-buffered Q pair), warp 9 = MMA issuer, event driven (polls the barriers of both warpgroups).  TMEM per
//   warpgroup: S [128 columns] | P [64, bf16 pairs] | O [64].  S = Q K^T -> registers -> ex2 -> bf16 P written to its own
//   TMEM columns and consumed by P V as the A operand straight from TMEM (V MN-major from its TMA tile); O accumulates in
//   TMEM with lazy rescaling (only when the row maximum grows by more than 2^8); the item ends with normalise + store.
// Backward (two atomic-free kernels, both recompute P from the saved log-sum-exp; 576 threads: TMA warp, MMA warp, 2 x 8
//   softmax warps = two threads per row), 64-wide query / key sub-tiles:
//   dK/dV kernel, one CTA per 128 keys:    S^T = K Q^T, dP^T = V dO^T -> P^T, dS^T (TMEM) -> dV += P^T dO, dK += dS^T Q
//   dQ kernel,    one CTA per 128 queries: S = Q K^T, dP = dO V^T -> dS (TMEM) -> dQ += dS K
// Every gradient element is produced by exactly one CTA: deterministic, no atomics.
#include "tc_common.cuh"

namespace asis {

using namespace tc;

constexpr int ATT_THREADS = 320;      // forward: TMA warp, MMA warp, 2 x 4 softmax warps
constexpr int BWD_THREADS = 576;      // backward: TMA warp, MMA warp, 2 x 8 softmax warps (two threads per row)
constexpr int TILE = 128;      // query / key rows per tile
constexpr int HD = 64;
constexpr int T16K = TILE * HD * 2;           // one 128 x 64 bf16 tile
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// write 32 consecutive bf16 of row `row` (columns [col0, col0+32), col0 % 32 == 0) into a K-major,
// 128B-swizzled [128 x 64*n] tile (64-column sub-tiles of 16 KB each)
__device__ __forceinline__ void store_row32_sw128(uint8_t *tile, int row, int col0, const float (&v)[32]) {
  uint8_t *sub = tile + (col0 >> 6) * T16K + (row >> 3) * 1024 + (row & 7) * 128;
  const int ch0 = (col0 & 63) >> 3;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[8 * c + 2 * i], v[8 * c + 2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t *>(&h);
    }
    *reinterpret_cast<uint4 *>(sub + (((ch0 + c) ^ (row & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__device__ __forceinline__ void store_out64(bf16 *dst, const float (&o)[64], float scale) {
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(o[8 * c + 2 * i] * scale, o[8 * c + 2 * i + 1] * scale);
      w[i] = *reinterpret_cast<uint32_t *>(&h);
    }
    reinterpret_cast<uint4 *>(dst)[c] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__device__ __forceinline__ void store_out32(bf16 *dst, const float (&o)[32], float scale) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(o[8 * c + 2 * i] * scale, o[8 * c + 2 * i + 1] * scale);
      w[i] = *reinterpret_cast<uint32_t *>(&h);
    }
    reinterpret_cast<uint4 *>(dst)[c] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// descriptors for the tile shapes used here
// K-major operand [rows x 64*n]: 64-column sub-tiles `sub_bytes` apart, K = columns, 16 per k-step
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t tile, int kstep, uint32_t sub_bytes = T16K) {
  return smem_desc(tile + (kstep >> 2) * sub_bytes + (kstep & 3) * 32, 16, 1024);
}
// MN-major operand [K rows x 64]: N = the 64 columns, 16 K-rows (2 KB) per k-step
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t tile, int kstep) {
  return smem_desc(tile + kstep * 2048, T16K, 1024);
}

// pack 32 floats to bf16 and write them as row `row`, columns [col0, col0+32) of a K-major 128B-swizzled
// tile whose 64-column sub-tiles hold `rows` rows each.  32-bit shared-window addresses and
// st.shared (generic 64-bit pointers cost two registers per precomputed address and spilled).
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void store_row32(uint8_t *tile, int rows, int row, int col0, const float (&v)[32]) {
  const uint32_t sub = smem_u32(tile) + (col0 >> 6) * (rows * 128) + (row >> 3) * 1024 + (row & 7) * 128;
  const int ch0 = (col0 & 63) >> 3;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[8 * c + 2 * i], v[8 * c + 2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t *>(&h);
    }
    st_shared_v4(sub + (((ch0 + c) ^ (row & 7)) << 4), w[0], w[1], w[2], w[3]);
  }
}

// 32 floats -> 16 words of two bf16 each (element 2i in the low half)
__device__ __forceinline__ void pack32_bf16(const float (&v)[32], uint32_t (&w)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t *>(&h);
  }
}

// One row (64 bf16 = 128 bytes) of a K-major, 128B-swizzled smem tile -> 32 TMEM columns of lane `row` (two consecutive
// K elements per column): the layout tcgen05.mma expects for an A operand in tensor memory.
__device__ __forceinline__ void row_to_tmem(const uint8_t *tile, int row, uint32_t taddr) {
  const uint8_t *src = tile + (row >> 3) * 1024 + (row & 7) * 128;
  uint32_t w[32];
#pragma unroll
  for (int ch = 0; ch < 8; ++ch) {
    const uint4 t = *reinterpret_cast<const uint4 *>(src + ((ch ^ (row & 7)) << 4));
    w[4 * ch] = t.x; w[4 * ch + 1] = t.y; w[4 * ch + 2] = t.z; w[4 * ch + 3] = t.w;
  }
  tmem_st32u(taddr, w);
}

struct AttnParams {
  int B, T, H;
  float scale_log2;  // hd^-0.5 * log2(e)
  float scale;
  bf16 *out;         // fwd: [B, T, H*64]
  float *lse;        // [B, H, T]   natural-log log-sum-exp of the scaled scores
  const float *dvec; // bwd: [B, H, Tp] rowsum(dO * O), Tp = ceil(T/64)*64, zero tail
  const float *lse2; // bwd: [B, H, Tp] lse * log2(e), zero tail
  bf16 *dqkv;        // bwd: [B, T, 3, H, 64]
};

constexpr int HALF = 64;                     // key / query tile width of the backward kernels
constexpr int T8K = HALF * HD * 2;           // one 64 x 64 bf16 tile
constexpr uint32_t TMEM_COLS = 512;
constexpr int NSB = 3;              // backward: rotating score buffers in TMEM (tile j uses buffer j % 3)

// ---- optional event trace (built with -DASIS_TRACE only: tools/attn_trace8.py, tools/attn_bwd_trace.py) -------------
#ifdef ASIS_TRACE
__device__ unsigned long long *g_attn_trace = nullptr;     // [16 slots][1024] clock64 stamps of CTA 0
#define ATTN_TRACE(slot, idx)                                                                  \
  do {                                                                                         \
    if (tr && blockIdx.x == 0 && lane == 0 && (idx) < 1024) tr[(slot) * 1024 + (idx)] = clock64(); \
  } while (0)
#else
#define ATTN_TRACE(slot, idx) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------------
// forward, version 8: every softmax warpgroup OWNS a query tile
// ------------------------------------------------------------------------------------------------
// A timeline of the previous forward (v7b) showed two things.  (1) The exponential phase of a
// key tile takes a warp ~2050 clk = exactly the MUFU throughput when the other warpgroup's warp on the same scheduler
// is in its own exponential phase (2 x 128 MUFU.EX2 x 8 clk): the kernel is MUFU bound while it runs.  (2) It does not
// run all the time: the two warpgroups split the KEY tiles of one query tile, so at the end of every item (14 key
// tiles) they meet, exchange (m, l, O) through shared memory and one of them merges and stores -- 7 k clk per item in
// which the other warpgroup and the tensor pipe idle: 26 % of the kernel.
// Here an item is a PAIR of query tiles (256 queries) of one (image, head); warpgroup w keeps (m, l, O) of query tile
// 2*pair + w over all key tiles and normalises / stores it alone: no exchange, no merge, no cross-warpgroup barrier.
// K and V tiles are fetched once per pair (half the TMA / L2 traffic), both warpgroups' MMAs read the same stages.
// TMEM (512 columns): per warpgroup S [128] | P [64] (bf16 pairs) | O [64].  P has its own columns, so S(j+1) may be
// issued as soon as the softmax warps have pulled S(j) into registers -- one score tile ahead is all that is needed.
constexpr int F8_STAGES = 4;
constexpr int F8_SMEM = 2 * 2 * T16K /*Q: 2 warpgroups x 2 buffers*/ + F8_STAGES * 2 * T16K /*K, V rings*/ + 1024 /*align*/ + 512 /*barriers*/;

__global__ void __launch_bounds__(ATT_THREADS, 1)
attn_fwd8_kernel(const __grid_constant__ CUtensorMap tmQKV, const AttnParams p, const int num_items, const int npair) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t *sQ = smem;                            // [buffer][warpgroup] tiles
  uint8_t *sK = sQ + 4 * T16K;
  uint8_t *sV = sK + F8_STAGES * T16K;
  uint64_t *bars = reinterpret_cast<uint64_t *>(sV + F8_STAGES * T16K);
  uint64_t *q_full = bars, *q_empty = q_full + 2, *k_full = q_empty + 2, *k_empty = k_full + F8_STAGES,
           *v_full = k_empty + F8_STAGES, *v_empty = v_full + F8_STAGES, *s_full = v_empty + F8_STAGES, *s_free = s_full + 2,
           *p_full = s_free + 2, *o_full = p_full + 2, *o_empty = o_full + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(o_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef ASIS_TRACE
  unsigned long long *tr = g_attn_trace;
#endif
  constexpr int TMA_WARP = 8, MMA_WARP = 9;      // the SMSP arbiter favours the highest warp id
  const int C = p.H * HD;
  const int nkv = (p.T + TILE - 1) / TILE;
  const int n_my = (num_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int G = n_my * nkv;

  if (warp == TMA_WARP && lane == 0) {
    tma_prefetch_desc(&tmQKV);
    for (int i = 0; i < 2; ++i) {
      mbar_init(q_full + i, 1);
      mbar_init(q_empty + i, 1);
      mbar_init(s_full + i, 1);
      mbar_init(s_free + i, 4);
      mbar_init(p_full + i, 4);
      mbar_init(o_full + i, 1);
      mbar_init(o_empty + i, 4);
    }
    for (int i = 0; i < F8_STAGES; ++i) {
      mbar_init(k_full + i, 1);
      mbar_init(k_empty + i, 1);
      mbar_init(v_full + i, 1);
      mbar_init(v_empty + i, 1);
    }
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  // warpgroup w: S at w*256, P at w*256 + 128, O at w*256 + 192
  constexpr uint32_t WG_COLS = 256, P_OFF = 128, O_OFF = 192;

  if (warp == TMA_WARP) {
    // K(i) is requested one tile ahead of V(i-1): the MMA warp issues S(g+1) before P V(g)
    for (int i = 0; i <= G; ++i) {
      if (i < G) {
        const int k = i / nkv, j = i - k * nkv;
        const int item = (int)blockIdx.x + k * (int)gridDim.x;
        const int bh = item / npair, pr = item - bh * npair, h = bh % p.H, b = bh / p.H;
        if (j == 0) {
          const int qbuf = k & 1;
          if (k >= 2) mbar_wait_wd(q_empty + qbuf, ((k >> 1) - 1) & 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(q_full + qbuf, 2 * T16K);
            tma_load_3d(&tmQKV, q_full + qbuf, sQ + (qbuf * 2 + 0) * T16K, h * HD, (2 * pr) * TILE, b);
            tma_load_3d(&tmQKV, q_full + qbuf, sQ + (qbuf * 2 + 1) * T16K, h * HD, (2 * pr + 1) * TILE, b);   // rows >= T: zero fill
          }
          __syncwarp();
        }
        const int st = i % F8_STAGES, use = i / F8_STAGES;
        if (use > 0) mbar_wait_wd(k_empty + st, (use - 1) & 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(k_full + st, T16K);
          tma_load_3d(&tmQKV, k_full + st, sK + st * T16K, C + h * HD, j * TILE, b);
        }
        __syncwarp();
      }
      const int g = i - 1;
      if (g >= 0) {
        const int k = g / nkv, j = g - k * nkv;
        const int item = (int)blockIdx.x + k * (int)gridDim.x;
        const int bh = item / npair, h = bh % p.H, b = bh / p.H;
        const int st = g % F8_STAGES, use = g / F8_STAGES;
        if (use > 0) mbar_wait_wd(v_empty + st, (use - 1) & 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(v_full + st, T16K);
          tma_load_3d(&tmQKV, v_full + st, sV + st * T16K, 2 * C + h * HD, j * TILE, b);
        }
        __syncwarp();
      }
    }
  } else if (warp == MMA_WARP) {
    constexpr uint32_t idesc_s = make_idesc(TILE, TILE, 0, 0);   // S = Q K^T : both K-major
    constexpr uint32_t idesc_o = make_idesc(TILE, HD, 0, 1);     // O = P V   : V is MN-major
    const uint64_t dQ = desc_kmajor(smem_u32(sQ), 0), dK = desc_kmajor(smem_u32(sK), 0), dV = desc_mnmajor(smem_u32(sV), 0);
    constexpr uint32_t STAGE16 = T16K >> 4;
    // Event-driven issue: each warpgroup has its own score stream (one tile ahead of its softmax) and its own P V
    // stream; the warp polls the barriers of both and issues whatever is ready.  (The first v8 walked the tiles in a
    // fixed order -- S(g+1) for both warpgroups, then P V(g) for w = 0, then for w = 1 -- which re-aligned the two
    // warpgroups every tile: they ran in lockstep, both in the MUFU-bound exponential phase for ~2400 clk, then both in
    // the load / max / wait phases for ~1000 clk with the MUFU pipe idle.  Decoupled, the warpgroup that wins the MUFU
    // arbitration pulls ahead and the phases interleave by themselves.)
    // A K (V) stage is released by whichever warpgroup issues its S (P V) of that tile second; tcgen05.commit covers
    // all earlier MMAs of this thread, so the release is ordered after both.
    struct Stream { int g, k, j, st; uint32_t ph; };
    Stream ss[2] = {{0, 0, 0, 0, 0}, {0, 0, 0, 0, 0}}, ps[2] = {{0, 0, 0, 0, 0}, {0, 0, 0, 0, 0}};
    auto step = [&](Stream &x) {
      ++x.g;
      if (++x.j == nkv) { x.j = 0; ++x.k; }
      if (++x.st == F8_STAGES) { x.st = 0; x.ph ^= 1; }
    };
    long long t_idle = 0;
    while (ps[0].g < G || ps[1].g < G) {
      bool progress = false;
#pragma unroll
      for (int w = 0; w < 2; ++w) {
        // ---- S_w(g) = Q_w K(g)^T: needs Q (first tile of an item), the K stage, and S_w(g-1) pulled into registers
        Stream &x = ss[w];
        if (x.g < G) {
          const int qbuf = x.k & 1;
          bool ok = mbar_test(k_full + x.st, x.ph);
          if (ok && x.j == 0) ok = mbar_test(q_full + qbuf, (x.k >> 1) & 1);
          if (ok && x.g > 0) ok = mbar_test(s_free + w, (x.g - 1) & 1);
          if (ok) {
            tc_fence_after();
            if (elect_one()) {
              const uint64_t a = dQ + (uint32_t)((qbuf * 2 + w) * STAGE16), bdesc = dK + (uint32_t)(x.st * STAGE16);
              const uint32_t d = tmem + w * WG_COLS;
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) umma_bf16(d, a + 2 * kk, bdesc + 2 * kk, idesc_s, kk > 0);
              umma_commit(s_full + w);
              if (ss[w ^ 1].g > x.g) {                     // the other warpgroup has issued this tile already
                umma_commit(k_empty + x.st);
                if (x.j == nkv - 1) umma_commit(q_empty + qbuf);      // both Q tiles may be refilled (item k + 2)
              }
            }
            __syncwarp();
            if (w == 1) ATTN_TRACE(2, x.g);
            step(x);
            progress = true;
          }
        }
        // ---- O_w (+)= P_w(g) V(g): needs P_w(g), the V stage, and (first tile of an item) the previous O_w read out
        Stream &y = ps[w];
        if (y.g < G) {
          bool ok = mbar_test(p_full + w, y.g & 1);
          if (ok) ok = mbar_test(v_full + y.st, y.ph);
          if (ok && y.j == 0 && y.k > 0) ok = mbar_test(o_empty + w, (y.k - 1) & 1);
          if (ok) {
            ATTN_TRACE(w, y.g);            // slots 0 / 1: P_w ready (seen by the MMA warp)
            tc_fence_after();
            if (elect_one()) {
              const uint64_t bdesc = dV + (uint32_t)(y.st * STAGE16);
              const uint32_t d = tmem + w * WG_COLS + O_OFF, a = tmem + w * WG_COLS + P_OFF;
              const uint32_t acc0 = y.j > 0;
#pragma unroll
              for (int kk = 0; kk < 8; ++kk)     // O_w (+)= P_w V, accumulated in TMEM over the item's key tiles
                umma_bf16_ts(d, a + kk * 8, bdesc + 128 * kk, idesc_o, kk > 0 ? 1u : acc0);
              umma_commit(o_full + w);
              if (ps[w ^ 1].g > y.g) umma_commit(v_empty + y.st);
            }
            __syncwarp();
            step(y);
            progress = true;
          }
        }
      }
      if (progress) {
        t_idle = 0;
      } else {                               // watchdog of the polling loop (as mbar_wait_wd): ~2 s without progress
        if (t_idle == 0) t_idle = clock64();
        else if (clock64() - t_idle > 4000000000LL) __trap();
      }
    }
  } else {
    const int w = warp >> 2;                        // warpgroup = query tile of the pair
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;            // row inside the tile == TMEM lane
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const uint32_t tS = tmem + lane_addr + w * WG_COLS, tP = tS + P_OFF, tO = tS + O_OFF;
    for (int k = 0; k < n_my; ++k) {
      const int item = (int)blockIdx.x + k * (int)gridDim.x;
      const int pr = item % npair, bh = item / npair, h = bh % p.H, b = bh / p.H;
      const int g0 = k * nkv;
      // running state in the log2 domain; O_w lives in TMEM and is only touched here when the running maximum grows
      // by more than 2^8 (lazy rescaling)
      float m_use = -INFINITY, l_run = 0.f;
      for (int j = 0; j < nkv; ++j) {
        const int g = g0 + j;
        const int kv0 = j * TILE;
        if (quarter == 0) ATTN_TRACE(3 + 6 * w, g);       // begin
        mbar_wait_wd(s_full + w, g & 1);
        tc_fence_after();
        if (quarter == 0) ATTN_TRACE(4 + 6 * w, g);       // S ready
        float s[4][32];
#pragma unroll
        for (int c = 0; c < 4; ++c) tmem_ld32_issue(tS + c * 32, s[c]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_free + w);            // S_w may be overwritten by the next score tile
        if (quarter == 0) ATTN_TRACE(5 + 6 * w, g);       // ld done
        if (kv0 + TILE > p.T) {                            // only the last key block has invalid columns
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (kv0 + c * 32 + i >= p.T) s[c][i] = -INFINITY;
        }
        // row maximum: 16 independent chains of 8, then a tree (four chains of 32 were a ~380-clk dependent sequence)
        float mx16[16];
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float a = fmaxf(s[c][q * 8], s[c][q * 8 + 1]);
#pragma unroll
            for (int i = 2; i < 8; i += 2) a = fmaxf(a, fmaxf(s[c][q * 8 + i], s[c][q * 8 + i + 1]));
            mx16[c * 4 + q] = a;
          }
#pragma unroll
        for (int st2 = 8; st2 >= 1; st2 >>= 1)
#pragma unroll
          for (int q = 0; q < st2; ++q) mx16[q] = fmaxf(mx16[q], mx16[q + st2]);
        const float m_new = fmaxf(m_use, mx16[0] * p.scale_log2);
        if (quarter == 0) ATTN_TRACE(6 + 6 * w, g);       // max done
        // The running maximum is settled from the scores alone (lazy: it only moves when it grows by more than 2^8), so
        // the exponentials do not wait for P V(g-1); O_w and the P columns are touched after them.
        float alpha = 1.f;
        bool grow = false;
        if (j == 0) {
          m_use = m_new;
        } else {
          grow = m_new - m_use > 8.f;
          if (grow) {
            alpha = fast_exp2(m_use - m_new);
            m_use = m_new;
            l_run *= alpha;
          }
        }
        float l4[4] = {0.f, 0.f, 0.f, 0.f};
        uint32_t pk[64];                                 // the 128 keys of the tile, two per word
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float e0 = fast_exp2(fmaf(s[c][i], p.scale_log2, -m_use));
            const float e1 = fast_exp2(fmaf(s[c][i + 1], p.scale_log2, -m_use));
            l4[(i >> 1) & 3] += e0 + e1;
            __nv_bfloat162 hh = __floats2bfloat162_rn(e0, e1);
            pk[c * 16 + (i >> 1)] = *reinterpret_cast<uint32_t *>(&hh);
          }
        if (quarter == 0) ATTN_TRACE(7 + 6 * w, g);       // exponentials done
        if (j > 0) {
          // P V(g-1) complete: O_w is consistent and the P columns are free.  Every phase of o_full[w] is observed
          // in order (here, or at the end of the item), so the parity waits cannot alias.
          mbar_wait_wd(o_full + w, (g - 1) & 1);
          tc_fence_after();
          if (__any_sync(0xffffffffu, grow)) {
#pragma unroll 1
            for (int c = 0; c < 2; ++c) {                // 32 columns at a time
              float o0[32];
              tmem_ld32(tO + c * 32, o0);
#pragma unroll
              for (int i = 0; i < 32; ++i) o0[i] *= alpha;
              tmem_st32(tO + c * 32, o0);
            }
          }
        }
        {
          uint32_t (&pk0)[32] = *reinterpret_cast<uint32_t (*)[32]>(&pk[0]);
          uint32_t (&pk1)[32] = *reinterpret_cast<uint32_t (*)[32]>(&pk[32]);
          tmem_st32u(tP, pk0);
          tmem_st32u(tP + 32, pk1);
        }
        l_run += (l4[0] + l4[1]) + (l4[2] + l4[3]);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full + w);
        if (quarter == 0) ATTN_TRACE(8 + 6 * w, g);       // P arrived
      }
      // ---- item epilogue: this warpgroup's query tile is complete -- normalise and store, nobody to wait for
      mbar_wait_wd(o_full + w, (g0 + nkv - 1) & 1);
      tc_fence_after();
      float o[64];
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float v[32];
        tmem_ld32(tO + c * 32, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) o[c * 32 + i] = v[i];
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty + w);           // the next item's first P V may overwrite O_w
      const int t = (2 * pr + w) * TILE + row;
      if (t < p.T) {
        store_out64(p.out + ((size_t)b * p.T + t) * C + h * HD, o, 1.f / l_run);
        p.lse[((size_t)b * p.H + h) * p.T + t] = (m_use + log2f(l_run)) * LN2;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// backward prep: D[b,h,t] = sum_e dO[b,t,h,e] * O[b,t,h,e] and lse * log2(e), both written with a
// row pitch Tp = ceil(T/64)*64 (zero tail), so that the kernels can bulk-copy 64-entry tiles and
// never need a bounds check
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) attn_bwd_prep_kernel(const bf16 *__restrict__ out, const bf16 *__restrict__ dout,
                                                            const float *__restrict__ lse, float *__restrict__ dvec,
                                                            float *__restrict__ lse2, int B, int T, int Tp, int H) {
  // one 8-lane group per (b, t, h) with t < Tp: 8 lanes x 8 bf16 = 64 elements
  const size_t gidx = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int sub = threadIdx.x & 7;
  const size_t total = (size_t)B * Tp * H;
  const bool in = gidx < total;
  const int h = in ? (int)(gidx % H) : 0;
  const size_t bt = in ? gidx / H : 0;
  const int t = (int)(bt % Tp);
  const int b = (int)(bt / Tp);
  const bool real = in && t < T;
  float acc = 0.f;
  if (real) {
    const size_t src = (((size_t)b * T + t) * H + h) * HD + sub * 8;
    const uint4 a = *reinterpret_cast<const uint4 *>(out + src);
    const uint4 d = *reinterpret_cast<const uint4 *>(dout + src);
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, dw[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __nv_bfloat162 x = *reinterpret_cast<const __nv_bfloat162 *>(&aw[i]);
      const __nv_bfloat162 y = *reinterpret_cast<const __nv_bfloat162 *>(&dw[i]);
      acc += __low2float(x) * __low2float(y) + __high2float(x) * __high2float(y);
    }
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  if (in && sub == 0) {
    const size_t o = ((size_t)b * H + h) * Tp + t;
    dvec[o] = real ? acc : 0.f;
    lse2[o] = real ? lse[((size_t)b * H + h) * T + t] * LOG2E : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------
// backward, dK / dV: one CTA per (128-key block, head, image); loops over 64-query tiles
// ------------------------------------------------------------------------------------------------
constexpr int BWD_STAGES = 4;
constexpr int BWD_SMEM = 2 * T16K /*resident pair*/ + BWD_STAGES * 2 * T8K /*streamed pair*/ +
                         BWD_STAGES * 2 * HALF * 4 /*lse, D tiles*/ + 1024 + 256;

__global__ void __launch_bounds__(BWD_THREADS, 1)
attn_bwd_dkdv_kernel(const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmQ,
                     const __grid_constant__ CUtensorMap tmDO, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t *sK = smem;
  uint8_t *sV = sK + T16K;
  uint8_t *sQ = sV + T16K;                 // BWD_STAGES x 8 KB
  uint8_t *sDO = sQ + BWD_STAGES * T8K;    // BWD_STAGES x 8 KB
  // P^T and dS^T (bf16) never touch shared memory: each softmax thread writes them back over the first half of the
  // TMEM columns it has just read (its 32 S^T columns -> 16 columns of packed P^T, its 32 dP^T columns -> 16 columns of
  // packed dS^T) and the second pair of GEMMs takes them as the A operand straight from TMEM, as the forward does.
  // With both staged in smem a 64-query tile moved ~150 KB through the 128 B/clk shared-memory port (4 x 24 KB of MMA
  // operand reads, 32 KB of st.shared, the TMA fills) = ~1170 clk against 512 clk of MMA: the kernel was
  // shared-memory bound (ncu: tensor pipe 30 %, 61 M shared wavefronts per launch).
  float *sLse = reinterpret_cast<float *>(sDO + BWD_STAGES * T8K);   // [BWD_STAGES][64]  lse * log2e of the stage's queries
  float *sD = sLse + BWD_STAGES * HALF;                       // [BWD_STAGES][64]
  uint64_t *bars = reinterpret_cast<uint64_t *>(sD + BWD_STAGES * HALF);
  uint64_t *kv_full = bars, *q_full = bars + 1, *q_empty = q_full + BWD_STAGES, *s_full = q_empty + BWD_STAGES,
           *p_full = s_full + NSB, *acc_full = p_full + 2, *op_full = acc_full + 1;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(op_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef ASIS_TRACE
  unsigned long long *tr = (blockIdx.y == 0 && blockIdx.z == 0) ? g_attn_trace : nullptr;   // CTA (0,0,0) only
#endif
  const int k0 = blockIdx.x * TILE, h = blockIdx.y, b = blockIdx.z;
  const int C = p.H * HD;
  const int nq = (p.T + HALF - 1) / HALF;
  const int Tp = nq * HALF;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmDO);
    mbar_init(kv_full, 1);
    for (int i = 0; i < BWD_STAGES; ++i) {
      mbar_init(q_full + i, 1);
      mbar_init(q_empty + i, 1);
    }
    for (int i = 0; i < 2; ++i) mbar_init(s_full + i, 1);
    for (int i = 0; i < 2; ++i) mbar_init(p_full + i, 8);
    mbar_init(acc_full, 1);
    mbar_init(op_full, 16);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  // Two score buffers (tile i uses i % 2): S^T at sb*128, dP^T at sb*128 + 64; dV at 256, dK at 320; the CTA's own K and
  // V tiles as TMEM-RESIDENT A operands at 384 / 416 (32 columns each).  A 128 x 64 x 16 MMA with both operands in shared
  // memory fetches 4 KB (A) + 2 KB (B) for 32 clk of math = 192 B/clk from a 128 B/clk port: the MMA warp's timeline
  // (tools/attn_bwd_trace.py) showed ~1150 clk to get 16 such MMAs accepted per 64-query tile, against 512 clk of math --
  // the kernel was paced by operand fetch.  K and V are the same for every tile of the CTA, so they are copied into
  // tensor memory once; with P^T / dS^T there as well every MMA of the kernel reads only its 2 KB B operand from smem.
  constexpr int NSBK = 2;
  const uint32_t tSC = tmem, tDV = tmem + NSBK * 2 * HALF, tDK = tDV + HD, tKop = tDK + HD, tVop = tKop + HD / 2;

  if (warp == 0) {
    const float *lse_b = p.lse2 + ((size_t)b * p.H + h) * Tp;
    const float *d_b = p.dvec + ((size_t)b * p.H + h) * Tp;
    if (elect_one()) {
      mbar_arrive_expect_tx(kv_full, 2 * T16K);
      tma_load_3d(&tmKV, kv_full, sK, C + h * HD, k0, b);
      tma_load_3d(&tmKV, kv_full, sV, 2 * C + h * HD, k0, b);
    }
    __syncwarp();
    for (int i = 0; i < nq; ++i) {
      const int st = i % BWD_STAGES, use = i / BWD_STAGES;
      if (use > 0) mbar_wait(q_empty + st, (use - 1) & 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(q_full + st, 2 * T8K + 2 * HALF * 4);
        tma_load_3d(&tmQ, q_full + st, sQ + st * T8K, h * HD, i * HALF, b);
        tma_load_3d(&tmDO, q_full + st, sDO + st * T8K, h * HD, i * HALF, b);
        bulk_load_1d(q_full + st, sLse + st * HALF, lse_b + i * HALF, HALF * 4);
        bulk_load_1d(q_full + st, sD + st * HALF, d_b + i * HALF, HALF * 4);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    {
      constexpr uint32_t idesc_s = make_idesc(TILE, HALF, 0, 0);   // [128 keys] x [64 queries]
      constexpr uint32_t idesc_g = make_idesc(TILE, HD, 0, 1);     // [128 keys] x [64 hd], B MN-major
      const uint32_t aQ = smem_u32(sQ), aDO = smem_u32(sDO);
      mbar_wait(op_full, 0);                // K and V are in tensor memory
      tc_fence_after();
      // Score buffer i % 2 is rewritten by tile i + 2; its previous readers are the softmax warps of tile i (done: the
      // P^T / dS^T of tile i exist) and the second GEMM pair of tile i, which this warp issued before -- tcgen05.mma
      // executes in issue order, so no barrier is needed.
      auto issue_scores = [&](int i) {      // S^T = K Q_i^T, dP^T = V dO_i^T into score buffer i % 3
        const int sb = i % NSBK, st = i % BWD_STAGES;
        mbar_wait(q_full + st, (i / BWD_STAGES) & 1);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ts(tSC + sb * 2 * HALF, tKop + k * 8, desc_kmajor(aQ + st * T8K, k), idesc_s, k > 0);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ts(tSC + sb * 2 * HALF + HALF, tVop + k * 8, desc_kmajor(aDO + st * T8K, k), idesc_s, k > 0);
          umma_commit(s_full + sb);
        }
        __syncwarp();
      };
      for (int i = 0; i < NSBK && i < nq; ++i) issue_scores(i);
      for (int i = 0; i < nq; ++i) {
        const int w = i & 1, u = i >> 1, st = i % BWD_STAGES;
        mbar_wait(p_full + w, u & 1);         // P^T and dS^T of tile i are in TMEM
        tc_fence_after();
        ATTN_TRACE(0, i);
        if (elect_one()) {
          // A operand from TMEM: 16 queries (one k-step) = 8 columns; queries [0,32) sit at columns [0,16) of the
          // buffer half, queries [32,64) at columns [32,48) (each thread wrote over the columns it had read)
          const uint32_t aP = tSC + (i % NSBK) * 2 * HALF, aDS = aP + HALF;
#pragma unroll
          for (int k = 0; k < 4; ++k)         // dV += P^T dO      (K = 64 queries)
            umma_bf16_ts(tDV, aP + (k >> 1) * 32 + (k & 1) * 8, desc_mnmajor(aDO + st * T8K, k), idesc_g, (i > 0 || k > 0));
#pragma unroll
          for (int k = 0; k < 4; ++k)         // dK += dS^T Q
            umma_bf16_ts(tDK, aDS + (k >> 1) * 32 + (k & 1) * 8, desc_mnmajor(aQ + st * T8K, k), idesc_g, (i > 0 || k > 0));
          umma_commit(q_empty + st);          // the Q/dO/lse/D stage may be refilled
          if (i == nq - 1) umma_commit(acc_full);
        }
        __syncwarp();
        ATTN_TRACE(1, i);
        if (i + NSBK < nq) issue_scores(i + NSBK);
        ATTN_TRACE(2, i);
      }
    }
  } else {
    // 8 warps per warpgroup: two threads per key row, each owns 32 of the tile's 64 query columns
    const int w = (warp - 2) >> 3;
    const int c = ((warp - 2) >> 2) & 1;     // column half
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;     // key row inside the tile
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    // once per CTA: the 256 softmax threads copy the K tile (column half 0) and the V tile (column half 1), one row each
    mbar_wait(kv_full, 0);
    row_to_tmem(c == 0 ? sK : sV, row, (c == 0 ? tKop : tVop) + lane_addr);
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(op_full);
    for (int i = w; i < nq; i += 2) {
      const int sb = i % NSBK, st = i % BWD_STAGES;
      if (quarter == 0 && c == 0) ATTN_TRACE(4, i);
      mbar_wait(q_full + st, (i / BWD_STAGES) & 1);   // lse / D tile of this stage (bulk copies) has landed
      mbar_wait(s_full + sb, (i / NSBK) & 1);
      tc_fence_after();
      if (quarter == 0 && c == 0) ATTN_TRACE(5, i);
      const float *myLse = sLse + st * HALF, *myD = sD + st * HALF;
      // No masking is needed here: query columns >= T have zero Q / dO rows (TMA zero fill) and
      // lse = D = 0, so their P^T multiplies zero dO rows and their dS^T is exactly 0; key rows >= T
      // only pollute their own (never stored) dV / dK rows.
      {
        float st_[32], dp[32];
        tmem_ld32_issue(tSC + lane_addr + sb * 2 * HALF + c * 32, st_);
        tmem_ld32_issue(tSC + lane_addr + sb * 2 * HALF + HALF + c * 32, dp);
        tmem_ld_wait();
        if (quarter == 0 && c == 0) ATTN_TRACE(6, i);
#pragma unroll
        for (int q4 = 0; q4 < 8; ++q4) {
          const float4 L = reinterpret_cast<const float4 *>(myLse)[c * 8 + q4];
          const float4 Dv = reinterpret_cast<const float4 *>(myD)[c * 8 + q4];
          const float ls[4] = {L.x, L.y, L.z, L.w}, ds[4] = {Dv.x, Dv.y, Dv.z, Dv.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int q = q4 * 4 + k;
            const float pr = fast_exp2(fmaf(st_[q], p.scale_log2, -ls[k]));
            st_[q] = pr;
            dp[q] = pr * (dp[q] - ds[k]);
          }
        }
        uint32_t pk[16];
        pack32_bf16(st_, pk);
        tmem_st16u(tSC + lane_addr + sb * 2 * HALF + c * 32, pk);             // P^T over the S^T columns just read
        pack32_bf16(dp, pk);
        tmem_st16u(tSC + lane_addr + sb * 2 * HALF + HALF + c * 32, pk);      // dS^T over the dP^T columns just read
      }
      if (quarter == 0 && c == 0) ATTN_TRACE(9, i);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full + w);
      if (quarter == 0 && c == 0) ATTN_TRACE(10, i);
    }
    mbar_wait(acc_full, 0);
    tc_fence_after();
    // warpgroup 0 writes dV, warpgroup 1 writes dK; each thread 32 of the 64 columns
    const int t = k0 + row;
    float v[32];
    tmem_ld32((w == 0 ? tDV : tDK) + lane_addr + c * 32, v);
    if (t < p.T)
      store_out32(p.dqkv + ((size_t)b * p.T + t) * 3 * C + (w == 0 ? 2 * C : C) + h * HD + c * 32, v, w == 0 ? 1.f : p.scale);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// backward, dQ: one CTA per (128-query block, head, image); loops over 64-key tiles
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BWD_THREADS, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO,
                   const __grid_constant__ CUtensorMap tmKV, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t *sQ = smem;
  uint8_t *sDO = sQ + T16K;
  uint8_t *sK = sDO + T16K;                // BWD_STAGES x 8 KB
  uint8_t *sV = sK + BWD_STAGES * T8K;     // BWD_STAGES x 8 KB
  // dS (bf16) is written back over the dP columns in TMEM and consumed from there (see the dK/dV kernel)
  uint64_t *bars = reinterpret_cast<uint64_t *>(sV + BWD_STAGES * T8K);
  uint64_t *q_full = bars, *kv_full = bars + 1, *kv_empty = kv_full + BWD_STAGES, *s_full = kv_empty + BWD_STAGES,
           *p_full = s_full + NSB, *acc_full = p_full + 2, *op_full = acc_full + 1;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(op_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * TILE, h = blockIdx.y, b = blockIdx.z;
  const int C = p.H * HD;
  const int nkv = (p.T + HALF - 1) / HALF;
  const int Tp = nkv * HALF;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmKV);
    mbar_init(q_full, 1);
    for (int i = 0; i < BWD_STAGES; ++i) {
      mbar_init(kv_full + i, 1);
      mbar_init(kv_empty + i, 1);
    }
    for (int i = 0; i < NSB; ++i) mbar_init(s_full + i, 1);
    for (int i = 0; i < 2; ++i) mbar_init(p_full + i, 8);
    mbar_init(acc_full, 1);
    mbar_init(op_full, 16);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  // S at sb*128, dP at sb*128 + 64 (3 buffers); dQ at 384; the CTA's own Q and dO tiles as TMEM-resident A operands at
  // 448 / 480 (see the dK/dV kernel: every MMA then reads only its 2 KB B operand from shared memory)
  const uint32_t tSC = tmem, tDQ = tmem + NSB * 2 * HALF, tQop = tDQ + HD, tDOop = tQop + HD / 2;

  if (warp == 0) {
    if (elect_one()) {
      mbar_arrive_expect_tx(q_full, 2 * T16K);
      tma_load_3d(&tmQ, q_full, sQ, h * HD, q0, b);
      tma_load_3d(&tmDO, q_full, sDO, h * HD, q0, b);
    }
    __syncwarp();
    for (int j = 0; j < nkv; ++j) {
      const int st = j % BWD_STAGES, use = j / BWD_STAGES;
      if (use > 0) mbar_wait(kv_empty + st, (use - 1) & 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(kv_full + st, 2 * T8K);
        tma_load_3d(&tmKV, kv_full + st, sK + st * T8K, C + h * HD, j * HALF, b);
        tma_load_3d(&tmKV, kv_full + st, sV + st * T8K, 2 * C + h * HD, j * HALF, b);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    {
      constexpr uint32_t idesc_s = make_idesc(TILE, HALF, 0, 0);
      constexpr uint32_t idesc_g = make_idesc(TILE, HD, 0, 1);
      const uint32_t aK = smem_u32(sK), aV = smem_u32(sV);
      mbar_wait(op_full, 0);                // Q and dO are in tensor memory
      tc_fence_after();
      auto issue_scores = [&](int j) {      // S = Q K_j^T, dP = dO V_j^T into score buffer j % 3
        const int sb = j % NSB, st = j % BWD_STAGES;    // (buffer reuse is ordered by the issue order of this warp's MMAs)
        mbar_wait(kv_full + st, (j / BWD_STAGES) & 1);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ts(tSC + sb * 2 * HALF, tQop + k * 8, desc_kmajor(aK + st * T8K, k), idesc_s, k > 0);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ts(tSC + sb * 2 * HALF + HALF, tDOop + k * 8, desc_kmajor(aV + st * T8K, k), idesc_s, k > 0);
          umma_commit(s_full + sb);
        }
        __syncwarp();
      };
      for (int j = 0; j < NSB && j < nkv; ++j) issue_scores(j);
      for (int j = 0; j < nkv; ++j) {
        const int w = j & 1, u = j >> 1, st = j % BWD_STAGES;
        mbar_wait(p_full + w, u & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t aDS = tSC + (j % NSB) * 2 * HALF + HALF;
#pragma unroll
          for (int k = 0; k < 4; ++k)         // dQ += dS K      (K = 64 keys), dS from TMEM
            umma_bf16_ts(tDQ, aDS + (k >> 1) * 32 + (k & 1) * 8, desc_mnmajor(aK + st * T8K, k), idesc_g, (j > 0 || k > 0));
          umma_commit(kv_empty + st);
          if (j == nkv - 1) umma_commit(acc_full);
        }
        __syncwarp();
        if (j + NSB < nkv) issue_scores(j + NSB);
      }
    }
  } else {
    const int w = (warp - 2) >> 3;
    const int c = ((warp - 2) >> 2) & 1;     // column half
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const int t = q0 + row;
    const bool row_ok = t < p.T;
    const float lse2 = t < Tp ? p.lse2[((size_t)b * p.H + h) * Tp + t] : 0.f;
    const float dsum = t < Tp ? p.dvec[((size_t)b * p.H + h) * Tp + t] : 0.f;
    // once per CTA: Q rows by column half 0, dO rows by column half 1
    mbar_wait(q_full, 0);
    row_to_tmem(c == 0 ? sQ : sDO, row, (c == 0 ? tQop : tDOop) + lane_addr);
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(op_full);
    for (int j = w; j < nkv; j += 2) {
      const int sb = j % NSB;
      mbar_wait(s_full + sb, (j / NSB) & 1);
      tc_fence_after();
      // No masking: key columns >= T multiply zero K rows in dQ += dS K; query rows >= T only
      // pollute their own (never stored) dQ rows.
      {
        float sv[32], dp[32];
        tmem_ld32_issue(tSC + lane_addr + sb * 2 * HALF + c * 32, sv);
        tmem_ld32_issue(tSC + lane_addr + sb * 2 * HALF + HALF + c * 32, dp);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 32; ++q) dp[q] = fast_exp2(fmaf(sv[q], p.scale_log2, -lse2)) * (dp[q] - dsum);
        uint32_t pk[16];
        pack32_bf16(dp, pk);
        tmem_st16u(tSC + lane_addr + sb * 2 * HALF + HALF + c * 32, pk);      // dS over the dP columns just read
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full + w);
    }
    mbar_wait(acc_full, 0);
    tc_fence_after();
    // the column-half-0 warps of each warpgroup write 32 of the 64 dQ columns
    if (c == 0) {
      float v[32];
      tmem_ld32(tDQ + lane_addr + w * 32, v);
      if (row_ok) store_out32(p.dqkv + ((size_t)b * p.T + t) * 3 * C + h * HD + w * 32, v, p.scale);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
#ifdef ASIS_TRACE
extern "C" int asis_debug_set_attn_trace(void *dev_buf) {
  unsigned long long *p = (unsigned long long *)dev_buf;
  return cudaMemcpyToSymbol(g_attn_trace, &p, sizeof(p)) == cudaSuccess ? 0 : -1;
}
#endif

static int set_smem(const void *fn, int bytes) {
  ASIS_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  return ASIS_OK;
}

int attention_tc_forward(const void *qkv, void *out, float *lse, int B, int T, int H, int hd, cudaStream_t st) {
  ASIS_REQUIRE(hd == HD, "attention(bf16): head_dim must be 64");
  ASIS_REQUIRE(aligned16(qkv) && aligned16(out), "attention(bf16): pointers must be 16-byte aligned");
  const int C = H * HD;
  CUtensorMap tq;
  if (int rc = make_tmap_3d(&tq, qkv, 3 * C, T, B, 3 * C, (uint64_t)T * 3 * C, HD, TILE, 1)) return rc;
  static bool configured = false;
  if (!configured) {
    if (int rc = set_smem((const void *)attn_fwd8_kernel, F8_SMEM)) return rc;
    configured = true;
  }
  AttnParams p{};
  p.B = B; p.T = T; p.H = H;
  p.scale = 1.0f / sqrtf((float)HD);
  p.scale_log2 = p.scale * LOG2E;
  p.out = (bf16 *)out;
  p.lse = lse;
  const int nqb = (T + TILE - 1) / TILE;
  const int npair = (nqb + 1) / 2;
  const int num_items = npair * H * B;
  const int grid = num_items < sm_count() ? num_items : sm_count();
  attn_fwd8_kernel<<<grid, ATT_THREADS, F8_SMEM, st>>>(tq, p, num_items, npair);
  ASIS_LAUNCHED();
  return ASIS_OK;
}

static int padded_T(int T) { return (T + HALF - 1) / HALF * HALF; }

size_t attention_tc_bwd_ws(int B, int T, int H, int hd) {
  (void)hd;
  return 2 * align_up((size_t)B * H * padded_T(T) * sizeof(float), 256);
}

int attention_tc_backward(const void *qkv, const void *out, const float *lse, const void *dout, void *dqkv, int B,
                          int T, int H, int hd, void *ws, cudaStream_t st) {
  ASIS_REQUIRE(hd == HD, "attention(bf16): head_dim must be 64");
  ASIS_REQUIRE(aligned16(qkv) && aligned16(out) && aligned16(dout) && aligned16(dqkv) && ws, "attention(bf16): pointers must be 16-byte aligned");
  const int C = H * HD;
  CUtensorMap tq128, tq64, tdo128, tdo64;
  if (int rc = make_tmap_3d(&tq128, qkv, 3 * C, T, B, 3 * C, (uint64_t)T * 3 * C, HD, TILE, 1)) return rc;
  if (int rc = make_tmap_3d(&tq64, qkv, 3 * C, T, B, 3 * C, (uint64_t)T * 3 * C, HD, HALF, 1)) return rc;
  if (int rc = make_tmap_3d(&tdo128, dout, C, T, B, C, (uint64_t)T * C, HD, TILE, 1)) return rc;
  if (int rc = make_tmap_3d(&tdo64, dout, C, T, B, C, (uint64_t)T * C, HD, HALF, 1)) return rc;
  static bool configured = false;
  if (!configured) {
    if (int rc = set_smem((const void *)attn_bwd_dkdv_kernel, BWD_SMEM)) return rc;
    if (int rc = set_smem((const void *)attn_bwd_dq_kernel, BWD_SMEM)) return rc;
    configured = true;
  }
  const int Tp = padded_T(T);
  float *dvec = (float *)ws;
  float *lse2 = (float *)((char *)ws + align_up((size_t)B * H * Tp * sizeof(float), 256));
  {
    const size_t groups = (size_t)B * Tp * H;
    const unsigned blocks = (unsigned)((groups * 8 + 255) / 256);
    attn_bwd_prep_kernel<<<blocks, 256, 0, st>>>((const bf16 *)out, (const bf16 *)dout, lse, dvec, lse2, B, T, Tp, H);
    ASIS_LAUNCHED();
  }
  AttnParams p{};
  p.B = B; p.T = T; p.H = H;
  p.scale = 1.0f / sqrtf((float)HD);
  p.scale_log2 = p.scale * LOG2E;
  p.lse = const_cast<float *>(lse);
  p.dvec = dvec;
  p.lse2 = lse2;
  p.dqkv = (bf16 *)dqkv;
  dim3 grid((T + TILE - 1) / TILE, H, B);
  attn_bwd_dkdv_kernel<<<grid, BWD_THREADS, BWD_SMEM, st>>>(tq128, tq64, tdo64, p);
  ASIS_LAUNCHED();
  attn_bwd_dq_kernel<<<grid, BWD_THREADS, BWD_SMEM, st>>>(tq128, tdo128, tq64, p);
  ASIS_LAUNCHED();
  return ASIS_OK;
}

}  // namespace asis
