// Fused spatial / temporal attention on tcgen05:  out = softmax(q k^T / sqrt(hd)) v  per head.
//
// Replaces the 'math' branch of Attention.forward between its two Linears (reference models/latte.py:50-70:
// reshape/permute/.contiguous(), q@k^T, *scale, softmax, @v, transpose/reshape) AND the two einops
// rearranges that regroup tokens between spatial and temporal blocks (latte.py:355,368).  The hidden state and
// the qkv buffer stay in ONE layout, rows = (b, f, n); the regrouping is done by the TMA box that fetches a tile:
//   spatial  (temporal=0): a tile is 128 consecutive tokens of one frame; keys = the frame's N tokens.
//            3-D map {hd, 3H, T}; Q box {64|16, 1, 128}, K/V box {64|16, 1, N}.
//            N < 128: 128/N whole sequences are packed per tile with a block-diagonal mask (r/N == c/N).
//   temporal (temporal=1): a tile is G = 128/F neighbouring tokens x all F frames, fetched with a 4-D map
//            {hd, 3H, N, B*F} and box {64|16, 1, G, F} -> tile row r = f*G + g; the G sequences are masked
//            block-diagonally (r % G == c % G).  Wasted tensor FLOPs (x G) are free; HBM traffic is minimal:
//            every q/k/v element is read once, every output written once, no transpose pass.
// head_dim 72 (XL) is not a multiple of the UMMA K=16 / N=16 granules: the first 64 dims use 128B-swizzled
// tiles, dims [64,80) a second 32B-swizzled tile whose out-of-range columns TMA zero-fills.
//
// CTA = 160 threads: warps 0-3 softmax/epilogue (thread = tile row = TMEM lane), warp 4 = TMA + MMA issuer.
//   S = Q K^T -> TMEM cols [0,Lk)  ->  registers: mask, max, exp2, sum -> P (16-bit) to smem (K-major SW128)
//   O = P V   -> TMEM cols [256,336) -> registers: * 1/sum -> global.
#include <cstdlib>
#include "common.h"
#include "ptx.cuh"

namespace b200 {

namespace {

constexpr int kThreads = 160;          // attn_long_kernel: warps 0-3 softmax/epilogue, warp 4 TMA + MMA issuer
constexpr int kAttnDefaultImpl = 3;    // launch_mode: which kernel serves the <= 256-key modes (see B200_ATTN_IMPL)

enum { MODE_FULL = 0, MODE_PACKED = 1, MODE_TEMPORAL = 2, MODE_CROSS = 3 };
volatile int g_attn_impl = 0;   // b200_set_attention_impl: 0 = default / environment, 2 or 3 = forced (A/B tests)

struct AttnDev {
  void* out;
  int T;            // total rows
  int D;            // heads * head_dim
  int heads, hd;
  int tokens;       // N
  int frames;       // F
  int group;        // PACKED: N (tokens per sequence); TEMPORAL: G = 128 / F  (power of two)
  int gshift;       // log2(group)
  int k_head0, v_head0;  // index of head 0 of K / V in the (hd, heads-like, rows) view of the K/V buffer
  int kv_rows_per_batch; // CROSS: rows of the K/V buffer per sample (= text length L, the number of valid keys)
  int q_rows_per_batch;  // CROSS: query rows per sample (F * N)
  int Lk;           // keys per tile: N (FULL, <= 256) or 128
  int tiles_per_seq;  // FULL: N / 128; TEMPORAL: N / G
  float scale_log2; // hd^-0.5 * log2(e)
  int dbg;          // B200_ATTN_DBG bits: 1 no TMA*, 2 no softmax math*, 4 no output stores*, 8 no MMA* (* v2 only, wrong results);
                    // v3: 4 no output stores*, 16 all exponentials on the MUFU pipe, 512 contiguous instead of strided work items
  const float* key_bias;  // CROSS: additive bias on the scores, fp32 [batch][128] (natural-log units, e.g. 0 / -10000), or nullptr
  const float* pos_bias;  // CROSS (v3 only): additive bias fp32 [heads][128][128] per (head, query row, key), or nullptr
  int kv_valid;           // CROSS: number of valid keys per sample (<= kv_rows_per_batch)
};

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// group is a power of two: PACKED compares sequence ids (index >> shift), TEMPORAL compares token ids (index & mask)
template <int MODE>
__device__ __forceinline__ int row_key(int r, int gshift) {
  if constexpr (MODE == MODE_PACKED) return r >> gshift;
  if constexpr (MODE == MODE_TEMPORAL) return r & ((1 << gshift) - 1);
  return 0;
}
template <int MODE>
__device__ __forceinline__ bool key_valid(int rkey, int col, int gshift) {
  if constexpr (MODE == MODE_FULL) return true;
  if constexpr (MODE == MODE_CROSS) return col < rkey;   // rkey carries the number of valid keys (text tokens)
  return row_key<MODE>(col, gshift) == rkey;
}

// ------------------------------------------------------------------------------------------------------------------
// Persistent, software-pipelined variant (the one the launchers use): one CTA per SM walks a list of (tile, head) work
// items with everything double-buffered, so the tensor pipe, the TMA engine and the two softmax warpgroups overlap
// across consecutive tiles instead of running back to back inside one short-lived CTA:
//   smem : 2 x {Q, K, V (+ head_dim tails)}             TMEM : 2 x 256 columns
//   per buffer: S = Q K^T -> cols [0,Lk) fp32;  P (16-bit, packed two per column) overwrites cols [0,Lk/2) in place
//               (tcgen05.st from the thread that owns the row);  O = P V (A operand from TMEM) -> cols [Lk/2, Lk/2+80).
//   warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM alloc), warps 2-5 / 6-9 = softmax+epilogue for even / odd tiles.
//   MMA issue order  S_0, S_1, PV_0, S_2, PV_1, ...: S_{i+1} runs on the tensor pipe while tile i is in its softmax.
// P never touches shared memory, which is what makes room for the second Q/K/V buffer.
constexpr int kPipeThreads = 320;

struct PipePlan {
  int q_main, k_main, v_main, q_tail, k_tail, v_tail, buf_bytes, bars, total;
};
__host__ __device__ inline PipePlan make_pipe_plan(int Lk, bool tail) {
  PipePlan s;
  s.q_main = 0;
  s.k_main = 128 * 128;
  s.v_main = s.k_main + Lk * 128;
  s.q_tail = s.v_main + Lk * 128;
  s.k_tail = s.q_tail + (tail ? 128 * 32 : 0);
  s.v_tail = s.k_tail + (tail ? Lk * 32 : 0);
  s.buf_bytes = s.v_tail + (tail ? Lk * 32 : 0);
  s.bars = 2 * s.buf_bytes;
  s.total = s.bars + 256 + 1024;
  return s;
}

template <bool BF16, bool TAIL, int MODE>
__global__ void __launch_bounds__(kPipeThreads, 1)
attn_pipe_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmQt,
                 const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmKVt, const AttnDev p,
                 const int total_items) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const PipePlan sp = make_pipe_plan(p.Lk, TAIL);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + sp.bars);
  uint64_t* qk_full = bars + 0;   // [2] TMA: Q and K of the buffer have landed
  uint64_t* v_full = bars + 2;    // [2] TMA: V has landed
  uint64_t* s_full = bars + 4;    // [2] MMA: S is complete in TMEM          (also: the Q/K smem of the buffer is free)
  uint64_t* p_full = bars + 6;    // [2] softmax (128 arrivals): P is in TMEM
  uint64_t* o_full = bars + 8;    // [2] MMA: O is complete in TMEM          (also: the V smem of the buffer is free)
  uint64_t* o_free = bars + 10;   // [2] epilogue (128 arrivals): O has been read, the TMEM buffer may be overwritten
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int Lk = p.Lk;
  const int H = p.heads;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    for (int b = 0; b < 2; ++b) {
      mbar_init(qk_full + b, 1);
      mbar_init(v_full + b, 1);
      mbar_init(s_full + b, 1);
      mbar_init(p_full + b, 128);
      mbar_init(o_full + b, 1);
      mbar_init(o_free + b, 128);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();   // qkv (written by the preceding GEMM) is visible from here

  const int first = blockIdx.x, step = gridDim.x;

  if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------------ TMA producer
      const uint32_t qk_bytes = 128 * 128 + Lk * 128 + (TAIL ? (128 * 32 + Lk * 32) : 0);
      const uint32_t v_bytes = Lk * 128 + (TAIL ? Lk * 32 : 0);
      int i = 0;
      for (int item = first; item < total_items; item += step, ++i) {
        const int b = i & 1;
        const uint32_t par = (i >> 1) & 1;
        uint8_t* buf = smem + b * sp.buf_bytes;
        const int head = item % H;
        const int tile = item / H;
        if (i >= 2) mbar_wait(s_full + b, par ^ 1);    // S of the tile that used this buffer is done: Q/K smem is free
        if (p.dbg & 1) {
          mbar_arrive(qk_full + b);
          if (i >= 2) mbar_wait(o_full + b, par ^ 1);
          mbar_arrive(v_full + b);
          continue;
        }
        mbar_arrive_expect_tx(qk_full + b, qk_bytes);
        if constexpr (MODE == MODE_TEMPORAL) {
          const int bb = tile / p.tiles_per_seq;
          const int n0 = (tile % p.tiles_per_seq) * p.group;
          const int bf0 = bb * p.frames;
          tma_load_4d(buf + sp.q_main, &tmQ, qk_full + b, 0, head, n0, bf0);
          tma_load_4d(buf + sp.k_main, &tmKV, qk_full + b, 0, p.k_head0 + head, n0, bf0);
          if constexpr (TAIL) {
            tma_load_4d(buf + sp.q_tail, &tmQt, qk_full + b, 64, head, n0, bf0);
            tma_load_4d(buf + sp.k_tail, &tmKVt, qk_full + b, 64, p.k_head0 + head, n0, bf0);
          }
          if (i >= 2) mbar_wait(o_full + b, par ^ 1);  // PV of the tile that used this buffer is done: V smem is free
          mbar_arrive_expect_tx(v_full + b, v_bytes);
          tma_load_4d(buf + sp.v_main, &tmKV, v_full + b, 0, p.v_head0 + head, n0, bf0);
          if constexpr (TAIL) tma_load_4d(buf + sp.v_tail, &tmKVt, v_full + b, 64, p.v_head0 + head, n0, bf0);
        } else {
          int q_row0, kv_row0;
          if constexpr (MODE == MODE_FULL) {
            const int s = tile / p.tiles_per_seq;
            kv_row0 = s * p.tokens;
            q_row0 = kv_row0 + (tile % p.tiles_per_seq) * 128;
          } else if constexpr (MODE == MODE_CROSS) {
            q_row0 = tile * 128;
            kv_row0 = (q_row0 / p.q_rows_per_batch) * p.kv_rows_per_batch;
          } else {
            q_row0 = kv_row0 = tile * 128;
          }
          tma_load_3d(buf + sp.q_main, &tmQ, qk_full + b, 0, head, q_row0);
          tma_load_3d(buf + sp.k_main, &tmKV, qk_full + b, 0, p.k_head0 + head, kv_row0);
          if constexpr (TAIL) {
            tma_load_3d(buf + sp.q_tail, &tmQt, qk_full + b, 64, head, q_row0);
            tma_load_3d(buf + sp.k_tail, &tmKVt, qk_full + b, 64, p.k_head0 + head, kv_row0);
          }
          if (i >= 2) mbar_wait(o_full + b, par ^ 1);
          mbar_arrive_expect_tx(v_full + b, v_bytes);
          tma_load_3d(buf + sp.v_main, &tmKV, v_full + b, 0, p.v_head0 + head, kv_row0);
          if constexpr (TAIL) tma_load_3d(buf + sp.v_tail, &tmKVt, v_full + b, 64, p.v_head0 + head, kv_row0);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ------------------------------------------------------------------ MMA issuer
      const int n_items = first < total_items ? (total_items - first + step - 1) / step : 0;
      const uint32_t idesc_s = umma_idesc_f16(BF16, 128, static_cast<uint32_t>(Lk), false, false);
      const uint32_t idesc_o = umma_idesc_f16(BF16, 128, 64, false, true);   // B = V is MN-major ([key][hd] in smem)
      const uint32_t idesc_ot = umma_idesc_f16(BF16, 128, 16, false, true);
      const int ksteps = Lk / 16;
      auto issue_s = [&](int i) {
        const int b = i & 1;
        const uint32_t par = (i >> 1) & 1;
        uint8_t* buf = smem + b * sp.buf_bytes;
        mbar_wait(qk_full + b, par);
        if (i >= 2) mbar_wait(o_free + b, par ^ 1);     // the epilogue of the previous user has drained the TMEM buffer
        tc_fence_after();
        const uint32_t tS = tmem_base + b * 256;
        const uint64_t dq = umma_smem_desc(smem_u32(buf + sp.q_main), 0, 1024, UMMA_LAYOUT_SW128);
        const uint64_t dk = umma_smem_desc(smem_u32(buf + sp.k_main), 0, 1024, UMMA_LAYOUT_SW128);
        if (!(p.dbg & 8)) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16_ss(tS, umma_desc_advance(dq, k * 32), umma_desc_advance(dk, k * 32), idesc_s, k > 0 ? 1u : 0u);
          if constexpr (TAIL) {
            const uint64_t dqt = umma_smem_desc(smem_u32(buf + sp.q_tail), 0, 256, UMMA_LAYOUT_SW32);
            const uint64_t dkt = umma_smem_desc(smem_u32(buf + sp.k_tail), 0, 256, UMMA_LAYOUT_SW32);
            umma_f16_ss(tS, dqt, dkt, idesc_s, 1u);
          }
        }
        umma_commit(s_full + b);
      };
      if (n_items > 0) issue_s(0);
      for (int i = 0; i < n_items; ++i) {
        if (i + 1 < n_items) issue_s(i + 1);
        const int b = i & 1;
        const uint32_t par = (i >> 1) & 1;
        uint8_t* buf = smem + b * sp.buf_bytes;
        mbar_wait(v_full + b, par);
        mbar_wait(p_full + b, par);
        tc_fence_after();
        const uint32_t tP = tmem_base + b * 256;
        const uint32_t tO = tP + (Lk >> 1);
        const uint64_t dv = umma_smem_desc(smem_u32(buf + sp.v_main), static_cast<uint32_t>(Lk) * 128, 1024, UMMA_LAYOUT_SW128);
        const uint64_t dvt = umma_smem_desc(smem_u32(buf + sp.v_tail), static_cast<uint32_t>(Lk) * 32, 256, UMMA_LAYOUT_SW32);
        for (int k = 0; k < ksteps && !(p.dbg & 8); ++k) {
          umma_f16_ts(tO, tP + k * 8, umma_desc_advance(dv, k * 16 * 128), idesc_o, k > 0 ? 1u : 0u);
          if constexpr (TAIL) umma_f16_ts(tO + 64, tP + k * 8, umma_desc_advance(dvt, k * 16 * 32), idesc_ot, k > 0 ? 1u : 0u);
        }
        umma_commit(o_full + b);
      }
    }
  } else {
    // -------------------------------------------------------------------- softmax + epilogue: thread = tile row
    const int wg = (warp - 2) >> 2;            // warpgroup 0 takes the even work items of this CTA, 1 the odd ones
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;
    const int nchunks = Lk / 32;
    const int rkey = MODE == MODE_CROSS ? p.kv_valid : row_key<MODE>(r, p.gshift);
    const uint32_t t_row = tmem_base + wg * 256 + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t t_o = t_row + (Lk >> 1);
    int i = wg;
    for (int item = first + wg * step; item < total_items; item += 2 * step, i += 2) {
      const uint32_t par = (i >> 1) & 1;
      const int head = item % H;
      const int tile = item / H;
      mbar_wait(s_full + wg, par);
      tc_fence_after();

      const int nch = (p.dbg & 2) ? 0 : nchunks;   // Lk / 32: 4 or 8
      // CROSS with a key bias (padded prompts): scores are s * scale + bias[sample][key]; the sample's 128 bias values are
      // read through the read-only path (same addresses for every thread of the tile)
      const float* brow = nullptr;
      if constexpr (MODE == MODE_CROSS) {
        if (p.key_bias) brow = p.key_bias + static_cast<size_t>((static_cast<long long>(tile) * 128) / p.q_rows_per_batch) * 128;
      }
      // pass 1: row maximum.  Two 32-column TMEM loads are in flight per wait (the loads, not the math, set the pace).
      float mx = -INFINITY;
      for (int c = 0; c < nch; c += 2) {
        uint32_t va[32], vb[32];
        tmem_ld_32x32b_x32(t_row + c * 32, va);
        tmem_ld_32x32b_x32(t_row + (c + 1) * 32, vb);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float a = __uint_as_float(va[j]), b = __uint_as_float(vb[j]);
          if (MODE == MODE_CROSS && brow) {
            a = fmaf(a, p.scale_log2, __ldg(brow + c * 32 + j) * 1.4426950408889634f);
            b = fmaf(b, p.scale_log2, __ldg(brow + (c + 1) * 32 + j) * 1.4426950408889634f);
          }
          if (key_valid<MODE>(rkey, c * 32 + j, p.gshift)) mx = fmaxf(mx, a);
          if (key_valid<MODE>(rkey, (c + 1) * 32 + j, p.gshift)) mx = fmaxf(mx, b);
        }
      }
      const float mscaled = (MODE == MODE_CROSS && brow) ? mx : mx * p.scale_log2;
      float sum = 0.f;
      // pass 2: P = exp2(s * scale - max), written over the S columns already consumed.  The load of chunk c+1 is in flight
      // while chunk c is exponentiated (P chunk c lands in S chunk c/2 <= c, never in a chunk still being loaded).
      auto emit = [&](const uint32_t (&v)[32], int c) {
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float b0 = -mscaled, b1 = -mscaled;
          if (MODE == MODE_CROSS && brow) {
            b0 = fmaf(__ldg(brow + c * 32 + 2 * j), 1.4426950408889634f, -mscaled);
            b1 = fmaf(__ldg(brow + c * 32 + 2 * j + 1), 1.4426950408889634f, -mscaled);
          }
          float e0 = ex2(fmaf(__uint_as_float(v[2 * j]), p.scale_log2, b0));
          float e1 = ex2(fmaf(__uint_as_float(v[2 * j + 1]), p.scale_log2, b1));
          if (!key_valid<MODE>(rkey, c * 32 + 2 * j, p.gshift)) e0 = 0.f;
          if (!key_valid<MODE>(rkey, c * 32 + 2 * j + 1, p.gshift)) e1 = 0.f;
          sum += e0 + e1;
          pk[j] = pack2<BF16>(e0, e1);
        }
        tmem_st_32x32b_x16(t_row + c * 16, pk);
      };
      if (nch > 0) {
        uint32_t va[32], vb[32];
        tmem_ld_32x32b_x32(t_row, va);
        tmem_ld_wait();
        for (int c = 0; c < nch; c += 2) {
          tmem_ld_32x32b_x32(t_row + (c + 1) * 32, vb);
          emit(va, c);
          tmem_ld_wait();
          if (c + 2 < nch) tmem_ld_32x32b_x32(t_row + (c + 2) * 32, va);
          emit(vb, c + 1);
          tmem_ld_wait();
        }
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(p_full + wg);

      long long out_row;
      bool row_ok = true;
      if constexpr (MODE == MODE_TEMPORAL) {
        const int bb = tile / p.tiles_per_seq;
        const int n0 = (tile % p.tiles_per_seq) * p.group;
        out_row = (static_cast<long long>(bb) * p.frames + r / p.group) * p.tokens + n0 + r % p.group;
      } else if constexpr (MODE == MODE_FULL) {
        out_row = static_cast<long long>(tile / p.tiles_per_seq) * p.tokens + (tile % p.tiles_per_seq) * 128 + r;
      } else {
        out_row = static_cast<long long>(tile) * 128 + r;
        row_ok = out_row < p.T;
      }
      uint16_t* optr = reinterpret_cast<uint16_t*>(p.out) + out_row * p.D + head * p.hd;
      const float inv = 1.0f / sum;

      mbar_wait(o_full + wg, par);
      tc_fence_after();
      uint32_t o0[32], o1[32], o2[16];
      tmem_ld_32x32b_x32(t_o, o0);
      tmem_ld_32x32b_x32(t_o + 32, o1);
      if constexpr (TAIL) tmem_ld_32x32b_x16(t_o + 64, o2);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(o_free + wg);                   // O is in registers: the MMA warp may start S of the tile after next
      if (row_ok && !(p.dbg & 4)) {
#pragma unroll
        for (int i4 = 0; i4 < 4; ++i4) {
          uint4 o;
          o.x = pack2<BF16>(__uint_as_float(o0[8 * i4 + 0]) * inv, __uint_as_float(o0[8 * i4 + 1]) * inv);
          o.y = pack2<BF16>(__uint_as_float(o0[8 * i4 + 2]) * inv, __uint_as_float(o0[8 * i4 + 3]) * inv);
          o.z = pack2<BF16>(__uint_as_float(o0[8 * i4 + 4]) * inv, __uint_as_float(o0[8 * i4 + 5]) * inv);
          o.w = pack2<BF16>(__uint_as_float(o0[8 * i4 + 6]) * inv, __uint_as_float(o0[8 * i4 + 7]) * inv);
          *reinterpret_cast<uint4*>(optr + i4 * 8) = o;
        }
#pragma unroll
        for (int i4 = 0; i4 < 4; ++i4) {
          uint4 o;
          o.x = pack2<BF16>(__uint_as_float(o1[8 * i4 + 0]) * inv, __uint_as_float(o1[8 * i4 + 1]) * inv);
          o.y = pack2<BF16>(__uint_as_float(o1[8 * i4 + 2]) * inv, __uint_as_float(o1[8 * i4 + 3]) * inv);
          o.z = pack2<BF16>(__uint_as_float(o1[8 * i4 + 4]) * inv, __uint_as_float(o1[8 * i4 + 5]) * inv);
          o.w = pack2<BF16>(__uint_as_float(o1[8 * i4 + 6]) * inv, __uint_as_float(o1[8 * i4 + 7]) * inv);
          *reinterpret_cast<uint4*>(optr + 32 + i4 * 8) = o;
        }
        if constexpr (TAIL) {
          const int tail8 = (p.hd - 64) / 8;  // 1 (hd 72) or 2 (hd 80)
#pragma unroll
          for (int i4 = 0; i4 < 2; ++i4) {
            if (i4 >= tail8) break;
            uint4 o;
            o.x = pack2<BF16>(__uint_as_float(o2[8 * i4 + 0]) * inv, __uint_as_float(o2[8 * i4 + 1]) * inv);
            o.y = pack2<BF16>(__uint_as_float(o2[8 * i4 + 2]) * inv, __uint_as_float(o2[8 * i4 + 3]) * inv);
            o.z = pack2<BF16>(__uint_as_float(o2[8 * i4 + 4]) * inv, __uint_as_float(o2[8 * i4 + 5]) * inv);
            o.w = pack2<BF16>(__uint_as_float(o2[8 * i4 + 6]) * inv, __uint_as_float(o2[8 * i4 + 7]) * inv);
            *reinterpret_cast<uint4*>(optr + 64 + i4 * 8) = o;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// v3 (round 2): the same TMEM-resident design, re-cut so that more of every engine's work overlaps.
//   * work is split by ROLE WARP, each an in-order stream with its own barriers: warp 0 = TMA producer for Q and K,
//     warp 3 = TMA producer for V, warp 1 = MMA issuer (+ TMEM allocator), warp 2 = output store (TMA bulk store),
//     warps 4.. = softmax/epilogue warpgroups.  No role ever waits on behalf of another.
//   * a "slot" = one tile in flight = one smem stage {Q, K, V} + one TMEM region.
//       LK = 256 (spatial, 256 keys):  2 slots x 256 TMEM columns; TWO warpgroups per tile, each owning 128 key columns
//                                      (row max and row sum exchanged through smem + a 256-thread named barrier), so the
//                                      S -> softmax -> PV chain of a tile is half as long;
//       LK = 128 (temporal / cross / packed / N = 128):  3 slots x 160 TMEM columns, one warpgroup per tile.
//     TMEM per slot: S fp32 [0,LK); P (16-bit, packed two per column) is written over the start of each warpgroup's own
//     S columns -- keys [0,128) -> cols [0,64), keys [128,256) -> cols [128,192); O main (64 cols) at [64,128), O tail
//     (16 cols, head_dim 72/80) at [192,208) resp. [128,144): columns that are dead by the time P V is issued.
//   * the output never leaves through per-thread stores: O * 1/sum goes registers -> the slot's V tile in shared memory
//     (dense [128][head_dim] rows; V is dead once P V has completed) -> ONE TMA bulk store per tile whose box does the
//     (b, f, n) regrouping for temporal tiles, exactly like the loads.  The V producer refills the stage when the store
//     has read it (v_free).
//   * temporal tiles with G = 8 tokens x 16 frames: a row has 16 live keys out of 128 (col % 8 == row % 8).  They are
//     picked out of the TMEM row with a select tree in ONE pass, so a row costs 16 exponentials instead of 128.
//   * spatial tiles: 5 of every 16 exponentials are evaluated on the FMA pipe (Cody-Waite split + degree-4 polynomial,
//     2.8e-6 relative error, far below the 16-bit rounding of P) because the 16-op/clk MUFU pipe is what bounds a
//     128 x 256 tile (2048 clk) once the chain overlaps.
template <int LK>
struct V3 {
  static constexpr int NSLOT = LK == 256 ? 2 : 3;
  static constexpr int WG_PER_TILE = LK == 256 ? 2 : 1;
  static constexpr int NWG = NSLOT * WG_PER_TILE;
  static constexpr int THREADS = 128 + NWG * 128;
  static constexpr int SLOT_COLS = LK == 256 ? 256 : 160;
  static constexpr int O_COL = 64;
  static constexpr int OT_COL = LK == 256 ? 192 : 128;
  static constexpr int TILE_THREADS = WG_PER_TILE * 128;
};

struct V3Plan {
  int q_main, q_tail, k_main, k_tail, v_main, v_tail, stage_bytes, xch, bias, bars, total;
};
__host__ __device__ inline V3Plan make_v3_plan(int LK, bool tail) {
  const int nslot = LK == 256 ? 2 : 3;
  V3Plan s;
  s.q_main = 0;
  s.q_tail = 128 * 128;
  s.k_main = s.q_tail + (tail ? 128 * 32 : 0);
  s.k_tail = s.k_main + LK * 128;
  s.v_main = s.k_tail + (tail ? LK * 32 : 0);
  s.v_tail = s.v_main + LK * 128;     // contiguous with v_main: the output staging tile [128][hd] spans both
  s.stage_bytes = s.v_tail + (tail ? LK * 32 : 0);
  s.xch = nslot * s.stage_bytes;                       // float [nslot][2 kinds][2 halves][128]
  s.bias = s.xch + nslot * 2 * 2 * 128 * 4;            // float [nslot][128]
  s.bars = s.bias + nslot * 128 * 4;
  s.total = s.bars + 256 + 1024;
  return s;
}

// 2^x for x <= 127 on the FMA pipe (arguments below -125 give 2^-125): x = n + f, n = round(x), f in [-0.5, 0.5]; 2^f by
// a degree-4 minimax polynomial (max relative error 2.8e-6), 2^n by adding n to the exponent field.  The spatial v3 tiles
// pass x <= 0; the streaming kernel's lazy maximum passes x up to +ST_TAU.
__device__ __forceinline__ float ex2_poly(float x) {
  x = fmaxf(x, -125.0f);
  const float t = x + 12582912.0f;              // 1.5 * 2^23: the integer n sits in the low mantissa bits
  const float f = x - (t - 12582912.0f);
  float pl = fmaf(0.009582852944731712f, f, 0.055906426161527634f);
  pl = fmaf(pl, f, 0.24024099111557007f);
  pl = fmaf(pl, f, 0.6931241750717163f);
  pl = fmaf(pl, f, 1.0f);
  return __int_as_float(__float_as_int(pl) + (__float_as_int(t) << 23));
}

__device__ __forceinline__ float sel8(const uint32_t* v, int g) {   // v[g], g in [0,8), without dynamic register indexing
  const uint32_t a0 = (g & 1) ? v[1] : v[0], a1 = (g & 1) ? v[3] : v[2], a2 = (g & 1) ? v[5] : v[4], a3 = (g & 1) ? v[7] : v[6];
  const uint32_t b0 = (g & 2) ? a1 : a0, b1 = (g & 2) ? a3 : a2;
  return __uint_as_float((g & 4) ? b1 : b0);
}

template <bool BF16, bool TAIL, int MODE, int LK, bool POLY>
__global__ void __launch_bounds__(V3<LK>::THREADS, 1)
attn_v3_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmQt,
               const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmKVt,
               const __grid_constant__ CUtensorMap tmO, const AttnDev p, const int total_items) {
  using C = V3<LK>;
  constexpr int NSLOT = C::NSLOT;
  static_assert(MODE == MODE_FULL || LK == 128, "only the unmasked spatial mode has 256-key tiles");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const V3Plan sp = make_v3_plan(LK, TAIL);
  float* xch = reinterpret_cast<float*>(smem + sp.xch);
  float* sbias = reinterpret_cast<float*>(smem + sp.bias);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + sp.bars);
  uint64_t* qk_full = bars + 0 * NSLOT;    // TMA: Q and K of the stage have landed
  uint64_t* v_full = bars + 1 * NSLOT;     // TMA: V has landed
  uint64_t* s_full = bars + 2 * NSLOT;     // MMA: S complete in TMEM (also: the stage's Q/K smem is free)
  uint64_t* p_full = bars + 3 * NSLOT;     // softmax (all threads of the tile): P is in TMEM
  uint64_t* o_full = bars + 4 * NSLOT;     // MMA: O complete in TMEM (also: V smem no longer read by the tensor pipe)
  uint64_t* o_free = bars + 5 * NSLOT;     // epilogue (all threads of the tile): O is in registers, the TMEM slot is free
  uint64_t* o_staged = bars + 6 * NSLOT;   // epilogue (all threads of the tile): the output tile is staged in the V smem
  uint64_t* v_free = bars + 7 * NSLOT;     // store warp: the bulk store has read the staging tile, V may be refilled
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8 * NSLOT);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int H = p.heads;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmO);
    for (int b = 0; b < NSLOT; ++b) {
      mbar_init(qk_full + b, 1);
      mbar_init(v_full + b, 1);
      mbar_init(s_full + b, 1);
      mbar_init(p_full + b, C::TILE_THREADS);
      mbar_init(o_full + b, 1);
      mbar_init(o_free + b, C::TILE_THREADS);
      mbar_init(o_staged + b, C::TILE_THREADS);
      mbar_init(v_free + b, 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();   // qkv (written by the preceding GEMM) is visible from here

  // work items (tile, head), head fastest: CTA c takes items c, c + grid, ...  (dbg bit 512, A/B: the contiguous run
  // [c*total/grid, (c+1)*total/grid) instead -- consecutive heads of one tile on one SM.  Measured: no gain for temporal
  // tiles, 13 % SLOWER for spatial ones, so strided stays.)
  const bool strided = (p.dbg & 512) == 0;
  const int item0 = strided ? static_cast<int>(blockIdx.x)
                            : static_cast<int>(static_cast<long long>(blockIdx.x) * total_items / gridDim.x);
  const int item1 = static_cast<int>(static_cast<long long>(blockIdx.x + 1) * total_items / gridDim.x);
  const int step = strided ? static_cast<int>(gridDim.x) : 1;
  const int n_items = strided ? (item0 < total_items ? (total_items - item0 + step - 1) / step : 0) : item1 - item0;

  // tile coordinates of local work item i: the TMA coordinates of its Q rows / K,V rows / output rows
  struct Coord { int head, c2, c3, kv2; };
  auto coord = [&](int i) {
    const int item = item0 + i * step;
    Coord c;
    c.head = item % H;
    const int tile = item / H;
    if constexpr (MODE == MODE_TEMPORAL) {
      c.c2 = (tile % p.tiles_per_seq) * p.group;      // first token of the group
      c.c3 = (tile / p.tiles_per_seq) * p.frames;     // first (b, f) image
      c.kv2 = c.c2;
    } else if constexpr (MODE == MODE_FULL) {
      const int s = tile / p.tiles_per_seq;
      c.kv2 = s * p.tokens;
      c.c2 = c.kv2 + (tile % p.tiles_per_seq) * 128;
      c.c3 = 0;
    } else if constexpr (MODE == MODE_CROSS) {
      c.c2 = tile * 128;
      c.kv2 = (c.c2 / p.q_rows_per_batch) * p.kv_rows_per_batch;
      c.c3 = c.c2 / p.q_rows_per_batch;               // sample index (key-bias row)
    } else {
      c.c2 = c.kv2 = tile * 128;
      c.c3 = 0;
    }
    return c;
  };

  if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------------ TMA producer: Q and K
      const uint32_t qk_bytes = 128 * 128 + LK * 128 + (TAIL ? (128 * 32 + LK * 32) : 0);
      for (int i = 0; i < n_items; ++i) {
        const int sl = i % NSLOT, u = i / NSLOT;
        uint8_t* buf = smem + sl * sp.stage_bytes;
        const Coord c = coord(i);
        if (u > 0) mbar_wait(s_full + sl, (u - 1) & 1);     // S of the tile that used this stage is done
        mbar_arrive_expect_tx(qk_full + sl, qk_bytes);
        if constexpr (MODE == MODE_TEMPORAL) {
          tma_load_4d(buf + sp.q_main, &tmQ, qk_full + sl, 0, c.head, c.c2, c.c3);
          tma_load_4d(buf + sp.k_main, &tmKV, qk_full + sl, 0, p.k_head0 + c.head, c.c2, c.c3);
          if constexpr (TAIL) {
            tma_load_4d(buf + sp.q_tail, &tmQt, qk_full + sl, 64, c.head, c.c2, c.c3);
            tma_load_4d(buf + sp.k_tail, &tmKVt, qk_full + sl, 64, p.k_head0 + c.head, c.c2, c.c3);
          }
        } else {
          tma_load_3d(buf + sp.q_main, &tmQ, qk_full + sl, 0, c.head, c.c2);
          tma_load_3d(buf + sp.k_main, &tmKV, qk_full + sl, 0, p.k_head0 + c.head, c.kv2);
          if constexpr (TAIL) {
            tma_load_3d(buf + sp.q_tail, &tmQt, qk_full + sl, 64, c.head, c.c2);
            tma_load_3d(buf + sp.k_tail, &tmKVt, qk_full + sl, 64, p.k_head0 + c.head, c.kv2);
          }
        }
      }
    }
  } else if (warp == 3) {
    if (lane == 0) {
      // ------------------------------------------------------------------ TMA producer: V
      const uint32_t v_bytes = LK * 128 + (TAIL ? LK * 32 : 0);
      for (int i = 0; i < n_items; ++i) {
        const int sl = i % NSLOT, u = i / NSLOT;
        uint8_t* buf = smem + sl * sp.stage_bytes;
        const Coord c = coord(i);
        if (u > 0) mbar_wait(v_free + sl, (u - 1) & 1);     // the previous tile's output has left the staging tile
        mbar_arrive_expect_tx(v_full + sl, v_bytes);
        if constexpr (MODE == MODE_TEMPORAL) {
          tma_load_4d(buf + sp.v_main, &tmKV, v_full + sl, 0, p.v_head0 + c.head, c.c2, c.c3);
          if constexpr (TAIL) tma_load_4d(buf + sp.v_tail, &tmKVt, v_full + sl, 64, p.v_head0 + c.head, c.c2, c.c3);
        } else {
          tma_load_3d(buf + sp.v_main, &tmKV, v_full + sl, 0, p.v_head0 + c.head, c.kv2);
          if constexpr (TAIL) tma_load_3d(buf + sp.v_tail, &tmKVt, v_full + sl, 64, p.v_head0 + c.head, c.kv2);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ------------------------------------------------------------------ MMA issuer
      constexpr uint32_t idesc_s = umma_idesc_f16(BF16, 128, LK, false, false);
      constexpr uint32_t idesc_o = umma_idesc_f16(BF16, 128, 64, false, true);   // B = V is MN-major ([key][hd] in smem)
      constexpr uint32_t idesc_ot = umma_idesc_f16(BF16, 128, 16, false, true);
      auto issue_s = [&](int i) {
        const int sl = i % NSLOT, u = i / NSLOT;
        uint8_t* buf = smem + sl * sp.stage_bytes;
        mbar_wait(qk_full + sl, u & 1);
        if (u > 0) mbar_wait(o_free + sl, (u - 1) & 1);      // the previous tile's O has been read out of this slot
        tc_fence_after();
        const uint32_t tS = tmem_base + sl * C::SLOT_COLS;
        const uint64_t dq = umma_smem_desc(smem_u32(buf + sp.q_main), 0, 1024, UMMA_LAYOUT_SW128);
        const uint64_t dk = umma_smem_desc(smem_u32(buf + sp.k_main), 0, 1024, UMMA_LAYOUT_SW128);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_f16_ss(tS, umma_desc_advance(dq, k * 32), umma_desc_advance(dk, k * 32), idesc_s, k > 0 ? 1u : 0u);
        if constexpr (TAIL) {
          const uint64_t dqt = umma_smem_desc(smem_u32(buf + sp.q_tail), 0, 256, UMMA_LAYOUT_SW32);
          const uint64_t dkt = umma_smem_desc(smem_u32(buf + sp.k_tail), 0, 256, UMMA_LAYOUT_SW32);
          umma_f16_ss(tS, dqt, dkt, idesc_s, 1u);
        }
        umma_commit(s_full + sl);
      };
      auto issue_pv = [&](int i) {
        const int sl = i % NSLOT, u = i / NSLOT;
        uint8_t* buf = smem + sl * sp.stage_bytes;
        mbar_wait(v_full + sl, u & 1);
        mbar_wait(p_full + sl, u & 1);
        tc_fence_after();
        const uint32_t tS = tmem_base + sl * C::SLOT_COLS;
        const uint64_t dv = umma_smem_desc(smem_u32(buf + sp.v_main), static_cast<uint32_t>(LK) * 128, 1024, UMMA_LAYOUT_SW128);
        const uint64_t dvt = umma_smem_desc(smem_u32(buf + sp.v_tail), static_cast<uint32_t>(LK) * 32, 256, UMMA_LAYOUT_SW32);
#pragma unroll
        for (int k = 0; k < LK / 16; ++k) {
          const uint32_t tP = tS + (k < 8 ? k * 8 : 128 + (k - 8) * 8);   // keys [128,256): P sits at columns [128,192)
          umma_f16_ts(tS + C::O_COL, tP, umma_desc_advance(dv, k * 16 * 128), idesc_o, k > 0 ? 1u : 0u);
          if constexpr (TAIL) umma_f16_ts(tS + C::OT_COL, tP, umma_desc_advance(dvt, k * 16 * 32), idesc_ot, k > 0 ? 1u : 0u);
        }
        umma_commit(o_full + sl);
      };
      // Issue order S_0 .. S_{NSLOT-2}, then (S_{i+NSLOT-1}, PV_i) for every i: the S of a later tile is queued before the
      // P V of the current one, so it runs on the tensor pipe while tile i is still in its softmax.  (A readiness-driven
      // order -- PV first whenever its P is there -- measured SLOWER, 30.7 -> 33.7 us per spatial launch: delaying S starves
      // the other slot's warpgroups more than an early PV helps this one's.)
      for (int j = 0; j < NSLOT - 1 && j < n_items; ++j) issue_s(j);
      for (int i = 0; i < n_items; ++i) {
        if (i + NSLOT - 1 < n_items) issue_s(i + NSLOT - 1);
        issue_pv(i);
      }
    }
  } else if (warp == 2) {
    if (lane == 0) {
      // ------------------------------------------------------------------ output store: staging tile -> global (TMA)
      for (int i = 0; i < n_items; ++i) {
        const int sl = i % NSLOT, u = i / NSLOT;
        const Coord c = coord(i);
        mbar_wait(o_staged + sl, u & 1);
        if (!(p.dbg & 4)) {
          const uint8_t* src = smem + sl * sp.stage_bytes + sp.v_main;
          if constexpr (MODE == MODE_TEMPORAL) tma_store_4d(&tmO, src, 0, c.head, c.c2, c.c3);
          else tma_store_3d(&tmO, src, 0, c.head, c.c2);
          tma_store_commit();
          tma_store_wait_read<0>();
        }
        mbar_arrive(v_free + sl);
      }
      tma_store_wait_all<0>();
    }
  } else {
    // -------------------------------------------------------------------- softmax + epilogue warpgroups
    const int wg = (warp - 4) >> 2;
    const int sl = wg / C::WG_PER_TILE;            // the slot this warpgroup serves
    const int h = wg % C::WG_PER_TILE;             // LK = 256: which 128 key columns
    const int q = warp & 3;                        // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;                   // tile row = TMEM lane
    const uint32_t t_slot = tmem_base + sl * C::SLOT_COLS + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t t_s = t_slot + h * 128;         // my S columns; my P is written over their first 64 columns
    float* xmax = xch + (sl * 4 + 0) * 128;        // [2 halves][128]
    float* xsum = xch + (sl * 4 + 2) * 128;
    float* bias_s = sbias + sl * 128;
    const int bar_id = 1 + sl;
    uint8_t* stage_out = smem + sl * sp.stage_bytes + sp.v_main;
    const int row_bytes = p.hd * 2;

    for (int i = sl; i < n_items; i += NSLOT) {
      const int u = i / NSLOT;
      float sum = 0.f;
      bool have_bias = false;
      const float* prow = nullptr;          // T5: this (head, query row)'s 128 relative-position biases
      if constexpr (MODE == MODE_CROSS) {
        have_bias = p.key_bias != nullptr || p.pos_bias != nullptr;
        if (have_bias) {        // this sample's additive key bias (natural-log units) -> smem, once per tile
          const Coord c = coord(i);
          bias_s[r] = p.key_bias ? __ldg(p.key_bias + static_cast<size_t>(c.c3) * 128 + r) * 1.4426950408889634f : 0.f;
          if (p.pos_bias) prow = p.pos_bias + (static_cast<size_t>(c.head) * 128 + r) * 128;
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        }
      }
      mbar_wait(s_full + sl, u & 1);
      tc_fence_after();

      bool done = false;
      if constexpr (MODE == MODE_TEMPORAL) done = p.group == 8;
      if (done) {
        // ---- one pass: the row's 16 live keys are columns g, g + 8, ..., g = r % 8
        const int g = r & 7;
        float xs[16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t v[32];
          tmem_ld_32x32b_x32(t_s + c * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < 4; ++k) xs[c * 4 + k] = sel8(v + 8 * k, g);
        }
        float mx = xs[0];
#pragma unroll
        for (int k = 1; k < 16; ++k) mx = fmaxf(mx, xs[k]);
        const float ms = mx * p.scale_log2;
        uint32_t pk16[16];
        float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const float e = ex2(fmaf(xs[k], p.scale_log2, -ms));
          part[k & 3] += e;
          pk16[k] = (g & 1) ? pack2<BF16>(0.f, e) : pack2<BF16>(e, 0.f);
        }
        sum = (part[0] + part[1]) + (part[2] + part[3]);
        const int w = g >> 1;   // which of the group's 4 packed words holds the live key
#pragma unroll
        for (int c = 0; c < 4; ++c) {     // 32 key columns = 16 packed words = 4 groups of 4 words
          uint32_t o16[16];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
#pragma unroll
            for (int j = 0; j < 4; ++j) o16[4 * k + j] = (j == w) ? pk16[c * 4 + k] : 0u;
          }
          tmem_st_32x32b_x16(t_s + c * 16, o16);
        }
      } else {
        // ---- two passes over my 128 key columns: row maximum, then P = exp2(s * scale (+ bias) - max)
        const int rkey = MODE == MODE_CROSS ? p.kv_valid : row_key<MODE>(r, p.gshift);
        float mx = -INFINITY;
#pragma unroll 1
        for (int c = 0; c < 4; c += 2) {
          uint32_t va[32], vb[32];
          tmem_ld_32x32b_x32(t_s + c * 32, va);
          tmem_ld_32x32b_x32(t_s + (c + 1) * 32, vb);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            float a = __uint_as_float(va[j]), b = __uint_as_float(vb[j]);
            if constexpr (MODE == MODE_CROSS) {
              if (have_bias) {
                a = fmaf(a, p.scale_log2, bias_s[c * 32 + j]);
                b = fmaf(b, p.scale_log2, bias_s[(c + 1) * 32 + j]);
                if (prow) {
                  a = fmaf(__ldg(prow + c * 32 + j), 1.4426950408889634f, a);
                  b = fmaf(__ldg(prow + (c + 1) * 32 + j), 1.4426950408889634f, b);
                }
              }
            }
            if (key_valid<MODE>(rkey, c * 32 + j, p.gshift)) mx = fmaxf(mx, a);
            if (key_valid<MODE>(rkey, (c + 1) * 32 + j, p.gshift)) mx = fmaxf(mx, b);
          }
        }
        if constexpr (LK == 256) {      // the other warpgroup holds the other half of the row
          xmax[h * 128 + r] = mx;
          asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
          mx = fmaxf(mx, xmax[(h ^ 1) * 128 + r]);
        }
        const float ms = have_bias ? mx : mx * p.scale_log2;
        // Straight-line and wide on purpose: all 16 scores of a chunk are scaled, THEN exponentiated, THEN summed into four
        // independent partial sums -- the FFMA -> MUFU -> FADD chain of one element is ~30 clk deep, so the elements must be
        // independent instructions for the scheduler (round-2 ncu: a per-element branch + one serial sum chain left each
        // softmax warp at one instruction per 5.4 clk).
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
        auto emit = [&](const uint32_t (&v)[16], int c) {
          float x[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            if (MODE == MODE_CROSS && have_bias) {
              x[j] = fmaf(__uint_as_float(v[j]), p.scale_log2, bias_s[c * 16 + j]) - ms;
              if (prow) x[j] = fmaf(__ldg(prow + c * 16 + j), 1.4426950408889634f, x[j]);
            } else {
              x[j] = fmaf(__uint_as_float(v[j]), p.scale_log2, -ms);
            }
          }
          float e[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            // every 4th exponential on the FMA pipe (spatial tiles only: their rows are 256 keys long): balances the
            // 16/clk MUFU pipe against the issue slots the polynomial costs
            if (POLY && (j & 3) == 3) e[j] = ex2_poly(x[j]);
            else e[j] = ex2(x[j]);
            if (!key_valid<MODE>(rkey, c * 16 + j, p.gshift)) e[j] = 0.f;
          }
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) pk[j] = pack2<BF16>(e[2 * j], e[2 * j + 1]);
#pragma unroll
          for (int j = 0; j < 16; ++j) s4[j & 3] += e[j];
          tmem_st_32x32b_x8(t_s + c * 8, pk);
        };
        uint32_t va[16], vb[16];
        tmem_ld_32x32b_x16(t_s, va);
        tmem_ld_wait();
#pragma unroll 1
        for (int c = 0; c < 8; c += 2) {
          tmem_ld_32x32b_x16(t_s + (c + 1) * 16, vb);
          emit(va, c);
          tmem_ld_wait();
          if (c + 2 < 8) tmem_ld_32x32b_x16(t_s + (c + 2) * 16, va);
          emit(vb, c + 1);
          tmem_ld_wait();
        }
        sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
      }
      if constexpr (LK == 256) xsum[h * 128 + r] = sum;
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(p_full + sl);
      if constexpr (LK == 256) {
        asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
        sum += xsum[(h ^ 1) * 128 + r];
      }
      const float inv = 1.0f / sum;

      // ---- epilogue: O * 1/sum -> 16-bit -> dense [128][hd] staging tile in the (dead) V smem of this stage
      mbar_wait(o_full + sl, u & 1);
      tc_fence_after();
      uint8_t* drow = stage_out + r * row_bytes;
      auto put32 = [&](const uint32_t (&o)[32], int col0) {
#pragma unroll
        for (int i4 = 0; i4 < 4; ++i4) {
          uint4 w;
          w.x = pack2<BF16>(__uint_as_float(o[8 * i4 + 0]) * inv, __uint_as_float(o[8 * i4 + 1]) * inv);
          w.y = pack2<BF16>(__uint_as_float(o[8 * i4 + 2]) * inv, __uint_as_float(o[8 * i4 + 3]) * inv);
          w.z = pack2<BF16>(__uint_as_float(o[8 * i4 + 4]) * inv, __uint_as_float(o[8 * i4 + 5]) * inv);
          w.w = pack2<BF16>(__uint_as_float(o[8 * i4 + 6]) * inv, __uint_as_float(o[8 * i4 + 7]) * inv);
          *reinterpret_cast<uint4*>(drow + (col0 + i4 * 8) * 2) = w;
        }
      };
      auto put_tail = [&](const uint32_t (&o)[16]) {
        const int tail8 = (p.hd - 64) / 8;   // 1 (hd 72) or 2 (hd 80)
#pragma unroll
        for (int i4 = 0; i4 < 2; ++i4) {
          if (i4 < tail8) {
            uint4 w;
            w.x = pack2<BF16>(__uint_as_float(o[8 * i4 + 0]) * inv, __uint_as_float(o[8 * i4 + 1]) * inv);
            w.y = pack2<BF16>(__uint_as_float(o[8 * i4 + 2]) * inv, __uint_as_float(o[8 * i4 + 3]) * inv);
            w.z = pack2<BF16>(__uint_as_float(o[8 * i4 + 4]) * inv, __uint_as_float(o[8 * i4 + 5]) * inv);
            w.w = pack2<BF16>(__uint_as_float(o[8 * i4 + 6]) * inv, __uint_as_float(o[8 * i4 + 7]) * inv);
            *reinterpret_cast<uint4*>(drow + (64 + i4 * 8) * 2) = w;
          }
        }
      };
      if constexpr (LK == 256) {
        uint32_t o0[32], ot[16];
        tmem_ld_32x32b_x32(t_slot + C::O_COL + h * 32, o0);
        if (TAIL && h == 0) tmem_ld_32x32b_x16(t_slot + C::OT_COL, ot);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(o_free + sl);
        put32(o0, h * 32);
        if (TAIL && h == 0) put_tail(ot);
      } else {
        uint32_t o0[32], o1[32], ot[16];
        tmem_ld_32x32b_x32(t_slot + C::O_COL, o0);
        tmem_ld_32x32b_x32(t_slot + C::O_COL + 32, o1);
        if constexpr (TAIL) tmem_ld_32x32b_x16(t_slot + C::OT_COL, ot);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(o_free + sl);
        put32(o0, 0);
        put32(o1, 32);
        if constexpr (TAIL) put_tail(ot);
      }
      fence_proxy_async_smem();       // the staging tile is read by the TMA engine
      mbar_arrive(o_staged + sl);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <bool BF16, bool TAIL, int MODE, int LK, bool POLY>
int launch_v3_lk(const CUtensorMap* m, const AttnDev& p, int total, cudaStream_t stream) {
  auto kern = attn_v3_kernel<BF16, TAIL, MODE, LK, POLY>;
  const int smem_bytes = make_v3_plan(LK, TAIL).total;
  B200_SET_SMEM_ONCE(kern, smem_bytes);
  int sms = 148;
  B200_TRY(device_sm_count(&sms));
  const int ctas = total < sms ? total : sms;
  B200_CHECK_CUDA(launch_pdl(kern, dim3(ctas), dim3(V3<LK>::THREADS), static_cast<size_t>(smem_bytes), stream, m[0], m[1], m[2], m[3], m[4], p, total));
  return B200_OK;
}

template <bool BF16, bool TAIL, int MODE>
int launch_v3(const CUtensorMap* m, const AttnDev& p, dim3 grid, cudaStream_t stream) {
  const int total = static_cast<int>(grid.x * grid.y);
  if constexpr (MODE == MODE_FULL) {
    if (p.Lk == 256) {
      if (p.dbg & 16) return launch_v3_lk<BF16, TAIL, MODE, 256, false>(m, p, total, stream);   // A/B: all exponentials on the MUFU pipe
      return launch_v3_lk<BF16, TAIL, MODE, 256, true>(m, p, total, stream);
    }
  }
  return launch_v3_lk<BF16, TAIL, MODE, 128, false>(m, p, total, stream);
}

template <bool BF16, bool TAIL, int MODE>
int launch_pipe(const CUtensorMap* m, const AttnDev& p, dim3 grid, cudaStream_t stream) {
  auto kern = attn_pipe_kernel<BF16, TAIL, MODE>;
  B200_SET_SMEM_ONCE(kern, make_pipe_plan(256, true).total);
  const int smem_bytes = make_pipe_plan(p.Lk, TAIL).total;
  const int total = static_cast<int>(grid.x * grid.y);
  int sms = 148;
  B200_TRY(device_sm_count(&sms));
  const int ctas = total < sms ? total : sms;
  B200_CHECK_CUDA(launch_pdl(kern, dim3(ctas), dim3(kPipeThreads), static_cast<size_t>(smem_bytes), stream, m[0], m[1], m[2], m[3], p, total));
  return B200_OK;
}

template <bool BF16, bool TAIL, int MODE>
int launch_mode(const CUtensorMap* m, const AttnDev& p, dim3 grid, cudaStream_t stream) {
  // B200_ATTN_IMPL: 3 = v3 (role warps, 2 warpgroups per 256-key tile / 3 tiles in flight, TMA-stored output),
  //                 2 = the round-1 two-tile pipeline (A/B switch)
  static const int env_impl = env_int("B200_ATTN_IMPL", kAttnDefaultImpl);
  const int forced = g_attn_impl;
  const int impl = forced ? forced : env_impl;
  if (impl == 2) return launch_pipe<BF16, TAIL, MODE>(m, p, grid, stream);
  return launch_v3<BF16, TAIL, MODE>(m, p, grid, stream);
}

// ------------------------------------------------------------------------------------------------------------------
// Long spatial sequences (N = 512 / 1024 tokens per frame: LatteT2V at 512 px): the keys are streamed in chunks of 256
// with the online-softmax recurrence.  S_c = Q K_c^T lands in TMEM columns [0,256); the softmax warps take the chunk
// maximum, rescale the running output O (TMEM columns [256,336), tcgen05.ld -> * alpha -> tcgen05.st) and the running
// sum, write P_c (16-bit, K-major SW128) to smem; O += P_c V_c accumulates in TMEM.  K_{c+1} is fetched as soon as
// S_c has been computed, V_{c+1} as soon as O += P_c V_c has been computed.
constexpr int L_SQ_MAIN = 0;
constexpr int L_SK_MAIN = L_SQ_MAIN + 128 * 128;
constexpr int L_SV_MAIN = L_SK_MAIN + 256 * 128;
constexpr int L_SP = L_SV_MAIN + 256 * 128;
constexpr int L_SQ_TAIL = L_SP + 128 * 256 * 2;
constexpr int L_SK_TAIL = L_SQ_TAIL + 128 * 32;
constexpr int L_SV_TAIL = L_SK_TAIL + 256 * 32;
constexpr int L_SBARS = L_SV_TAIL + 256 * 32;
constexpr int L_SMEM_BYTES = L_SBARS + 128 + 1024;
constexpr int L_OCOL = 256;

template <bool BF16, bool TAIL>
__global__ void __launch_bounds__(kThreads, 1)
attn_long_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmQt,
                 const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmKVt, const AttnDev p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L_SBARS);
  uint64_t* bar_q = bars + 0;
  uint64_t* bar_k = bars + 1;
  uint64_t* bar_v = bars + 2;
  uint64_t* bar_s = bars + 3;
  uint64_t* bar_p = bars + 4;
  uint64_t* bar_o = bars + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tile = blockIdx.x;
  const int head = blockIdx.y;
  const int nchunk = p.tokens / 256;
  const int seq = tile / p.tiles_per_seq;
  const int kv_row0 = seq * p.tokens;
  const int q_row0 = kv_row0 + (tile % p.tiles_per_seq) * 128;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    mbar_init(bar_q, 1);
    mbar_init(bar_k, 1);
    mbar_init(bar_v, 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_p, 128);
    mbar_init(bar_o, 1);
    fence_mbar_init();
  }
  if (warp == 4) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 4) {
    if (lane == 0) {
      const uint32_t k_bytes = 256 * 128 + (TAIL ? 256 * 32 : 0);
      auto load_k = [&](int c) {
        mbar_arrive_expect_tx(bar_k, k_bytes);
        tma_load_3d(smem + L_SK_MAIN, &tmKV, bar_k, 0, p.k_head0 + head, kv_row0 + c * 256);
        if constexpr (TAIL) tma_load_3d(smem + L_SK_TAIL, &tmKVt, bar_k, 64, p.k_head0 + head, kv_row0 + c * 256);
      };
      auto load_v = [&](int c) {
        mbar_arrive_expect_tx(bar_v, k_bytes);
        tma_load_3d(smem + L_SV_MAIN, &tmKV, bar_v, 0, p.v_head0 + head, kv_row0 + c * 256);
        if constexpr (TAIL) tma_load_3d(smem + L_SV_TAIL, &tmKVt, bar_v, 64, p.v_head0 + head, kv_row0 + c * 256);
      };
      mbar_arrive_expect_tx(bar_q, 128 * 128 + (TAIL ? 128 * 32 : 0));
      tma_load_3d(smem + L_SQ_MAIN, &tmQ, bar_q, 0, head, q_row0);
      if constexpr (TAIL) tma_load_3d(smem + L_SQ_TAIL, &tmQt, bar_q, 64, head, q_row0);
      load_k(0);
      load_v(0);

      const uint32_t idesc_s = umma_idesc_f16(BF16, 128, 256, false, false);
      const uint32_t idesc_o = umma_idesc_f16(BF16, 128, 64, false, true);
      const uint32_t idesc_ot = umma_idesc_f16(BF16, 128, 16, false, true);
      const uint64_t dq = umma_smem_desc(smem_u32(smem + L_SQ_MAIN), 0, 1024, UMMA_LAYOUT_SW128);
      const uint64_t dk = umma_smem_desc(smem_u32(smem + L_SK_MAIN), 0, 1024, UMMA_LAYOUT_SW128);
      const uint64_t dqt = umma_smem_desc(smem_u32(smem + L_SQ_TAIL), 0, 256, UMMA_LAYOUT_SW32);
      const uint64_t dkt = umma_smem_desc(smem_u32(smem + L_SK_TAIL), 0, 256, UMMA_LAYOUT_SW32);
      const uint64_t dv = umma_smem_desc(smem_u32(smem + L_SV_MAIN), 256 * 128, 1024, UMMA_LAYOUT_SW128);
      const uint64_t dvt = umma_smem_desc(smem_u32(smem + L_SV_TAIL), 256 * 32, 256, UMMA_LAYOUT_SW32);
      mbar_wait(bar_q, 0);
      for (int c = 0; c < nchunk; ++c) {
        const uint32_t par = c & 1;
        mbar_wait(bar_k, par);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_f16_ss(tmem_base, umma_desc_advance(dq, k * 32), umma_desc_advance(dk, k * 32), idesc_s, k > 0 ? 1u : 0u);
        if constexpr (TAIL) umma_f16_ss(tmem_base, dqt, dkt, idesc_s, 1u);
        umma_commit(bar_s);
        mbar_wait(bar_s, par);                 // S_c computed: the K buffer is free
        if (c + 1 < nchunk) load_k(c + 1);
        mbar_wait(bar_v, par);
        mbar_wait(bar_p, par);                 // P_c written, O rescaled
        tc_fence_after();
        for (int k = 0; k < 16; ++k) {
          const uint64_t dp = umma_smem_desc(smem_u32(smem + L_SP + (k >> 2) * (128 * 128)) + (k & 3) * 32, 0, 1024, UMMA_LAYOUT_SW128);
          const uint32_t accum = (c > 0 || k > 0) ? 1u : 0u;
          umma_f16_ss(tmem_base + L_OCOL, dp, umma_desc_advance(dv, k * 16 * 128), idesc_o, accum);
          if constexpr (TAIL) umma_f16_ss(tmem_base + L_OCOL + 64, dp, umma_desc_advance(dvt, k * 16 * 32), idesc_ot, accum);
        }
        umma_commit(bar_o);
        if (c + 1 < nchunk) {
          mbar_wait(bar_o, par);               // O += P_c V_c computed: the V buffer (and P) are free
          load_v(c + 1);
        }
      }
    }
  } else {
    const int r = warp * 32 + lane;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    float m_run = -INFINITY, l_run = 0.f;
    uint8_t* prow = smem + L_SP + r * 128;
    const int sw = r & 7;
    for (int c = 0; c < nchunk; ++c) {
      const uint32_t par = c & 1;
      mbar_wait(bar_s, par);
      tc_fence_after();
      float cmax = -INFINITY;
      for (int j8 = 0; j8 < 8; ++j8) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(t_row + j8 * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) cmax = fmaxf(cmax, __uint_as_float(v[j]));
      }
      const float m_new = fmaxf(m_run, cmax);
      const float alpha = ex2((m_run - m_new) * p.scale_log2);   // 0 for the first chunk (m_run = -inf)
      l_run *= alpha;
      m_run = m_new;
      if (c > 0) {
        mbar_wait(bar_o, (c - 1) & 1);          // O += P_{c-1} V_{c-1} has completed: O and the P buffer are ours again
        tc_fence_after();
#pragma unroll 1
        for (int cc = 0; cc < (TAIL ? 5 : 4); ++cc) {
          uint32_t v[16];
          tmem_ld_32x32b_x16(t_row + L_OCOL + cc * 16, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) * alpha);
          tmem_st_32x32b_x16(t_row + L_OCOL + cc * 16, v);
        }
        tmem_st_wait();
      }
      const float mscaled = m_new * p.scale_log2;
      for (int j8 = 0; j8 < 8; ++j8) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(t_row + j8 * 32, v);
        tmem_ld_wait();
        float e[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          e[j] = ex2(fmaf(__uint_as_float(v[j]), p.scale_log2, -mscaled));
          l_run += e[j];
        }
        uint8_t* atom = prow + (j8 >> 1) * (128 * 128);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint4 o;
          o.x = pack2<BF16>(e[8 * i + 0], e[8 * i + 1]);
          o.y = pack2<BF16>(e[8 * i + 2], e[8 * i + 3]);
          o.z = pack2<BF16>(e[8 * i + 4], e[8 * i + 5]);
          o.w = pack2<BF16>(e[8 * i + 6], e[8 * i + 7]);
          const int chunk = ((j8 & 1) * 4 + i) ^ sw;
          *reinterpret_cast<uint4*>(atom + chunk * 16) = o;
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(bar_p);
    }
    const long long out_row = q_row0 + r;
    uint16_t* optr = reinterpret_cast<uint16_t*>(p.out) + out_row * p.D + head * p.hd;
    const float inv = 1.0f / l_run;
    mbar_wait(bar_o, (nchunk - 1) & 1);
    tc_fence_after();
#pragma unroll 1
    for (int c2 = 0; c2 < 2; ++c2) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(t_row + L_OCOL + c2 * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint4 o;
        o.x = pack2<BF16>(__uint_as_float(v[8 * i + 0]) * inv, __uint_as_float(v[8 * i + 1]) * inv);
        o.y = pack2<BF16>(__uint_as_float(v[8 * i + 2]) * inv, __uint_as_float(v[8 * i + 3]) * inv);
        o.z = pack2<BF16>(__uint_as_float(v[8 * i + 4]) * inv, __uint_as_float(v[8 * i + 5]) * inv);
        o.w = pack2<BF16>(__uint_as_float(v[8 * i + 6]) * inv, __uint_as_float(v[8 * i + 7]) * inv);
        *reinterpret_cast<uint4*>(optr + c2 * 32 + i * 8) = o;
      }
    }
    if constexpr (TAIL) {
      uint32_t v[16];
      tmem_ld_32x32b_x16(t_row + L_OCOL + 64, v);
      tmem_ld_wait();
      const int tail8 = (p.hd - 64) / 8;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        if (i >= tail8) break;
        uint4 o;
        o.x = pack2<BF16>(__uint_as_float(v[8 * i + 0]) * inv, __uint_as_float(v[8 * i + 1]) * inv);
        o.y = pack2<BF16>(__uint_as_float(v[8 * i + 2]) * inv, __uint_as_float(v[8 * i + 3]) * inv);
        o.z = pack2<BF16>(__uint_as_float(v[8 * i + 4]) * inv, __uint_as_float(v[8 * i + 5]) * inv);
        o.w = pack2<BF16>(__uint_as_float(v[8 * i + 6]) * inv, __uint_as_float(v[8 * i + 7]) * inv);
        *reinterpret_cast<uint4*>(optr + 64 + i * 8) = o;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <bool BF16, bool TAIL>
int launch_long(const CUtensorMap* m, const AttnDev& p, dim3 grid, cudaStream_t stream) {
  auto kern = attn_long_kernel<BF16, TAIL>;
  B200_SET_SMEM_ONCE(kern, L_SMEM_BYTES);
  B200_CHECK_CUDA(launch_pdl(kern, grid, dim3(kThreads), static_cast<size_t>(L_SMEM_BYTES), stream, m[0], m[1], m[2], m[3], p));
  return B200_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Long spatial sequences (N = 512 / 1024 tokens per frame: LatteT2V at 512 px), round 2: a persistent, role-warp,
// online-softmax kernel in the shape of the v3 kernel above.
//   * work item = (frame, head, 256 query rows) = TWO 128-row query tiles that share every K/V byte the item streams;
//     keys arrive in chunks of 128 through a 3-stage TMA ring {K, V};
//   * TMEM: S_0 [0,128)  S_1 [128,256)  O_0 [256,336)  O_1 [336,416).  P_t (16-bit, packed) overwrites the start of S_t;
//   * MMA issue order S_0(0) S_1(0) | PV_0(c) S_0(c+1) PV_1(c) S_1(c+1) | ...: while warpgroup 0 exponentiates S_0(c) the
//     tensor pipe computes S_1(c) and P_1 V of the previous chunk -- two tiles ping-pong on one pipe;
//   * online softmax with a LAZY running maximum: the row maximum m only moves (and O_t, l are rescaled, tcgen05.ld ->
//     * alpha -> tcgen05.st) when the new chunk's maximum exceeds it by more than 2^8; until then P may grow up to 256,
//     which 16-bit P and the fp32 accumulators hold exactly as well.  The rescale of a warp's 32 rows is skipped when no
//     row needs it (warp vote), which is nearly always after the first chunks;
//   * the epilogue stages O_t / l into the item's (dead) Q tile and leaves through one TMA bulk store per tile.
// Warps: 0 = TMA producer K/V ring, 3 = TMA producer Q, 1 = MMA issuer (+ TMEM allocator), 2 = output store,
//        4-7 = softmax/epilogue tile 0, 8-11 = tile 1.
constexpr int ST_THREADS = 384;
constexpr int ST_NST = 3;            // K/V ring depth
constexpr int ST_CK = 128;           // keys per chunk
constexpr float ST_TAU = 8.0f;       // lazy-maximum threshold, log2 units

struct StPlan {
  int q_buf, q_tile, q_tail, kv_stage, k_main, k_tail, v_main, v_tail, ring, bars, total;
};
__host__ __device__ inline StPlan make_st_plan(bool tail) {
  StPlan s;
  s.q_tile = 128 * 128 + (tail ? 128 * 32 : 0);     // one 128-row query tile (main + tail), also its output staging tile
  s.q_tail = 128 * 128;
  s.q_buf = 2 * s.q_tile;                           // Q_0, Q_1 of one item
  s.k_main = 0;
  s.k_tail = ST_CK * 128;
  s.v_main = s.k_tail + (tail ? ST_CK * 32 : 0);
  s.v_tail = s.v_main + ST_CK * 128;
  s.kv_stage = s.v_tail + (tail ? ST_CK * 32 : 0);
  s.ring = 2 * s.q_buf;
  s.bars = s.ring + ST_NST * s.kv_stage;
  s.total = s.bars + 512 + 1024;
  return s;
}

template <bool BF16, bool TAIL>
__global__ void __launch_bounds__(ST_THREADS, 1)
attn_stream_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmQt,
                   const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmKVt,
                   const __grid_constant__ CUtensorMap tmO, const AttnDev p, const int total_items) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const StPlan sp = make_st_plan(TAIL);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + sp.bars);
  uint64_t* q_full = bars + 0;              // [2] TMA: both query tiles of the item have landed
  uint64_t* q_free = bars + 2;              // [2] store warp (2 arrivals): both output tiles have left the Q buffer
  uint64_t* k_full = bars + 4;              // [NST]
  uint64_t* v_full = bars + 4 + ST_NST;     // [NST]
  uint64_t* k_free = bars + 4 + 2 * ST_NST; // [NST] MMA commit: S_1 of the chunk is done
  uint64_t* v_free = bars + 4 + 3 * ST_NST; // [NST] MMA commit: P_1 V of the chunk is done
  uint64_t* s_full = bars + 4 + 4 * ST_NST; // [2] MMA commit: S_t of a chunk is complete (and every earlier MMA)
  uint64_t* p_full = s_full + 2;            // [2] softmax (128 arrivals): P_t written, O_t rescaled
  uint64_t* o_full = s_full + 4;            // [2] MMA commit: O_t of the item is complete
  uint64_t* o_free = s_full + 6;            // [2] epilogue (128 arrivals): O_t has been read out of TMEM
  uint64_t* o_staged = s_full + 8;          // [2] epilogue (128 arrivals): the output tile is staged
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_full + 10);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int H = p.heads;
  const int C = p.tokens / ST_CK;                    // chunks per item
  const int pairs_per_seq = p.tokens / 256;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 2; ++i) {
      mbar_init(q_full + i, 1);
      mbar_init(q_free + i, 2);
      mbar_init(s_full + i, 1);
      mbar_init(p_full + i, 128);
      mbar_init(o_full + i, 1);
      mbar_init(o_free + i, 128);
      mbar_init(o_staged + i, 128);
    }
    for (int i = 0; i < ST_NST; ++i) {
      mbar_init(k_full + i, 1);
      mbar_init(v_full + i, 1);
      mbar_init(k_free + i, 1);
      mbar_init(v_free + i, 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  const int first = blockIdx.x, step = gridDim.x;
  const int n_items = first < total_items ? (total_items - first + step - 1) / step : 0;
  struct Coord { int head, q_row0, kv_row0; };
  auto coord = [&](int n) {
    const int item = first + n * step;
    Coord c;
    c.head = item % H;
    const int qp = item / H;                       // (sequence, query pair)
    c.kv_row0 = (qp / pairs_per_seq) * p.tokens;
    c.q_row0 = c.kv_row0 + (qp % pairs_per_seq) * 256;
    return c;
  };

  if (warp == 3) {
    if (lane == 0) {
      // ------------------------------------------------------------------ TMA producer: the item's two query tiles
      const uint32_t q_bytes = 2 * (128 * 128 + (TAIL ? 128 * 32 : 0));
      for (int n = 0; n < n_items; ++n) {
        const int b = n & 1, u = n >> 1;
        uint8_t* buf = smem + b * sp.q_buf;
        const Coord c = coord(n);
        if (u > 0) mbar_wait(q_free + b, (u - 1) & 1);
        mbar_arrive_expect_tx(q_full + b, q_bytes);
        for (int t = 0; t < 2; ++t) {
          tma_load_3d(buf + t * sp.q_tile, &tmQ, q_full + b, 0, c.head, c.q_row0 + t * 128);
          if constexpr (TAIL) tma_load_3d(buf + t * sp.q_tile + sp.q_tail, &tmQt, q_full + b, 64, c.head, c.q_row0 + t * 128);
        }
      }
    }
  } else if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------------ TMA producer: K / V chunk ring
      const uint32_t kb = ST_CK * 128 + (TAIL ? ST_CK * 32 : 0);
      int g = 0;
      for (int n = 0; n < n_items; ++n) {
        const Coord c = coord(n);
        for (int ch = 0; ch < C; ++ch, ++g) {
          const int st = g % ST_NST, u = g / ST_NST;
          uint8_t* buf = smem + sp.ring + st * sp.kv_stage;
          const int row = c.kv_row0 + ch * ST_CK;
          if (u > 0) mbar_wait(k_free + st, (u - 1) & 1);
          mbar_arrive_expect_tx(k_full + st, kb);
          tma_load_3d(buf + sp.k_main, &tmKV, k_full + st, 0, p.k_head0 + c.head, row);
          if constexpr (TAIL) tma_load_3d(buf + sp.k_tail, &tmKVt, k_full + st, 64, p.k_head0 + c.head, row);
          if (u > 0) mbar_wait(v_free + st, (u - 1) & 1);
          mbar_arrive_expect_tx(v_full + st, kb);
          tma_load_3d(buf + sp.v_main, &tmKV, v_full + st, 0, p.v_head0 + c.head, row);
          if constexpr (TAIL) tma_load_3d(buf + sp.v_tail, &tmKVt, v_full + st, 64, p.v_head0 + c.head, row);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ------------------------------------------------------------------ MMA issuer
      constexpr uint32_t idesc_s = umma_idesc_f16(BF16, 128, ST_CK, false, false);
      constexpr uint32_t idesc_o = umma_idesc_f16(BF16, 128, 64, false, true);    // B = V is MN-major ([key][hd] in smem)
      constexpr uint32_t idesc_ot = umma_idesc_f16(BF16, 128, 16, false, true);
      int g = 0;                                   // global chunk counter (ring position)
      uint32_t sp_phase = 0;                       // phase of s_full / p_full: one completion per chunk, both tiles in step
      auto issue_s = [&](const uint8_t* qbuf, const uint8_t* kbuf, int t) {
        const uint32_t tS = tmem_base + t * 128;
        const uint64_t dq = umma_smem_desc(smem_u32(qbuf + t * sp.q_tile), 0, 1024, UMMA_LAYOUT_SW128);
        const uint64_t dk = umma_smem_desc(smem_u32(kbuf + sp.k_main), 0, 1024, UMMA_LAYOUT_SW128);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_f16_ss(tS, umma_desc_advance(dq, k * 32), umma_desc_advance(dk, k * 32), idesc_s, k > 0 ? 1u : 0u);
        if constexpr (TAIL) {
          const uint64_t dqt = umma_smem_desc(smem_u32(qbuf + t * sp.q_tile + sp.q_tail), 0, 256, UMMA_LAYOUT_SW32);
          const uint64_t dkt = umma_smem_desc(smem_u32(kbuf + sp.k_tail), 0, 256, UMMA_LAYOUT_SW32);
          umma_f16_ss(tS, dqt, dkt, idesc_s, 1u);
        }
        umma_commit(s_full + t);
      };
      auto issue_pv = [&](const uint8_t* vbuf, int t, bool first_chunk) {
        const uint32_t tP = tmem_base + t * 128;
        const uint32_t tO = tmem_base + 256 + t * 80;
        const uint64_t dv = umma_smem_desc(smem_u32(vbuf + sp.v_main), ST_CK * 128, 1024, UMMA_LAYOUT_SW128);
        const uint64_t dvt = umma_smem_desc(smem_u32(vbuf + sp.v_tail), ST_CK * 32, 256, UMMA_LAYOUT_SW32);
#pragma unroll
        for (int k = 0; k < ST_CK / 16; ++k) {
          const uint32_t acc = (first_chunk && k == 0) ? 0u : 1u;
          umma_f16_ts(tO, tP + k * 8, umma_desc_advance(dv, k * 16 * 128), idesc_o, acc);
          if constexpr (TAIL) umma_f16_ts(tO + 64, tP + k * 8, umma_desc_advance(dvt, k * 16 * 32), idesc_ot, acc);
        }
      };
      for (int n = 0; n < n_items; ++n) {
        const int qb = n & 1;
        const uint8_t* qbuf = smem + qb * sp.q_buf;
        mbar_wait(q_full + qb, (n >> 1) & 1);
        {   // S_0(0), S_1(0)
          const int st = g % ST_NST;
          const uint8_t* kv = smem + sp.ring + st * sp.kv_stage;
          mbar_wait(k_full + st, (g / ST_NST) & 1);
          tc_fence_after();
          issue_s(qbuf, kv, 0);
          issue_s(qbuf, kv, 1);
          umma_commit(k_free + st);
        }
        for (int ch = 0; ch < C; ++ch, ++g) {
          const int st = g % ST_NST;
          const uint8_t* kv = smem + sp.ring + st * sp.kv_stage;
          const int st_n = (g + 1) % ST_NST;
          const uint8_t* kv_n = smem + sp.ring + st_n * sp.kv_stage;
          const bool more = ch + 1 < C;
          mbar_wait(v_full + st, (g / ST_NST) & 1);
          if (more) mbar_wait(k_full + st_n, ((g + 1) / ST_NST) & 1);
          for (int t = 0; t < 2; ++t) {
            if (ch == 0 && n > 0) mbar_wait(o_free + t, (n - 1) & 1);   // the previous item's O_t has been read out
            mbar_wait(p_full + t, sp_phase);
            tc_fence_after();
            issue_pv(kv, t, ch == 0);
            if (more) issue_s(qbuf, kv_n, t);        // S_t(c+1) overwrites P_t(c): queued behind the P V that reads it
            else umma_commit(o_full + t);
          }
          umma_commit(v_free + st);
          if (more) umma_commit(k_free + st_n);
          sp_phase ^= 1;
        }
      }
    }
  } else if (warp == 2) {
    if (lane == 0) {
      // ------------------------------------------------------------------ output store
      for (int n = 0; n < n_items; ++n) {
        const int qb = n & 1;
        const Coord c = coord(n);
        for (int t = 0; t < 2; ++t) {
          mbar_wait(o_staged + t, n & 1);
          if (!(p.dbg & 4)) {
            tma_store_3d(&tmO, smem + qb * sp.q_buf + t * sp.q_tile, 0, c.head, c.q_row0 + t * 128);
            tma_store_commit();
            tma_store_wait_read<0>();
          }
          mbar_arrive(q_free + qb);
        }
      }
      tma_store_wait_all<0>();
    }
  } else {
    // -------------------------------------------------------------------- softmax + epilogue: warpgroup t owns query tile t
    const int t = (warp - 4) >> 2;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t t_s = tmem_base + t * 128 + lane_off;
    const uint32_t t_o = tmem_base + 256 + t * 80 + lane_off;
    const int row_bytes = p.hd * 2;
    uint32_t phase = 0;
    for (int n = 0; n < n_items; ++n) {
      float m_run = -INFINITY, l_run = 0.f;      // running maximum (raw score units) and sum, this thread's row
      for (int ch = 0; ch < C; ++ch) {
        mbar_wait(s_full + t, phase);
        tc_fence_after();
        // pass 1: chunk maximum
        float mx = -INFINITY;
#pragma unroll 1
        for (int c = 0; c < 4; c += 2) {
          uint32_t va[32], vb[32];
          tmem_ld_32x32b_x32(t_s + c * 32, va);
          tmem_ld_32x32b_x32(t_s + (c + 1) * 32, vb);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) mx = fmaxf(mx, fmaxf(__uint_as_float(va[j]), __uint_as_float(vb[j])));
        }
        // lazy running maximum: move it only when this chunk exceeds it by more than 2^TAU
        float alpha = 1.0f;
        const bool grow = (mx - m_run) * p.scale_log2 > ST_TAU;      // always true for the first chunk (m_run = -inf)
        if (grow) {
          alpha = ch == 0 ? 0.f : ex2((m_run - mx) * p.scale_log2);
          m_run = mx;
        }
        if (ch > 0 && __any_sync(0xffffffffu, grow)) {               // O_t is stable: every MMA before S_t(ch) has completed
          l_run *= alpha;
#pragma unroll 1
          for (int cc = 0; cc < (TAIL ? 5 : 4); ++cc) {
            uint32_t v[16];
            tmem_ld_32x32b_x16(t_o + cc * 16, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) * alpha);
            tmem_st_32x32b_x16(t_o + cc * 16, v);
          }
        }
        const float ms = m_run * p.scale_log2;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
        auto emit = [&](const uint32_t (&v)[16], int c) {
          float e[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float x = fmaf(__uint_as_float(v[j]), p.scale_log2, -ms);
            e[j] = (j & 3) == 3 ? ex2_poly(x) : ex2(x);        // x <= TAU: ex2_poly handles positive arguments too
          }
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) pk[j] = pack2<BF16>(e[2 * j], e[2 * j + 1]);
#pragma unroll
          for (int j = 0; j < 16; ++j) s4[j & 3] += e[j];
          tmem_st_32x32b_x8(t_s + c * 8, pk);
        };
        uint32_t va[16], vb[16];
        tmem_ld_32x32b_x16(t_s, va);
        tmem_ld_wait();
#pragma unroll 1
        for (int c = 0; c < 8; c += 2) {
          tmem_ld_32x32b_x16(t_s + (c + 1) * 16, vb);
          emit(va, c);
          tmem_ld_wait();
          if (c + 2 < 8) tmem_ld_32x32b_x16(t_s + (c + 2) * 16, va);
          emit(vb, c + 1);
          tmem_ld_wait();
        }
        l_run += (s4[0] + s4[1]) + (s4[2] + s4[3]);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(p_full + t);
        phase ^= 1;
      }
      // ---- epilogue of the item: O_t / l -> 16-bit -> staging tile (the item's Q_t smem) -> TMA store by warp 2
      const float inv = 1.0f / l_run;
      mbar_wait(o_full + t, n & 1);
      tc_fence_after();
      uint32_t o0[32], o1[32], ot[16];
      tmem_ld_32x32b_x32(t_o, o0);
      tmem_ld_32x32b_x32(t_o + 32, o1);
      if constexpr (TAIL) tmem_ld_32x32b_x16(t_o + 64, ot);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(o_free + t);
      uint8_t* drow = smem + (n & 1) * sp.q_buf + t * sp.q_tile + r * row_bytes;
      auto put8 = [&](const uint32_t* o, int col) {
        uint4 w;
        w.x = pack2<BF16>(__uint_as_float(o[0]) * inv, __uint_as_float(o[1]) * inv);
        w.y = pack2<BF16>(__uint_as_float(o[2]) * inv, __uint_as_float(o[3]) * inv);
        w.z = pack2<BF16>(__uint_as_float(o[4]) * inv, __uint_as_float(o[5]) * inv);
        w.w = pack2<BF16>(__uint_as_float(o[6]) * inv, __uint_as_float(o[7]) * inv);
        *reinterpret_cast<uint4*>(drow + col * 2) = w;
      };
#pragma unroll
      for (int i4 = 0; i4 < 4; ++i4) { put8(o0 + 8 * i4, i4 * 8); put8(o1 + 8 * i4, 32 + i4 * 8); }
      if constexpr (TAIL) {
        const int tail8 = (p.hd - 64) / 8;
#pragma unroll
        for (int i4 = 0; i4 < 2; ++i4)
          if (i4 < tail8) put8(ot + 8 * i4, 64 + i4 * 8);
      }
      fence_proxy_async_smem();
      mbar_arrive(o_staged + t);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <bool BF16, bool TAIL>
int launch_stream(const CUtensorMap* m, const AttnDev& p, int total_items, cudaStream_t stream) {
  auto kern = attn_stream_kernel<BF16, TAIL>;
  const int smem_bytes = make_st_plan(TAIL).total;
  B200_SET_SMEM_ONCE(kern, smem_bytes);
  int sms = 148;
  B200_TRY(device_sm_count(&sms));
  const int ctas = total_items < sms ? total_items : sms;
  B200_CHECK_CUDA(launch_pdl(kern, dim3(ctas), dim3(ST_THREADS), static_cast<size_t>(smem_bytes), stream, m[0], m[1], m[2], m[3], m[4], p, total_items));
  return B200_OK;
}

template <bool BF16, bool TAIL>
int launch_tail(int mode, const CUtensorMap* m, const AttnDev& p, dim3 grid, cudaStream_t s) {
  switch (mode) {
    case MODE_FULL: return launch_mode<BF16, TAIL, MODE_FULL>(m, p, grid, s);
    case MODE_PACKED: return launch_mode<BF16, TAIL, MODE_PACKED>(m, p, grid, s);
    case MODE_CROSS: return launch_mode<BF16, TAIL, MODE_CROSS>(m, p, grid, s);
    default: return launch_mode<BF16, TAIL, MODE_TEMPORAL>(m, p, grid, s);
  }
}

}  // namespace

int set_attention_impl(int impl) {
  B200_REQUIRE(impl == 0 || impl == 2 || impl == 3, B200_ERR_UNSUPPORTED, "attention implementation %d unknown (0 default, 2, 3)", impl);
  g_attn_impl = impl;
  return B200_OK;
}

int launch_attention(const AttnArgs& a, cudaStream_t stream) {
  B200_REQUIRE(a.batch > 0 && a.frames > 0 && a.tokens > 0 && a.heads > 0, B200_ERR_SHAPE, "attention: bad shape");
  B200_REQUIRE(a.head_dim == 64 || a.head_dim == 72 || a.head_dim == 80, B200_ERR_UNSUPPORTED,
               "attention: head_dim %d unsupported (64, 72, 80)", a.head_dim);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(a.qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(a.out) & 15) == 0,
               B200_ERR_ALIGN, "attention: qkv/out must be 16-byte aligned");
  B200_TRY(check_arch());
  const int H = a.heads, hd = a.head_dim, D = H * hd;
  const long long T = static_cast<long long>(a.batch) * a.frames * a.tokens;
  const bool tail = hd > 64;

  AttnDev p;
  p.out = a.out;
  p.T = static_cast<int>(T);
  p.D = D;
  p.heads = H;
  p.hd = hd;
  p.tokens = a.tokens;
  p.frames = a.frames;
  p.scale_log2 = (1.0f / sqrtf(static_cast<float>(hd))) * 1.4426950408889634f;
  static const int dbg = env_int("B200_ATTN_DBG", 0);
  p.dbg = dbg;
  p.key_bias = nullptr;
  p.pos_bias = nullptr;
  p.kv_valid = 0;

  p.group = 1;
  p.gshift = 0;
  p.k_head0 = H;
  p.v_head0 = 2 * H;
  p.kv_rows_per_batch = 0;
  p.q_rows_per_batch = 1;
  auto ilog2 = [](int v) { int s = 0; while ((1 << s) < v) ++s; return s; };

  CUtensorMap maps[5];
  int mode;
  dim3 grid;
  if (!a.temporal) {
    const uint64_t dims[3] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(3 * H), static_cast<uint64_t>(T)};
    const uint64_t str[2] = {static_cast<uint64_t>(hd) * 2, static_cast<uint64_t>(3 * D) * 2};
    uint32_t kv_rows;
    if (a.tokens > 256) {
      B200_REQUIRE(a.tokens % 256 == 0, B200_ERR_UNSUPPORTED, "attention: spatial sequence length %d must be a multiple of 256", a.tokens);
      static const int env_impl = env_int("B200_ATTN_IMPL", kAttnDefaultImpl);
      const int forced = g_attn_impl;
      const bool streaming = (forced ? forced : env_impl) != 2;     // impl 2 = the round-1 one-tile-per-CTA kernel (A/B)
      p.Lk = 256;
      p.tiles_per_seq = a.tokens / 128;
      const uint32_t kv_rows = streaming ? 128u : 256u;
      const uint32_t boxQ[3] = {64, 1, 128}, boxQt[3] = {16, 1, 128};
      const uint32_t boxK[3] = {64, 1, kv_rows}, boxKt[3] = {16, 1, kv_rows};
      B200_TRY(make_tmap_16bit(&maps[0], a.qkv, 3, dims, str, boxQ, TMAP_SW_128));
      B200_TRY(make_tmap_16bit(&maps[2], a.qkv, 3, dims, str, boxK, TMAP_SW_128));
      if (tail) {
        B200_TRY(make_tmap_16bit(&maps[1], a.qkv, 3, dims, str, boxQt, TMAP_SW_32));
        B200_TRY(make_tmap_16bit(&maps[3], a.qkv, 3, dims, str, boxKt, TMAP_SW_32));
      } else {
        maps[1] = maps[0];
        maps[3] = maps[2];
      }
      if (streaming) {
        const uint64_t odims[3] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(H), static_cast<uint64_t>(T)};
        const uint64_t ostr[2] = {static_cast<uint64_t>(hd) * 2, static_cast<uint64_t>(D) * 2};
        const uint32_t obox[3] = {static_cast<uint32_t>(hd), 1, 128};
        B200_TRY(make_tmap_16bit(&maps[4], a.out, 3, odims, ostr, obox, TMAP_SW_NONE));
        const int items = a.batch * a.frames * (a.tokens / 256) * H;
        if (a.bf16) return tail ? launch_stream<true, true>(maps, p, items, stream) : launch_stream<true, false>(maps, p, items, stream);
        return tail ? launch_stream<false, true>(maps, p, items, stream) : launch_stream<false, false>(maps, p, items, stream);
      }
      const dim3 lgrid(a.batch * a.frames * p.tiles_per_seq, H);
      if (a.bf16) return tail ? launch_long<true, true>(maps, p, lgrid, stream) : launch_long<true, false>(maps, p, lgrid, stream);
      return tail ? launch_long<false, true>(maps, p, lgrid, stream) : launch_long<false, false>(maps, p, lgrid, stream);
    }
    if (a.tokens >= 128) {
      B200_REQUIRE(a.tokens == 128 || a.tokens == 256, B200_ERR_UNSUPPORTED,
                   "attention: spatial sequence length %d unsupported (<=64 power of two, 128, 256, multiples of 256)", a.tokens);
      mode = MODE_FULL;
      p.Lk = a.tokens;
      p.tiles_per_seq = a.tokens / 128;
      kv_rows = a.tokens;
      grid = dim3(a.batch * a.frames * p.tiles_per_seq, H);
    } else {
      B200_REQUIRE(128 % a.tokens == 0, B200_ERR_UNSUPPORTED, "attention: spatial sequence length %d must divide 128", a.tokens);
      mode = MODE_PACKED;
      p.Lk = 128;
      p.group = a.tokens;
      p.gshift = ilog2(a.tokens);
      p.tiles_per_seq = 1;
      kv_rows = 128;
      grid = dim3(static_cast<unsigned>((T + 127) / 128), H);
    }
    const uint32_t boxQ[3] = {64, 1, 128}, boxQt[3] = {16, 1, 128};
    const uint32_t boxK[3] = {64, 1, kv_rows}, boxKt[3] = {16, 1, kv_rows};
    B200_TRY(make_tmap_16bit(&maps[0], a.qkv, 3, dims, str, boxQ, TMAP_SW_128));
    B200_TRY(make_tmap_16bit(&maps[2], a.qkv, 3, dims, str, boxK, TMAP_SW_128));
    if (tail) {
      B200_TRY(make_tmap_16bit(&maps[1], a.qkv, 3, dims, str, boxQt, TMAP_SW_32));
      B200_TRY(make_tmap_16bit(&maps[3], a.qkv, 3, dims, str, boxKt, TMAP_SW_32));
    } else {
      maps[1] = maps[0];
      maps[3] = maps[2];
    }
    {   // output tile store: dense [128][hd] rows of the staging tile -> rows (b, f, n) of out, columns of this head
      const uint64_t odims[3] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(H), static_cast<uint64_t>(T)};
      const uint64_t ostr[2] = {static_cast<uint64_t>(hd) * 2, static_cast<uint64_t>(D) * 2};
      const uint32_t obox[3] = {static_cast<uint32_t>(hd), 1, 128};
      B200_TRY(make_tmap_16bit(&maps[4], a.out, 3, odims, ostr, obox, TMAP_SW_NONE));
    }
  } else {
    const int F = a.frames;
    B200_REQUIRE(F >= 4 && F <= 128 && 128 % F == 0, B200_ERR_UNSUPPORTED,
                 "attention: temporal length %d unsupported (power of two in [4,128])", F);
    const int G = 128 / F;
    B200_REQUIRE(a.tokens % G == 0, B200_ERR_UNSUPPORTED, "attention: tokens %d must be a multiple of %d", a.tokens, G);
    mode = MODE_TEMPORAL;
    p.Lk = 128;
    p.group = G;
    p.gshift = ilog2(G);
    p.tiles_per_seq = a.tokens / G;
    grid = dim3(a.batch * p.tiles_per_seq, H);
    const uint64_t dims[4] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(3 * H), static_cast<uint64_t>(a.tokens),
                              static_cast<uint64_t>(a.batch) * F};
    const uint64_t str[3] = {static_cast<uint64_t>(hd) * 2, static_cast<uint64_t>(3 * D) * 2,
                             static_cast<uint64_t>(3 * D) * 2 * a.tokens};
    const uint32_t box[4] = {64, 1, static_cast<uint32_t>(G), static_cast<uint32_t>(F)};
    const uint32_t boxt[4] = {16, 1, static_cast<uint32_t>(G), static_cast<uint32_t>(F)};
    B200_TRY(make_tmap_16bit(&maps[0], a.qkv, 4, dims, str, box, TMAP_SW_128));
    maps[2] = maps[0];
    if (tail) {
      B200_TRY(make_tmap_16bit(&maps[1], a.qkv, 4, dims, str, boxt, TMAP_SW_32));
      maps[3] = maps[1];
    } else {
      maps[1] = maps[0];
      maps[3] = maps[0];
    }
    {   // output store with the same (token group) x (frames) box as the loads: tile row f*G + g -> out row (b*F + f)*N + n0 + g
      const uint64_t odims[4] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(H), static_cast<uint64_t>(a.tokens),
                                 static_cast<uint64_t>(a.batch) * F};
      const uint64_t ostr[3] = {static_cast<uint64_t>(hd) * 2, static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(D) * 2 * a.tokens};
      const uint32_t obox[4] = {static_cast<uint32_t>(hd), 1, static_cast<uint32_t>(G), static_cast<uint32_t>(F)};
      B200_TRY(make_tmap_16bit(&maps[4], a.out, 4, odims, ostr, obox, TMAP_SW_NONE));
    }
  }
  if (a.bf16) return tail ? launch_tail<true, true>(mode, maps, p, grid, stream) : launch_tail<true, false>(mode, maps, p, grid, stream);
  return tail ? launch_tail<false, true>(mode, maps, p, grid, stream) : launch_tail<false, false>(mode, maps, p, grid, stream);
}

int launch_cross_attention(const CrossAttnArgs& a, cudaStream_t stream) {
  B200_REQUIRE(a.batch > 0 && a.q_rows_per_batch > 0 && a.heads > 0, B200_ERR_SHAPE, "cross attention: bad shape");
  B200_REQUIRE(a.head_dim == 64 || a.head_dim == 72 || a.head_dim == 80, B200_ERR_UNSUPPORTED,
               "cross attention: head_dim %d unsupported (64, 72, 80)", a.head_dim);
  B200_REQUIRE(a.kv_len >= 1 && a.kv_len <= 128, B200_ERR_UNSUPPORTED, "cross attention: %d keys per sample (1..128 built)", a.kv_len);
  B200_REQUIRE(a.q_rows_per_batch % 128 == 0, B200_ERR_UNSUPPORTED, "cross attention: query rows per sample %d must be a multiple of 128",
               a.q_rows_per_batch);
  B200_REQUIRE(((reinterpret_cast<uintptr_t>(a.q) | reinterpret_cast<uintptr_t>(a.kv) | reinterpret_cast<uintptr_t>(a.out)) & 15) == 0,
               B200_ERR_ALIGN, "cross attention: q/kv/out must be 16-byte aligned");
  B200_TRY(check_arch());
  const int H = a.heads, hd = a.head_dim, D = H * hd;
  const long long T = static_cast<long long>(a.batch) * a.q_rows_per_batch;
  const long long R = static_cast<long long>(a.batch) * (a.kv_batch_rows > 0 ? a.kv_batch_rows : a.kv_len);
  const bool tail = hd > 64;
  AttnDev p{};
  p.out = a.out; p.T = static_cast<int>(T); p.D = D; p.heads = H; p.hd = hd;
  p.tokens = a.q_rows_per_batch; p.frames = 1; p.group = 1; p.gshift = 0; p.Lk = 128; p.tiles_per_seq = 1;
  p.scale_log2 = (a.scale > 0.f ? a.scale : 1.0f / sqrtf(static_cast<float>(hd))) * 1.4426950408889634f;
  p.k_head0 = 0; p.v_head0 = H; p.q_rows_per_batch = a.q_rows_per_batch;
  p.kv_rows_per_batch = a.kv_batch_rows > 0 ? a.kv_batch_rows : a.kv_len;
  p.kv_valid = a.kv_len;
  B200_REQUIRE(p.kv_rows_per_batch >= a.kv_len, B200_ERR_SHAPE, "cross attention: kv_batch_rows %d < kv_len %d", a.kv_batch_rows, a.kv_len);
  B200_REQUIRE(!a.pos_bias || (a.q_rows_per_batch == 128 && (reinterpret_cast<uintptr_t>(a.pos_bias) & 15) == 0), B200_ERR_UNSUPPORTED,
               "cross attention: pos_bias needs 128 query rows per sample (one tile) and 16-byte alignment");
  p.pos_bias = a.pos_bias;
  static const int dbg = env_int("B200_ATTN_DBG", 0);
  p.dbg = dbg;
  B200_REQUIRE(!a.key_bias || (reinterpret_cast<uintptr_t>(a.key_bias) & 15) == 0, B200_ERR_ALIGN, "cross attention: key_bias must be 16-byte aligned");
  p.key_bias = a.key_bias;
  CUtensorMap maps[5];
  const uint64_t qdims[3] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(H), static_cast<uint64_t>(T)};
  const uint64_t qstr[2] = {static_cast<uint64_t>(hd) * 2, static_cast<uint64_t>(a.q_row_stride) * 2};
  const uint64_t kdims[3] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(2 * H), static_cast<uint64_t>(R)};
  const uint64_t kstr[2] = {static_cast<uint64_t>(hd) * 2, static_cast<uint64_t>(a.kv_row_stride) * 2};
  const uint32_t box[3] = {64, 1, 128}, boxt[3] = {16, 1, 128};
  B200_REQUIRE(a.q_row_stride >= D && a.kv_row_stride >= 2 * D && a.q_row_stride % 8 == 0 && a.kv_row_stride % 8 == 0, B200_ERR_SHAPE, "cross attention: bad row strides");
  B200_TRY(make_tmap_16bit(&maps[0], a.q, 3, qdims, qstr, box, TMAP_SW_128));
  B200_TRY(make_tmap_16bit(&maps[2], a.kv, 3, kdims, kstr, box, TMAP_SW_128));
  if (tail) {
    B200_TRY(make_tmap_16bit(&maps[1], a.q, 3, qdims, qstr, boxt, TMAP_SW_32));
    B200_TRY(make_tmap_16bit(&maps[3], a.kv, 3, kdims, kstr, boxt, TMAP_SW_32));
  } else {
    maps[1] = maps[0];
    maps[3] = maps[2];
  }
  {
    const uint64_t odims[3] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(H), static_cast<uint64_t>(T)};
    const uint64_t ostr[2] = {static_cast<uint64_t>(hd) * 2, static_cast<uint64_t>(D) * 2};
    const uint32_t obox[3] = {static_cast<uint32_t>(hd), 1, 128};
    B200_TRY(make_tmap_16bit(&maps[4], a.out, 3, odims, ostr, obox, TMAP_SW_NONE));
  }
  const dim3 grid(static_cast<unsigned>(T / 128), H);
  if (a.pos_bias) {   // the per-(head, row, key) bias exists in the v3 kernel only
    if (a.bf16) return tail ? launch_v3<true, true, MODE_CROSS>(maps, p, grid, stream) : launch_v3<true, false, MODE_CROSS>(maps, p, grid, stream);
    return tail ? launch_v3<false, true, MODE_CROSS>(maps, p, grid, stream) : launch_v3<false, false, MODE_CROSS>(maps, p, grid, stream);
  }
  if (a.bf16) return tail ? launch_tail<true, true>(MODE_CROSS, maps, p, grid, stream) : launch_tail<true, false>(MODE_CROSS, maps, p, grid, stream);
  return tail ? launch_tail<false, true>(MODE_CROSS, maps, p, grid, stream) : launch_tail<false, false>(MODE_CROSS, maps, p, grid, stream);
}

}  // namespace b200
