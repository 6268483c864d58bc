// K2 — single-token decode attention against a KV cache for sm_100a, plus the small bandwidth-bound helpers
// of the path (split-K reduce, KV append, LSE merge for the ring, fp32 -> 16-bit cast).
//
// Replaces _paged_attention_fwd_kernel / triton_paged_attention_forward
// (kernels/triton/attention_kernels.py:628-808, :1206-1311) and _reshape_and_cache_kernel (:811-905).
//
// Decode attention has ~1 FLOP per KV byte (MHA), so it is an HBM-streaming kernel, not a tensor-core one:
//   * each KV row (D 16-bit values) is read exactly once with 128-bit ld.global.nc.L1::no_allocate loads,
//     fully coalesced (D/8 lanes cover a row, a warp instruction covers 32/(D/8) consecutive rows);
//   * every warp keeps 16 independent 16-byte loads in flight per lane (8 K + 8 V); 8 warps per CTA and 2-3
//     CTAs per SM give > 128 KB in flight per SM;
//   * flash-decoding split-K: grid = (splits, Hkv, B); per-split partial (O, LSE) are merged by a tiny reduce
//     kernel, so all 148 SMs stream even for small B*Hkv;
//   * GQA: one CTA serves the G = Hq/Hkv query heads that share a KV head, so K/V bytes are read once per group.

#include "common.cuh"
#include "host_common.h"

namespace b200 {
namespace decode {

constexpr int NUM_WARPS = 8;
constexpr int NUM_THREADS = NUM_WARPS * 32;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ uint4 ld_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

struct Params {
  const void* q;        // [B, Hq, D]
  const void* k_cache;
  const void* v_cache;
  void* o;              // [B, Hq, D]
  float* lse;           // [B, Hq] or null
  float* part_o;        // [B, Hq, splits, D] fp32 (normalised partial outputs)
  float* part_lse;      // [B, Hq, splits]
  const int32_t* context_lens;
  const int32_t* block_table;
  int B, Hq, Hkv;
  int splits;
  float scale_log2;     // softmax_scale * log2(e)
  int64_t kv_batch_stride, kv_token_stride;  // contiguous layout, elements
  int max_blocks_per_seq, block_size, num_layers, layer_idx;
  int capacity;         // keys the cache of one sequence can hold: device-side context lengths are clamped to it, so a
                        // length that ran past the cache (e.g. advanced on the device under a CUDA graph) cannot turn into
                        // an out-of-bounds block-table read
};

template <int D, int G, typename T, bool PAGED>
__global__ void __launch_bounds__(NUM_THREADS, 2)
decode_kernel(const Params p) {
  // 16-byte loads in flight per lane for K (and again for V); G is 1 or 2 here (wider groups run decode_gqa_mma_kernel)
  constexpr int NLOAD = 8;
  constexpr int LPR = D / 8;          // lanes per KV row
  constexpr int RPW = 32 / LPR;       // rows per warp-wide load
  constexpr int TILE = NLOAD * RPW;   // keys per warp iteration

  const int split = blockIdx.x;
  const int kvh = blockIdx.y;
  const int b = blockIdx.z;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR;         // which 8-element slice of the row
  const int rsel = lane / LPR;        // which row of the warp-wide load

  const int ctx = max(0, min(p.context_lens[b], p.capacity));
  // per-batch split range, aligned to TILE
  int chunk = (ctx + p.splits - 1) / p.splits;
  chunk = ((chunk + TILE - 1) / TILE) * TILE;
  const int k_begin = min(split * chunk, ctx);
  const int k_end = min(k_begin + chunk, ctx);

  // query slices (pre-scaled by softmax_scale * log2 e)
  float qf[G][8];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const T* qp = reinterpret_cast<const T*>(p.q) + (static_cast<int64_t>(b) * p.Hq + kvh * G + g) * D + sub * 8;
    uint4 raw = *reinterpret_cast<const uint4*>(qp);
    float2 f;
    f = Pack2<T>::unpack(raw.x); qf[g][0] = f.x * p.scale_log2; qf[g][1] = f.y * p.scale_log2;
    f = Pack2<T>::unpack(raw.y); qf[g][2] = f.x * p.scale_log2; qf[g][3] = f.y * p.scale_log2;
    f = Pack2<T>::unpack(raw.z); qf[g][4] = f.x * p.scale_log2; qf[g][5] = f.y * p.scale_log2;
    f = Pack2<T>::unpack(raw.w); qf[g][6] = f.x * p.scale_log2; qf[g][7] = f.y * p.scale_log2;
  }

  float m_run[G], l_run[G], acc[G][8];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    m_run[g] = -INFINITY;
    l_run[g] = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[g][e] = 0.f;
  }

  const T* kc = reinterpret_cast<const T*>(p.k_cache);
  const T* vc = reinterpret_cast<const T*>(p.v_cache);
  const int32_t* bt = PAGED ? p.block_table + static_cast<int64_t>(b) * p.max_blocks_per_seq : nullptr;
  const bool bs_pow2 = PAGED && ((p.block_size & (p.block_size - 1)) == 0);
  const int bs_shift = bs_pow2 ? (31 - __clz(p.block_size)) : 0;

  for (int t0 = k_begin + warp * TILE; t0 < k_end; t0 += NUM_WARPS * TILE) {
    uint4 kraw[NLOAD], vraw[NLOAD];
    bool valid[NLOAD];
    // ---- issue all loads of the tile ----
#pragma unroll
    for (int i = 0; i < NLOAD; ++i) {
      const int key = t0 + i * RPW + rsel;
      valid[i] = key < k_end;
      int64_t off;
      if constexpr (PAGED) {
        int blk = 0, in_blk = 0;
        if (valid[i]) {
          const int bi = bs_pow2 ? (key >> bs_shift) : (key / p.block_size);
          in_blk = bs_pow2 ? (key & (p.block_size - 1)) : (key - bi * p.block_size);
          blk = bt[bi];
        }
        off = ((static_cast<int64_t>(blk) * p.num_layers + p.layer_idx) * p.block_size + in_blk) *
                  (static_cast<int64_t>(p.Hkv) * D) +
              kvh * D + sub * 8;
      } else {
        off = static_cast<int64_t>(b) * p.kv_batch_stride + static_cast<int64_t>(key) * p.kv_token_stride +
              kvh * D + sub * 8;
      }
      if (valid[i]) {
        kraw[i] = ld_stream(kc + off);
        vraw[i] = ld_stream(vc + off);
      } else {
        kraw[i] = make_uint4(0, 0, 0, 0);
        vraw[i] = make_uint4(0, 0, 0, 0);
      }
    }
    // ---- scores ----
    float s[G][NLOAD];
#pragma unroll
    for (int i = 0; i < NLOAD; ++i) {
      float kf[8];
      float2 f;
      f = Pack2<T>::unpack(kraw[i].x); kf[0] = f.x; kf[1] = f.y;
      f = Pack2<T>::unpack(kraw[i].y); kf[2] = f.x; kf[3] = f.y;
      f = Pack2<T>::unpack(kraw[i].z); kf[4] = f.x; kf[5] = f.y;
      f = Pack2<T>::unpack(kraw[i].w); kf[6] = f.x; kf[7] = f.y;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        float d = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) d = fmaf(qf[g][e], kf[e], d);
#pragma unroll
        for (int x = LPR / 2; x >= 1; x >>= 1) d += __shfl_xor_sync(0xffffffffu, d, x);
        s[g][i] = valid[i] ? d : -INFINITY;
      }
    }
    // ---- online softmax update (one rescale per tile) ----
    float pr[G][NLOAD];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      float tmax = s[g][0];
#pragma unroll
      for (int i = 1; i < NLOAD; ++i) tmax = fmaxf(tmax, s[g][i]);
#pragma unroll
      for (int x = LPR; x < 32; x <<= 1) tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, x));
      const float m_new = fmaxf(m_run[g], tmax);
      const float m_safe = (m_new == -INFINITY) ? 0.f : m_new;
      const float corr = fast_exp2(m_run[g] - m_safe);  // m_run = -inf -> 0
      m_run[g] = m_new;
      l_run[g] *= corr;
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[g][e] *= corr;
#pragma unroll
      for (int i = 0; i < NLOAD; ++i) {
        pr[g][i] = fast_exp2(s[g][i] - m_safe);
        l_run[g] += pr[g][i];
      }
    }
    // ---- P V ----
#pragma unroll
    for (int i = 0; i < NLOAD; ++i) {
      float vf[8];
      float2 f;
      f = Pack2<T>::unpack(vraw[i].x); vf[0] = f.x; vf[1] = f.y;
      f = Pack2<T>::unpack(vraw[i].y); vf[2] = f.x; vf[3] = f.y;
      f = Pack2<T>::unpack(vraw[i].z); vf[4] = f.x; vf[5] = f.y;
      f = Pack2<T>::unpack(vraw[i].w); vf[6] = f.x; vf[7] = f.y;
#pragma unroll
      for (int g = 0; g < G; ++g) {
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[g][e] = fmaf(pr[g][i], vf[e], acc[g][e]);
      }
    }
  }

  // ---- combine the row groups of a warp (they share m_run) ----
#pragma unroll
  for (int g = 0; g < G; ++g) {
#pragma unroll
    for (int x = LPR; x < 32; x <<= 1) {
      l_run[g] += __shfl_xor_sync(0xffffffffu, l_run[g], x);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[g][e] += __shfl_xor_sync(0xffffffffu, acc[g][e], x);
    }
  }

  // ---- combine the warps of the CTA through shared memory ----
  __shared__ float sm_m[NUM_WARPS][G];
  __shared__ float sm_l[NUM_WARPS][G];
  __shared__ float sm_acc[NUM_WARPS][G][D];
  if (rsel == 0) {
#pragma unroll
    for (int g = 0; g < G; ++g) {
#pragma unroll
      for (int e = 0; e < 8; ++e) sm_acc[warp][g][sub * 8 + e] = acc[g][e];
      if (sub == 0) {
        sm_m[warp][g] = m_run[g];
        sm_l[warp][g] = l_run[g];
      }
    }
  }
  __syncthreads();

  for (int idx = threadIdx.x; idx < G * D; idx += NUM_THREADS) {
    const int g = idx / D;
    const int d = idx - g * D;
    float m = -INFINITY;
#pragma unroll
    for (int w = 0; w < NUM_WARPS; ++w) m = fmaxf(m, sm_m[w][g]);
    const float m_safe = (m == -INFINITY) ? 0.f : m;
    float l = 0.f, o = 0.f;
#pragma unroll
    for (int w = 0; w < NUM_WARPS; ++w) {
      const float c = fast_exp2(sm_m[w][g] - m_safe);
      l = fmaf(sm_l[w][g], c, l);
      o = fmaf(sm_acc[w][g][d], c, o);
    }
    const float inv_l = l > 0.f ? 1.0f / l : 0.f;
    const float out = o * inv_l;
    const float lse = l > 0.f ? (m + log2f(l)) * kLn2 : -INFINITY;
    const int h = kvh * G + g;
    if (p.splits == 1) {
      T* op = reinterpret_cast<T*>(p.o) + (static_cast<int64_t>(b) * p.Hq + h) * D + d;
      if constexpr (Pack2<T>::kIsBf16) *op = __float2bfloat16_rn(out);
      else *op = __float2half_rn(out);
      if (d == 0 && p.lse != nullptr) p.lse[static_cast<int64_t>(b) * p.Hq + h] = lse;
    } else {
      const int64_t row = (static_cast<int64_t>(b) * p.Hq + h) * p.splits + split;
      p.part_o[row * D + d] = out;
      if (d == 0) p.part_lse[row] = lse;
    }
  }
}


// ---------------------------------------------------------------------------------------------------------------
// GQA decode on the legacy tensor-core path (mma.sync m16n8k16): the G query heads that share a KV head are the M rows
// of the MMA, so the FMA / shuffle / exp work per KV byte no longer grows with G (the CUDA-core kernel above becomes
// ALU-bound for G >= 4). Still an HBM-streaming kernel — every K/V byte is loaded exactly once with 128-bit loads in a
// fragment-friendly order, no shared-memory staging:
//   Q K^T : lane (g,t) loads K[key g][32m + 8t .. +8) — the contraction (head-dim) index may be permuted freely as long
//           as the Q fragments use the same permutation, so one uint4 feeds two k-steps (b0,b1 = words x,y then z,w);
//   P V   : lane (g,t) loads V rows of keys {2t, 2t+1, 2t+8, 2t+9} at dims [64d + 8g, +8); PRMT pairs the two keys of a
//           column into a B fragment. Output column n of n-tile (d, j) is dim 64d + 8n + j (undone at the final store).
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void mma_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                          uint32_t b1) {
  if constexpr (Pack2<T>::kIsBf16) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
  } else {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
  }
}

constexpr int GQA_WARPS = 4;
constexpr bool kGqaRingDefault = false;
// resident CTAs per SM the register allocation is capped for: two tiles of K/V are staged in registers per lane
// (D = 128: 128 of ~250 registers -> 2 CTAs; D = 64: 64 of ~170 -> 3 CTAs, measured 4721 vs 4002 GB/s with 2)
template <int D> struct GqaMinCtas { static constexpr int value = D == 128 ? 2 : 3; };

// RING = true: every warp stages its K/V tiles through a private ring in shared memory instead of registers: each lane
// issues the same 16-byte pieces it would have loaded (cp.async.cg, zero-filled for keys past the end) into its own
// 16-byte column of a [slot][lane] array — no lane ever reads another lane's bytes, so there is no layout, bank-conflict or
// synchronisation question — and reads them back as MMA fragments when the tile's copy group has completed. Two tiles per
// warp are in flight while a third is consumed (the register-staged variant keeps one), and the staging registers go
// from 128 to 64 per lane. The combine buffers of the epilogue alias the ring. (A first version used one 256-byte
// cp.async.bulk per key row and mbarriers: slower, 5309 vs 5810 GB/s — 32 small bulk copies per 8 KB tile.)
constexpr int GQA_RING_STAGES = 3;
template <int D> struct GqaRing {
  static constexpr int SLOTS = 2 * (D / 32) + (D / 64) * 4;       // 16-byte pieces per lane and tile (K: 2 x MB, V: DG x 4)
  static constexpr int TILE_BYTES = SLOTS * 32 * 16;              // 8 KB at D = 128
  static constexpr int RING_BYTES = GQA_WARPS * GQA_RING_STAGES * TILE_BYTES;
  static constexpr int COMB_BYTES = (2 * GQA_WARPS * 16 + GQA_WARPS * 16 * D) * 4;
  static constexpr int SMEM_BYTES = RING_BYTES > COMB_BYTES ? RING_BYTES : COMB_BYTES;
};
// 16-byte async copy global -> shared; src_bytes = 0 zero-fills the destination (keys past the end of the sequence)
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}

template <int D, typename T, bool PAGED, bool RING>
__global__ void __launch_bounds__(GQA_WARPS * 32, GqaMinCtas<D>::value)
decode_gqa_mma_kernel(const Params p, const int G) {
  constexpr int TILE = 16;       // keys per warp iteration
  constexpr int MB = D / 32;     // 32-dim blocks of the head dimension (two MMA k-steps each)
  constexpr int DG = D / 64;     // 64-dim groups of the output
  constexpr int NT = D / 8;      // n-tiles of the P V product

  const int split = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;

  const int ctx = max(0, min(p.context_lens[b], p.capacity));
  int chunk = (ctx + p.splits - 1) / p.splits;
  chunk = ((chunk + TILE - 1) / TILE) * TILE;
  const int k_begin = min(split * chunk, ctx);
  const int k_end = min(k_begin + chunk, ctx);

  // Q fragments for rows g and g+8 (zero rows beyond the group)
  uint32_t qa[MB][4], qb[MB][4];
  {
    const T* qbase = reinterpret_cast<const T*>(p.q) + (static_cast<int64_t>(b) * p.Hq + kvh * G) * D;
#pragma unroll
    for (int m = 0; m < MB; ++m) {
      uint4 ra = make_uint4(0, 0, 0, 0), rb = make_uint4(0, 0, 0, 0);
      if (g < G) ra = *reinterpret_cast<const uint4*>(qbase + static_cast<int64_t>(g) * D + 32 * m + 8 * t);
      if (g + 8 < G) rb = *reinterpret_cast<const uint4*>(qbase + static_cast<int64_t>(g + 8) * D + 32 * m + 8 * t);
      qa[m][0] = ra.x; qa[m][1] = ra.y; qa[m][2] = ra.z; qa[m][3] = ra.w;
      qb[m][0] = rb.x; qb[m][1] = rb.y; qb[m][2] = rb.z; qb[m][3] = rb.w;
    }
  }
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  float o[NT][4];
#pragma unroll
  for (int n = 0; n < NT; ++n) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }

  const T* kc = reinterpret_cast<const T*>(p.k_cache);
  const T* vc = reinterpret_cast<const T*>(p.v_cache);
  const int32_t* bt = PAGED ? p.block_table + static_cast<int64_t>(b) * p.max_blocks_per_seq : nullptr;
  auto row_offset = [&](int key) -> int64_t {  // element offset of (key, kvh, dim 0)
    if constexpr (PAGED) {
      const int bi = key / p.block_size;
      const int in_blk = key - bi * p.block_size;
      return ((static_cast<int64_t>(bt[bi]) * p.num_layers + p.layer_idx) * p.block_size + in_blk) *
                 (static_cast<int64_t>(p.Hkv) * D) + kvh * D;
    } else {
      return static_cast<int64_t>(b) * p.kv_batch_stride + static_cast<int64_t>(key) * p.kv_token_stride + kvh * D;
    }
  };

  // Software pipeline over the warp's tiles: the 16 128-bit loads of tile i+1 are issued BEFORE the MMAs / softmax of
  // tile i, so every warp always has a full tile (8 KB) in flight instead of only during its load phase (the kernel is
  // HBM-bound: 67.8 % of DRAM peak without the prefetch, profiles/r1_decode_v1_ncu.txt). Two register buffers, loop
  // unrolled by two so their roles are static.
  auto issue_tile = [&](const int t0, uint4 (&kr)[2][MB], uint4 (&vr)[DG][4]) {
#pragma unroll
    for (int kg = 0; kg < 2; ++kg) {
      const int key = t0 + kg * 8 + g;
      const bool valid = key < k_end;
      const int64_t off = valid ? row_offset(key) + 8 * t : 0;
#pragma unroll
      for (int m = 0; m < MB; ++m) kr[kg][m] = valid ? ld_stream(kc + off + 32 * m) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int key = t0 + 2 * t + (j & 1) + (j >> 1) * 8;
      const bool valid = key < k_end;
      const int64_t off = valid ? row_offset(key) + 8 * g : 0;
#pragma unroll
      for (int d = 0; d < DG; ++d) vr[d][j] = valid ? ld_stream(vc + off + 64 * d) : make_uint4(0, 0, 0, 0);
    }
  };
  auto compute_tile = [&](const int t0, const uint4 (&kr)[2][MB], const uint4 (&vr)[DG][4]) {
    // ---- S = Q K^T (rows g, g+8; keys kg*8 + 2t, +1) ----
    float sc[2][4];
#pragma unroll
    for (int kg = 0; kg < 2; ++kg) {
      sc[kg][0] = sc[kg][1] = sc[kg][2] = sc[kg][3] = 0.f;
#pragma unroll
      for (int m = 0; m < MB; ++m) {
        mma_16816<T>(sc[kg], qa[m][0], qb[m][0], qa[m][1], qb[m][1], kr[kg][m].x, kr[kg][m].y);
        mma_16816<T>(sc[kg], qa[m][2], qb[m][2], qa[m][3], qb[m][3], kr[kg][m].z, kr[kg][m].w);
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = t0 + kg * 8 + 2 * t + (e & 1);
        sc[kg][e] = key < k_end ? sc[kg][e] * p.scale_log2 : -INFINITY;
      }
    }
    // ---- online softmax for the two rows this lane holds ----
    float pr[2][4];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      float tmax = fmaxf(fmaxf(sc[0][2 * r], sc[0][2 * r + 1]), fmaxf(sc[1][2 * r], sc[1][2 * r + 1]));
      tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, 1));
      tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, 2));
      const float m_new = fmaxf(m_run[r], tmax);
      const float m_safe = (m_new == -INFINITY) ? 0.f : m_new;
      const float corr = fast_exp2(m_run[r] - m_safe);
      m_run[r] = m_new;
      l_run[r] *= corr;
#pragma unroll
      for (int n = 0; n < NT; ++n) { o[n][2 * r] *= corr; o[n][2 * r + 1] *= corr; }
#pragma unroll
      for (int kg = 0; kg < 2; ++kg) {
        pr[kg][2 * r] = fast_exp2(sc[kg][2 * r] - m_safe);
        pr[kg][2 * r + 1] = fast_exp2(sc[kg][2 * r + 1] - m_safe);
        l_run[r] += pr[kg][2 * r] + pr[kg][2 * r + 1];
      }
    }
    // ---- O += P V ----
    const uint32_t pa0 = Pack2<T>::pack(pr[0][0], pr[0][1]), pa1 = Pack2<T>::pack(pr[0][2], pr[0][3]);
    const uint32_t pa2 = Pack2<T>::pack(pr[1][0], pr[1][1]), pa3 = Pack2<T>::pack(pr[1][2], pr[1][3]);
#pragma unroll
    for (int d = 0; d < DG; ++d) {
      const uint32_t w0[4] = {vr[d][0].x, vr[d][0].y, vr[d][0].z, vr[d][0].w};
      const uint32_t w1[4] = {vr[d][1].x, vr[d][1].y, vr[d][1].z, vr[d][1].w};
      const uint32_t w2[4] = {vr[d][2].x, vr[d][2].y, vr[d][2].z, vr[d][2].w};
      const uint32_t w3[4] = {vr[d][3].x, vr[d][3].y, vr[d][3].z, vr[d][3].w};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t sel = (j & 1) ? 0x7632u : 0x5410u;
        const uint32_t b0 = __byte_perm(w0[j >> 1], w1[j >> 1], sel);  // (V[key 2t][dim], V[key 2t+1][dim])
        const uint32_t b1 = __byte_perm(w2[j >> 1], w3[j >> 1], sel);  // (V[key 2t+8][dim], V[key 2t+9][dim])
        mma_16816<T>(o[d * 8 + j], pa0, pa1, pa2, pa3, b0, b1);
      }
    }
  };
  constexpr int STEP = GQA_WARPS * TILE;
  extern __shared__ __align__(128) uint8_t gqa_dsm[];
  if constexpr (RING) {
    using R = GqaRing<D>;
    constexpr int NSTG = GQA_RING_STAGES;
    // this lane's 16-byte column of slot 0 of stage 0
    const uint32_t ring0 = smem_u32(gqa_dsm) + static_cast<uint32_t>(warp * NSTG * R::TILE_BYTES + lane * 16);
    const int first_t0 = k_begin + warp * TILE;
    const int n_tiles = first_t0 < k_end ? (k_end - first_t0 + STEP - 1) / STEP : 0;
    auto issue_ring = [&](const int i) {  // tile i of this warp -> stage i % NSTG (one commit group, possibly empty)
      if (i < n_tiles) {
        const int t0 = first_t0 + i * STEP;
        const uint32_t st = ring0 + static_cast<uint32_t>((i % NSTG) * R::TILE_BYTES);
#pragma unroll
        for (int kg = 0; kg < 2; ++kg) {
          const int key = t0 + kg * 8 + g;
          const bool valid = key < k_end;
          const T* src = kc + (valid ? row_offset(key) + 8 * t : 0);
#pragma unroll
          for (int m = 0; m < MB; ++m) cp_async16(st + static_cast<uint32_t>((kg * MB + m) * 512), src + 32 * m, valid ? 16u : 0u);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int key = t0 + 2 * t + (j & 1) + (j >> 1) * 8;
          const bool valid = key < k_end;
          const T* src = vc + (valid ? row_offset(key) + 8 * g : 0);
#pragma unroll
          for (int d = 0; d < DG; ++d) cp_async16(st + static_cast<uint32_t>((2 * MB + d * 4 + j) * 512), src + 64 * d, valid ? 16u : 0u);
        }
      }
      cp_async_commit();
    };
#pragma unroll
    for (int i = 0; i < NSTG - 1; ++i) issue_ring(i);
    for (int i = 0; i < n_tiles; ++i) {
      issue_ring(i + NSTG - 1);          // refills the stage consumed in iteration i - 1 (its fragments are in registers)
      cp_async_wait<NSTG - 1>();         // all groups but the NSTG - 1 most recent are complete: tile i has landed
      const uint32_t st = ring0 + static_cast<uint32_t>((i % NSTG) * R::TILE_BYTES);
      uint4 kr[2][MB], vr[DG][4];
#pragma unroll
      for (int kg = 0; kg < 2; ++kg)
#pragma unroll
        for (int m = 0; m < MB; ++m) kr[kg][m] = lds128(st + static_cast<uint32_t>((kg * MB + m) * 512));
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int d = 0; d < DG; ++d) vr[d][j] = lds128(st + static_cast<uint32_t>((2 * MB + d * 4 + j) * 512));
      compute_tile(first_t0 + i * STEP, kr, vr);
    }
    cp_async_wait<0>();
    __syncthreads();  // the combine buffers below alias the ring
  } else {
    uint4 krA[2][MB], vrA[DG][4], krB[2][MB], vrB[DG][4];
    int t0 = k_begin + warp * TILE;
    if (t0 < k_end) issue_tile(t0, krA, vrA);
    for (; t0 < k_end; t0 += 2 * STEP) {
      if (t0 + STEP < k_end) issue_tile(t0 + STEP, krB, vrB);
      compute_tile(t0, krA, vrA);
      if (t0 + 2 * STEP < k_end) issue_tile(t0 + 2 * STEP, krA, vrA);
      if (t0 + STEP < k_end) compute_tile(t0 + STEP, krB, vrB);
    }
  }

  // ---- combine: lanes of a row quad, then the warps of the CTA through shared memory ----
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
  }
  float* comb;
  if constexpr (RING) {
    comb = reinterpret_cast<float*>(gqa_dsm);
  } else {
    __shared__ float comb_static[2 * GQA_WARPS * 16 + GQA_WARPS * 16 * D];
    comb = comb_static;
  }
  float* sm_m = comb;                          // [warp][16]
  float* sm_l = comb + GQA_WARPS * 16;         // [warp][16]
  float* sm_acc = comb + 2 * GQA_WARPS * 16;   // [warp][16][D]
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int row = g + 8 * r;
    if (row < G) {
      if (t == 0) { sm_m[warp * 16 + row] = m_run[r]; sm_l[warp * 16 + row] = l_run[r]; }
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        const int d = n >> 3, j = n & 7;
        sm_acc[(warp * 16 + row) * D + 64 * d + 8 * (2 * t) + j] = o[n][2 * r];
        sm_acc[(warp * 16 + row) * D + 64 * d + 8 * (2 * t + 1) + j] = o[n][2 * r + 1];
      }
    }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < G * D; idx += GQA_WARPS * 32) {
    const int row = idx / D, d = idx - row * D;
    float m = -INFINITY;
#pragma unroll
    for (int w = 0; w < GQA_WARPS; ++w) m = fmaxf(m, sm_m[w * 16 + row]);
    const float m_safe = (m == -INFINITY) ? 0.f : m;
    float l = 0.f, acc = 0.f;
#pragma unroll
    for (int w = 0; w < GQA_WARPS; ++w) {
      const float c = fast_exp2(sm_m[w * 16 + row] - m_safe);
      l = fmaf(sm_l[w * 16 + row], c, l);
      acc = fmaf(sm_acc[(w * 16 + row) * D + d], c, acc);
    }
    const float out = l > 0.f ? acc / l : 0.f;
    const float lse = l > 0.f ? (m + log2f(l)) * kLn2 : -INFINITY;
    const int h = kvh * G + row;
    if (p.splits == 1) {
      T* op = reinterpret_cast<T*>(p.o) + (static_cast<int64_t>(b) * p.Hq + h) * D + d;
      if constexpr (Pack2<T>::kIsBf16) *op = __float2bfloat16_rn(out);
      else *op = __float2half_rn(out);
      if (d == 0 && p.lse != nullptr) p.lse[static_cast<int64_t>(b) * p.Hq + h] = lse;
    } else {
      const int64_t prow = (static_cast<int64_t>(b) * p.Hq + h) * p.splits + split;
      p.part_o[prow * D + d] = out;
      if (d == 0) p.part_lse[prow] = lse;
    }
  }
}

// merge the per-split partials: o = sum_s exp(lse_s - lse) o_s
template <int D, typename T>
__global__ void decode_reduce_kernel(const float* __restrict__ part_o, const float* __restrict__ part_lse,
                                     void* __restrict__ o, float* __restrict__ lse, int splits) {
  const int64_t row = blockIdx.x;  // b * Hq + h
  const int d = threadIdx.x;
  float m = -INFINITY;
  for (int s = 0; s < splits; ++s) m = fmaxf(m, part_lse[row * splits + s]);
  const float m_safe = (m == -INFINITY) ? 0.f : m;
  float l = 0.f, acc = 0.f;
  for (int s = 0; s < splits; ++s) {
    const float w = __expf(part_lse[row * splits + s] - m_safe);
    l += w;
    acc = fmaf(w, part_o[(row * splits + s) * D + d], acc);
  }
  const float out = l > 0.f ? acc / l : 0.f;
  T* op = reinterpret_cast<T*>(o) + row * D + d;
  if constexpr (Pack2<T>::kIsBf16) *op = __float2bfloat16_rn(out);
  else *op = __float2half_rn(out);
  if (d == 0 && lse != nullptr) lse[row] = l > 0.f ? m + __logf(l) : -INFINITY;
}

template <typename T>
__global__ void kv_append_kernel(const T* __restrict__ key, const T* __restrict__ value, T* __restrict__ k_cache,
                                 T* __restrict__ v_cache, const int32_t* __restrict__ context_lens, int row_elems,
                                 int layout, int64_t kv_batch_stride, int64_t kv_token_stride,
                                 const int32_t* __restrict__ block_table, int max_blocks_per_seq, int block_size,
                                 int num_layers, int layer_idx, int capacity) {
  const int b = blockIdx.x;
  const int pos = context_lens[b] - 1;  // the appended token is the last valid one (attention_kernels.py:862-866)
  // a position past the cache is dropped, never written: it would index beyond the block table / the sequence's rows and
  // land in another sequence's block
  if (pos < 0 || pos >= capacity) return;
  int64_t base;
  if (layout == B200_KV_PAGED) {
    const int bi = pos / block_size;
    const int in_blk = pos - bi * block_size;
    const int blk = block_table[static_cast<int64_t>(b) * max_blocks_per_seq + bi];
    base = ((static_cast<int64_t>(blk) * num_layers + layer_idx) * block_size + in_blk) * row_elems;
  } else {
    base = static_cast<int64_t>(b) * kv_batch_stride + static_cast<int64_t>(pos) * kv_token_stride;
  }
  const uint4* ks = reinterpret_cast<const uint4*>(key + static_cast<int64_t>(b) * row_elems);
  const uint4* vs = reinterpret_cast<const uint4*>(value + static_cast<int64_t>(b) * row_elems);
  uint4* kd = reinterpret_cast<uint4*>(k_cache + base);
  uint4* vd = reinterpret_cast<uint4*>(v_cache + base);
  for (int i = threadIdx.x; i < row_elems / 8; i += blockDim.x) {
    kd[i] = ks[i];
    vd[i] = vs[i];
  }
}

// in-place LSE merge of an incoming (o_b, lse_b) block into the fp32 ring accumulator
template <typename T>
__global__ void lse_merge_kernel(float* __restrict__ o_acc, float* __restrict__ lse_acc, const T* __restrict__ o_b,
                                 const float* __restrict__ lse_b, int B, int Sq, int Hq, int D, int64_t sb, int64_t ss,
                                 int64_t sh) {
  // one thread per 8 output elements; threads of a (b, s, h) row are adjacent
  const int vec_per_row = D / 8;
  const int64_t total = static_cast<int64_t>(B) * Sq * Hq * vec_per_row;
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int v = static_cast<int>(idx % vec_per_row);
  const int64_t row = idx / vec_per_row;  // (b * Sq + s) * Hq + h
  const int h = static_cast<int>(row % Hq);
  const int64_t bs_ = row / Hq;
  const int s = static_cast<int>(bs_ % Sq);
  const int b = static_cast<int>(bs_ / Sq);
  const int64_t li = (static_cast<int64_t>(b) * Hq + h) * Sq + s;
  const float la = lse_acc[li];
  const float lb = lse_b[li];
  const float m = fmaxf(la, lb);
  float wa, wb, lnew;
  if (m == -INFINITY) {
    wa = 0.f; wb = 0.f; lnew = -INFINITY;
  } else {
    const float ea = __expf(la - m), eb = __expf(lb - m);
    const float sum = ea + eb;
    wa = ea / sum; wb = eb / sum;
    lnew = m + __logf(sum);
  }
  float* oa = o_acc + row * D + v * 8;
  const T* ob = o_b + static_cast<int64_t>(b) * sb + static_cast<int64_t>(s) * ss + static_cast<int64_t>(h) * sh + v * 8;
  const uint4 raw = *reinterpret_cast<const uint4*>(ob);
  float4 a0 = *reinterpret_cast<float4*>(oa);
  float4 a1 = *reinterpret_cast<float4*>(oa + 4);
  float2 f;
  f = Pack2<T>::unpack(raw.x); a0.x = a0.x * wa + f.x * wb; a0.y = a0.y * wa + f.y * wb;
  f = Pack2<T>::unpack(raw.y); a0.z = a0.z * wa + f.x * wb; a0.w = a0.w * wa + f.y * wb;
  f = Pack2<T>::unpack(raw.z); a1.x = a1.x * wa + f.x * wb; a1.y = a1.y * wa + f.y * wb;
  f = Pack2<T>::unpack(raw.w); a1.z = a1.z * wa + f.x * wb; a1.w = a1.w * wa + f.y * wb;
  *reinterpret_cast<float4*>(oa) = a0;
  *reinterpret_cast<float4*>(oa + 4) = a1;
  __syncwarp();
  if (v == 0) lse_acc[li] = lnew;
}

template <typename T>
__global__ void cast_out_kernel(const float* __restrict__ o_acc, T* __restrict__ o, int B, int Sq, int Hq, int D,
                                int64_t sb, int64_t ss, int64_t sh) {
  const int vec_per_row = D / 8;
  const int64_t total = static_cast<int64_t>(B) * Sq * Hq * vec_per_row;
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int v = static_cast<int>(idx % vec_per_row);
  const int64_t row = idx / vec_per_row;
  const int h = static_cast<int>(row % Hq);
  const int64_t bs_ = row / Hq;
  const int s = static_cast<int>(bs_ % Sq);
  const int b = static_cast<int>(bs_ / Sq);
  const float4 a0 = *reinterpret_cast<const float4*>(o_acc + row * D + v * 8);
  const float4 a1 = *reinterpret_cast<const float4*>(o_acc + row * D + v * 8 + 4);
  uint4 pk;
  pk.x = Pack2<T>::pack(a0.x, a0.y);
  pk.y = Pack2<T>::pack(a0.z, a0.w);
  pk.z = Pack2<T>::pack(a1.x, a1.y);
  pk.w = Pack2<T>::pack(a1.z, a1.w);
  T* op = o + static_cast<int64_t>(b) * sb + static_cast<int64_t>(s) * ss + static_cast<int64_t>(h) * sh + v * 8;
  *reinterpret_cast<uint4*>(op) = pk;
}

template <int D, int G, typename T>
int launch_decode(const Params& p, bool paged, cudaStream_t stream) {
  dim3 grid(p.splits, p.Hkv, p.B);
  if (paged) decode_kernel<D, G, T, true><<<grid, NUM_THREADS, 0, stream>>>(p);
  else decode_kernel<D, G, T, false><<<grid, NUM_THREADS, 0, stream>>>(p);
  B200_CUDA_OK(cudaGetLastError());
  note_launch("decode_kernel");
  if (p.splits > 1) {
    decode_reduce_kernel<D, T><<<p.B * p.Hq, D, 0, stream>>>(p.part_o, p.part_lse, p.o, p.lse, p.splits);
    B200_CUDA_OK(cudaGetLastError());
    note_launch("decode_reduce_kernel");
  }
  return B200_OK;
}

template <int D, typename T>
int launch_decode_gqa(int G, const Params& p, bool paged, cudaStream_t stream) {
  dim3 grid(p.splits, p.Hkv, p.B);
  // B200_GQA_RING=0/1 selects the register-staged / shared-memory-ring variant (read per call)
  const char* ring_env = getenv("B200_GQA_RING");
  const bool ring = ring_env != nullptr ? ring_env[0] == '1' : kGqaRingDefault;
  if (ring) {
    constexpr int kSmem = GqaRing<D>::SMEM_BYTES;
    static bool attr_p[64] = {}, attr_c[64] = {};
    if (paged) {
      B200_CUDA_OK(set_max_dynamic_smem(reinterpret_cast<const void*>(decode_gqa_mma_kernel<D, T, true, true>), kSmem, attr_p));
      decode_gqa_mma_kernel<D, T, true, true><<<grid, GQA_WARPS * 32, kSmem, stream>>>(p, G);
    } else {
      B200_CUDA_OK(set_max_dynamic_smem(reinterpret_cast<const void*>(decode_gqa_mma_kernel<D, T, false, true>), kSmem, attr_c));
      decode_gqa_mma_kernel<D, T, false, true><<<grid, GQA_WARPS * 32, kSmem, stream>>>(p, G);
    }
    B200_CUDA_OK(cudaGetLastError());
    note_launch("decode_gqa_ring_kernel");
  } else {
    if (paged) decode_gqa_mma_kernel<D, T, true, false><<<grid, GQA_WARPS * 32, 0, stream>>>(p, G);
    else decode_gqa_mma_kernel<D, T, false, false><<<grid, GQA_WARPS * 32, 0, stream>>>(p, G);
    B200_CUDA_OK(cudaGetLastError());
    note_launch("decode_gqa_mma_kernel");
  }
  if (p.splits > 1) {
    decode_reduce_kernel<D, T><<<p.B * p.Hq, D, 0, stream>>>(p.part_o, p.part_lse, p.o, p.lse, p.splits);
    B200_CUDA_OK(cudaGetLastError());
    note_launch("decode_reduce_kernel");
  }
  return B200_OK;
}

template <int D, typename T>
int dispatch_group(int G, const Params& p, bool paged, cudaStream_t stream) {
  // wide groups: the query heads of a KV head become the rows of mma.sync tiles (any G up to 16)
  if (G >= 3 && G <= 16) return launch_decode_gqa<D, T>(G, p, paged, stream);
  switch (G) {
    case 1: return launch_decode<D, 1, T>(p, paged, stream);
    case 2: return launch_decode<D, 2, T>(p, paged, stream);
    default:
      return set_error(B200_ERR_UNSUPPORTED, "decode: Hq/Hkv = %d is not supported (1 .. 16)", G);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// FP8 (e4m3) paged KV cache. One format for every writer and reader:
//   stored byte = cvt.rn.satfinite.e4m3(x / scale)   x in fp32, correctly rounded division (__fdiv_rn); |x / scale| past
//                                                     448 and +-inf saturate to +-448, NaN stays NaN
//   value read  = byte * scale                        one fp32 k_scale and one v_scale per layer
// The readers never multiply per element: k_scale is folded into the softmax scale on the host, v_scale multiplies each
// output row once before its store. Half the bytes of a 16-bit cache: decode streams half as much from HBM, and the same
// memory holds twice the tokens.
// uint4 values are built by aggregate initialisation, not make_uint4: more call sites of that static inline header
// function change how NVVM inlines it into decode_gqa_mma_kernel, and the 16-bit kernels must compile as before.
// ---------------------------------------------------------------------------------------------------------------
namespace fp8 {

// two fp32 -> two e4m3 bytes (lo in bits 0-7, hi in bits 8-15)
__device__ __forceinline__ uint32_t quant2(float lo, float hi, float scale) {
  uint16_t r;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(__fdiv_rn(hi, scale)), "f"(__fdiv_rn(lo, scale)));
  return r;
}
// four 16-bit values (two packed words) -> four bytes
template <typename T>
__device__ __forceinline__ uint32_t quant4(uint32_t a, uint32_t b, float scale) {
  const float2 x = Pack2<T>::unpack(a), y = Pack2<T>::unpack(b);
  return quant2(x.x, x.y, scale) | (quant2(y.x, y.y, scale) << 16);
}
// the two e4m3 bytes in bits 0-15 of v -> f16x2 (byte 0 in the low half); exact: every e4m3 value is an f16 value
__device__ __forceinline__ uint32_t widen2(uint32_t v) {
  uint32_t r;
  asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(r) : "h"(static_cast<uint16_t>(v)));
  return r;
}
__device__ __forceinline__ float2 half2_to_float2(uint32_t h) { return Pack2<__half>::unpack(h); }
// ld_stream predicated on `valid` (zeros otherwise), without a branch: keeps the staged tiles in registers
__device__ __forceinline__ uint4 ld_stream_if(const void* p, bool valid) {
  uint4 r;
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\t"
               "mov.b32 %0, 0;\n\tmov.b32 %1, 0;\n\tmov.b32 %2, 0;\n\tmov.b32 %3, 0;\n\t"
               "@q ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];\n\t}"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p), "r"(static_cast<int>(valid)));
  return r;
}
__device__ __forceinline__ uint2 ld_stream8_if(const void* p, bool valid) {
  uint2 r;
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %3, 0;\n\tmov.b32 %0, 0;\n\tmov.b32 %1, 0;\n\t"
               "@q ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];\n\t}"
               : "=r"(r.x), "=r"(r.y)
               : "l"(p), "r"(static_cast<int>(valid)));
  return r;
}

// Quantizing append: the n_tokens newest K,V rows of every sequence ([B, n_tokens, Hkv, D], 16-bit) go to positions
// [context_lens[b] - n_tokens, context_lens[b]). n_tokens = 1 is the decode append, n_tokens = S the prompt scatter of
// prefill, so both quantize by the same rule. A position past the cache is dropped, as in kv_append_kernel. Each thread
// turns 16 values (two 16-byte loads) into one 16-byte store.
template <typename T>
__global__ void kv_append_kernel(const T* __restrict__ key, const T* __restrict__ value, uint8_t* __restrict__ k_cache,
                                 uint8_t* __restrict__ v_cache, const int32_t* __restrict__ context_lens, int n_tokens,
                                 int row_elems, const int32_t* __restrict__ block_table, int max_blocks_per_seq,
                                 int block_size, int num_layers, int layer_idx, float k_scale, float v_scale) {
  const int i = blockIdx.x, b = blockIdx.y;
  const int pos = context_lens[b] - n_tokens + i;
  if (pos < 0 || pos >= max_blocks_per_seq * block_size) return;
  const int bi = pos / block_size;
  const int in_blk = pos - bi * block_size;
  const int blk = block_table[static_cast<int64_t>(b) * max_blocks_per_seq + bi];
  const int64_t dst = ((static_cast<int64_t>(blk) * num_layers + layer_idx) * block_size + in_blk) * row_elems;
  const int64_t src = (static_cast<int64_t>(b) * n_tokens + i) * row_elems;
  const uint4* ks = reinterpret_cast<const uint4*>(key + src);
  const uint4* vs = reinterpret_cast<const uint4*>(value + src);
  uint4* kd = reinterpret_cast<uint4*>(k_cache + dst);
  uint4* vd = reinterpret_cast<uint4*>(v_cache + dst);
  for (int c = threadIdx.x; c < row_elems / 16; c += blockDim.x) {
    const uint4 k0 = ks[2 * c], k1 = ks[2 * c + 1], v0 = vs[2 * c], v1 = vs[2 * c + 1];
    kd[c] = uint4{quant4<T>(k0.x, k0.y, k_scale), quant4<T>(k0.z, k0.w, k_scale), quant4<T>(k1.x, k1.y, k_scale),
                       quant4<T>(k1.z, k1.w, k_scale)};
    vd[c] = uint4{quant4<T>(v0.x, v0.y, v_scale), quant4<T>(v0.z, v0.w, v_scale), quant4<T>(v1.x, v1.y, v_scale),
                       quant4<T>(v1.z, v1.w, v_scale)};
  }
}

// 16 e4m3 bytes -> 16 floats
__device__ __forceinline__ void widen16(const uint4 r, float (&f)[16]) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 a = half2_to_float2(widen2(w[j])), c = half2_to_float2(widen2(w[j] >> 16));
    f[4 * j] = a.x; f[4 * j + 1] = a.y; f[4 * j + 2] = c.x; f[4 * j + 3] = c.y;
  }
}

// G = 1, 2 on CUDA cores, the loop of decode_kernel over e4m3 rows: a 16-byte load carries 16 values, so D/16 lanes
// cover a row and a warp-wide load covers twice the rows of the 16-bit kernel. p.scale_log2 includes k_scale.
template <int D, int G, typename T>
__global__ void __launch_bounds__(NUM_THREADS, 2)
decode_kernel(const Params p, const float v_scale) {
  constexpr int NLOAD = 8 / G;        // 16-byte loads in flight per lane for K (and again for V); G = 2 needs the registers
  constexpr int LPR = D / 16;         // lanes per KV row
  constexpr int RPW = 32 / LPR;       // rows per warp-wide load
  constexpr int TILE = NLOAD * RPW;   // keys per warp iteration

  const int split = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sub = lane % LPR;         // which 16-element slice of the row
  const int rsel = lane / LPR;        // which row of the warp-wide load

  const int ctx = max(0, min(p.context_lens[b], p.capacity));
  int chunk = (ctx + p.splits - 1) / p.splits;
  chunk = ((chunk + TILE - 1) / TILE) * TILE;
  const int k_begin = min(split * chunk, ctx);
  const int k_end = min(k_begin + chunk, ctx);

  float qf[G][16];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const T* qp = reinterpret_cast<const T*>(p.q) + (static_cast<int64_t>(b) * p.Hq + kvh * G + g) * D + sub * 16;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint4 raw = *reinterpret_cast<const uint4*>(qp + 8 * h);
      const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = Pack2<T>::unpack(w[j]);
        qf[g][8 * h + 2 * j] = f.x * p.scale_log2;
        qf[g][8 * h + 2 * j + 1] = f.y * p.scale_log2;
      }
    }
  }
  float m_run[G], l_run[G], acc[G][16];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    m_run[g] = -INFINITY;
    l_run[g] = 0.f;
#pragma unroll
    for (int e = 0; e < 16; ++e) acc[g][e] = 0.f;
  }

  const uint8_t* kc = reinterpret_cast<const uint8_t*>(p.k_cache);
  const uint8_t* vc = reinterpret_cast<const uint8_t*>(p.v_cache);
  const int32_t* bt = p.block_table + static_cast<int64_t>(b) * p.max_blocks_per_seq;
  const bool bs_pow2 = (p.block_size & (p.block_size - 1)) == 0;
  const int bs_shift = bs_pow2 ? (31 - __clz(p.block_size)) : 0;

  for (int t0 = k_begin + warp * TILE; t0 < k_end; t0 += NUM_WARPS * TILE) {
    uint4 kraw[NLOAD], vraw[NLOAD];
    bool valid[NLOAD];
#pragma unroll
    for (int i = 0; i < NLOAD; ++i) {
      const int key = t0 + i * RPW + rsel;
      valid[i] = key < k_end;
      if (valid[i]) {   // bytes of keys at or past the end are never loaded
        const int bi = bs_pow2 ? (key >> bs_shift) : (key / p.block_size);
        const int in_blk = bs_pow2 ? (key & (p.block_size - 1)) : (key - bi * p.block_size);
        const int64_t off = ((static_cast<int64_t>(bt[bi]) * p.num_layers + p.layer_idx) * p.block_size + in_blk) *
                                (static_cast<int64_t>(p.Hkv) * D) + kvh * D + sub * 16;
        kraw[i] = ld_stream(kc + off);
        vraw[i] = ld_stream(vc + off);
      } else {
        kraw[i] = uint4{0, 0, 0, 0};
        vraw[i] = uint4{0, 0, 0, 0};
      }
    }
    float s[G][NLOAD];
#pragma unroll
    for (int i = 0; i < NLOAD; ++i) {
      float kf[16];
      widen16(kraw[i], kf);
#pragma unroll
      for (int g = 0; g < G; ++g) {
        float d = 0.f;
#pragma unroll
        for (int e = 0; e < 16; ++e) d = fmaf(qf[g][e], kf[e], d);
#pragma unroll
        for (int x = LPR / 2; x >= 1; x >>= 1) d += __shfl_xor_sync(0xffffffffu, d, x);
        s[g][i] = valid[i] ? d : -INFINITY;
      }
    }
    float pr[G][NLOAD];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      float tmax = s[g][0];
#pragma unroll
      for (int i = 1; i < NLOAD; ++i) tmax = fmaxf(tmax, s[g][i]);
#pragma unroll
      for (int x = LPR; x < 32; x <<= 1) tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, x));
      const float m_new = fmaxf(m_run[g], tmax);
      const float m_safe = (m_new == -INFINITY) ? 0.f : m_new;
      const float corr = fast_exp2(m_run[g] - m_safe);
      m_run[g] = m_new;
      l_run[g] *= corr;
#pragma unroll
      for (int e = 0; e < 16; ++e) acc[g][e] *= corr;
#pragma unroll
      for (int i = 0; i < NLOAD; ++i) {
        pr[g][i] = fast_exp2(s[g][i] - m_safe);
        l_run[g] += pr[g][i];
      }
    }
#pragma unroll
    for (int i = 0; i < NLOAD; ++i) {
      float vf[16];
      widen16(vraw[i], vf);
#pragma unroll
      for (int g = 0; g < G; ++g) {
#pragma unroll
        for (int e = 0; e < 16; ++e) acc[g][e] = fmaf(pr[g][i], vf[e], acc[g][e]);
      }
    }
  }

#pragma unroll
  for (int g = 0; g < G; ++g) {
#pragma unroll
    for (int x = LPR; x < 32; x <<= 1) {
      l_run[g] += __shfl_xor_sync(0xffffffffu, l_run[g], x);
#pragma unroll
      for (int e = 0; e < 16; ++e) acc[g][e] += __shfl_xor_sync(0xffffffffu, acc[g][e], x);
    }
  }
  __shared__ float sm_m[NUM_WARPS][G];
  __shared__ float sm_l[NUM_WARPS][G];
  __shared__ float sm_acc[NUM_WARPS][G][D];
  if (rsel == 0) {
#pragma unroll
    for (int g = 0; g < G; ++g) {
#pragma unroll
      for (int e = 0; e < 16; ++e) sm_acc[warp][g][sub * 16 + e] = acc[g][e];
      if (sub == 0) {
        sm_m[warp][g] = m_run[g];
        sm_l[warp][g] = l_run[g];
      }
    }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < G * D; idx += NUM_THREADS) {
    const int g = idx / D;
    const int d = idx - g * D;
    float m = -INFINITY;
#pragma unroll
    for (int w = 0; w < NUM_WARPS; ++w) m = fmaxf(m, sm_m[w][g]);
    const float m_safe = (m == -INFINITY) ? 0.f : m;
    float l = 0.f, o = 0.f;
#pragma unroll
    for (int w = 0; w < NUM_WARPS; ++w) {
      const float c = fast_exp2(sm_m[w][g] - m_safe);
      l = fmaf(sm_l[w][g], c, l);
      o = fmaf(sm_acc[w][g][d], c, o);
    }
    const float out = l > 0.f ? o / l * v_scale : 0.f;
    const float lse = l > 0.f ? (m + log2f(l)) * kLn2 : -INFINITY;
    const int h = kvh * G + g;
    if (p.splits == 1) {
      T* op = reinterpret_cast<T*>(p.o) + (static_cast<int64_t>(b) * p.Hq + h) * D + d;
      if constexpr (Pack2<T>::kIsBf16) *op = __float2bfloat16_rn(out);
      else *op = __float2half_rn(out);
      if (d == 0 && p.lse != nullptr) p.lse[static_cast<int64_t>(b) * p.Hq + h] = lse;
    } else {
      const int64_t row = (static_cast<int64_t>(b) * p.Hq + h) * p.splits + split;
      p.part_o[row * D + d] = out;
      if (d == 0) p.part_lse[row] = lse;
    }
  }
}

// G = 3..16 on mma.sync m16n8k16, the register-staged schedule of decode_gqa_mma_kernel over e4m3 rows.
//   Q K^T : lane (g,t) loads K[key g][64m + 16t .. +16): one 16-byte load, widened to eight f16x2 words, feeds four
//           k-steps (word pair j of the load is k-step j; the Q fragments carry the same permutation of the contraction
//           index). A warp iteration covers 32 keys, four n-tiles of 8, so a tile is as many bytes as the 16-bit kernel's.
//   P V   : lane (g,t) loads the D/8 bytes V[key][D/8 * g .. +D/8) of keys {2t, 2t+1, 2t+8, 2t+9} of each 16-key k-step;
//           PRMT pairs byte j of two keys and one cvt widens the pair into a B fragment. Output column c of n-tile j is
//           dim D/8 * c + j (undone at the final store).
// The MMA runs in f16 for both q types. ptxas has no e4m3 -> bf16x2 conversion on sm_100a; an exact widening by bit
// operations (shift the 7 magnitude bits into bf16 position, multiply by 2^120) costs four instructions per pair instead
// of one, on a kernel whose issue slots already carry the MMAs, the widening and the softmax of twice the keys per byte.
// A bf16 q is converted to f16 once per CTA instead: exact for |q| in [2^-14, 65504] (bf16 has 8 significant bits, f16
// has 11), which covers the projected queries of a model by orders of magnitude; P in f16 rounds finer than bf16 would.
template <int D, typename T>
__global__ void __launch_bounds__(GQA_WARPS * 32, GqaMinCtas<D>::value)
decode_gqa_mma_kernel(const Params p, const int G, const float v_scale) {
  constexpr int TILE = 32;       // keys per warp iteration
  constexpr int MB = D / 64;     // 64-dim blocks of the head dimension (one 16-byte K load per lane, four k-steps)
  constexpr int VW = D / 8;      // V bytes a lane loads per key (= n-tiles of the P V product)
  constexpr int VWORDS = VW / 4;

  const int split = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;

  const int ctx = max(0, min(p.context_lens[b], p.capacity));
  int chunk = (ctx + p.splits - 1) / p.splits;
  chunk = ((chunk + TILE - 1) / TILE) * TILE;
  const int k_begin = min(split * chunk, ctx);
  const int k_end = min(k_begin + chunk, ctx);

  // Q fragments (f16) for rows g and g+8 (zero rows beyond the group): word i of block m = dims 64m + 16t + 2i, +1
  uint32_t qa[MB][8], qb[MB][8];
  {
    const T* qbase = reinterpret_cast<const T*>(p.q) + (static_cast<int64_t>(b) * p.Hq + kvh * G) * D;
#pragma unroll
    for (int m = 0; m < MB; ++m) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint4 ra = uint4{0, 0, 0, 0}, rb = uint4{0, 0, 0, 0};
        if (g < G) ra = *reinterpret_cast<const uint4*>(qbase + static_cast<int64_t>(g) * D + 64 * m + 16 * t + 8 * h);
        if (g + 8 < G) rb = *reinterpret_cast<const uint4*>(qbase + static_cast<int64_t>(g + 8) * D + 64 * m + 16 * t + 8 * h);
        const uint32_t wa[4] = {ra.x, ra.y, ra.z, ra.w}, wb[4] = {rb.x, rb.y, rb.z, rb.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if constexpr (Pack2<T>::kIsBf16) {
            const float2 fa = Pack2<T>::unpack(wa[j]), fb = Pack2<T>::unpack(wb[j]);
            qa[m][4 * h + j] = Pack2<__half>::pack(fa.x, fa.y);
            qb[m][4 * h + j] = Pack2<__half>::pack(fb.x, fb.y);
          } else {
            qa[m][4 * h + j] = wa[j];
            qb[m][4 * h + j] = wb[j];
          }
        }
      }
    }
  }
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  float o[VW][4];
#pragma unroll
  for (int n = 0; n < VW; ++n) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }

  const uint8_t* kc = reinterpret_cast<const uint8_t*>(p.k_cache);
  const uint8_t* vc = reinterpret_cast<const uint8_t*>(p.v_cache);
  const int32_t* bt = p.block_table + static_cast<int64_t>(b) * p.max_blocks_per_seq;
  auto row_offset = [&](int key) -> int64_t {  // byte offset of (key, kvh, dim 0)
    const int bi = key / p.block_size;
    const int in_blk = key - bi * p.block_size;
    return ((static_cast<int64_t>(bt[bi]) * p.num_layers + p.layer_idx) * p.block_size + in_blk) *
               (static_cast<int64_t>(p.Hkv) * D) + kvh * D;
  };

  auto issue_tile = [&](const int t0, uint4 (&kr)[4][MB], uint32_t (&vr)[2][4][VWORDS]) {
#pragma unroll
    for (int kg = 0; kg < 4; ++kg) {
      const int key = t0 + kg * 8 + g;
      const bool valid = key < k_end;
      const int64_t off = valid ? row_offset(key) + 16 * t : 0;
#pragma unroll
      for (int m = 0; m < MB; ++m) kr[kg][m] = ld_stream_if(kc + off + 64 * m, valid);
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int key = t0 + 16 * s + 2 * t + (j & 1) + (j >> 1) * 8;
        const bool valid = key < k_end;
        const int64_t off = valid ? row_offset(key) + VW * g : 0;
        if constexpr (VWORDS == 4) {
          const uint4 r = ld_stream_if(vc + off, valid);
          vr[s][j][0] = r.x; vr[s][j][1] = r.y; vr[s][j][2] = r.z; vr[s][j][3] = r.w;
        } else {
          const uint2 r = ld_stream8_if(vc + off, valid);
          vr[s][j][0] = r.x; vr[s][j][1] = r.y;
        }
      }
    }
  };
  // the two 16-key halves of a tile one after the other: the scores and probabilities of 16 keys are live at a time
  auto compute_tile = [&](const int t0, const uint4 (&kr)[4][MB], const uint32_t (&vr)[2][4][VWORDS]) {
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      // ---- S = Q K^T (rows g, g+8; keys 16s + kg*8 + 2t, +1) ----
      float sc[2][4];
#pragma unroll
      for (int kg = 0; kg < 2; ++kg) {
        sc[kg][0] = sc[kg][1] = sc[kg][2] = sc[kg][3] = 0.f;
#pragma unroll
        for (int m = 0; m < MB; ++m) {
          const uint4 kw = kr[2 * s + kg][m];
          const uint32_t w[4] = {kw.x, kw.y, kw.z, kw.w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
            mma_16816<__half>(sc[kg], qa[m][2 * j], qb[m][2 * j], qa[m][2 * j + 1], qb[m][2 * j + 1], widen2(w[j]),
                              widen2(w[j] >> 16));
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = t0 + 16 * s + kg * 8 + 2 * t + (e & 1);
          sc[kg][e] = key < k_end ? sc[kg][e] * p.scale_log2 : -INFINITY;
        }
      }
      // ---- online softmax for the two rows this lane holds ----
      float pr[2][4];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        float tmax = fmaxf(fmaxf(sc[0][2 * r], sc[0][2 * r + 1]), fmaxf(sc[1][2 * r], sc[1][2 * r + 1]));
        tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, 1));
        tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, 2));
        const float m_new = fmaxf(m_run[r], tmax);
        const float m_safe = (m_new == -INFINITY) ? 0.f : m_new;
        const float corr = fast_exp2(m_run[r] - m_safe);
        m_run[r] = m_new;
        l_run[r] *= corr;
#pragma unroll
        for (int n = 0; n < VW; ++n) { o[n][2 * r] *= corr; o[n][2 * r + 1] *= corr; }
#pragma unroll
        for (int kg = 0; kg < 2; ++kg) {
          pr[kg][2 * r] = fast_exp2(sc[kg][2 * r] - m_safe);
          pr[kg][2 * r + 1] = fast_exp2(sc[kg][2 * r + 1] - m_safe);
          l_run[r] += pr[kg][2 * r] + pr[kg][2 * r + 1];
        }
      }
      // ---- O += P V ----
      const uint32_t pa0 = Pack2<__half>::pack(pr[0][0], pr[0][1]), pa1 = Pack2<__half>::pack(pr[0][2], pr[0][3]);
      const uint32_t pa2 = Pack2<__half>::pack(pr[1][0], pr[1][1]), pa3 = Pack2<__half>::pack(pr[1][2], pr[1][3]);
#pragma unroll
      for (int q4 = 0; q4 < VWORDS; ++q4) {
        // bytes of keys (2t, 2t+1) and (2t+8, 2t+9), interleaved: [k0.b0, k1.b0, k0.b1, k1.b1] and [k0.b2, k1.b2, ...]
        const uint32_t lo01 = __byte_perm(vr[s][0][q4], vr[s][1][q4], 0x5140);
        const uint32_t hi01 = __byte_perm(vr[s][0][q4], vr[s][1][q4], 0x7362);
        const uint32_t lo23 = __byte_perm(vr[s][2][q4], vr[s][3][q4], 0x5140);
        const uint32_t hi23 = __byte_perm(vr[s][2][q4], vr[s][3][q4], 0x7362);
        mma_16816<__half>(o[4 * q4 + 0], pa0, pa1, pa2, pa3, widen2(lo01), widen2(lo23));
        mma_16816<__half>(o[4 * q4 + 1], pa0, pa1, pa2, pa3, widen2(lo01 >> 16), widen2(lo23 >> 16));
        mma_16816<__half>(o[4 * q4 + 2], pa0, pa1, pa2, pa3, widen2(hi01), widen2(hi23));
        mma_16816<__half>(o[4 * q4 + 3], pa0, pa1, pa2, pa3, widen2(hi01 >> 16), widen2(hi23 >> 16));
      }
    }
  };
  constexpr int STEP = GQA_WARPS * TILE;
  {
    uint4 krA[4][MB], krB[4][MB];
    uint32_t vrA[2][4][VWORDS], vrB[2][4][VWORDS];
    int t0 = k_begin + warp * TILE;
    if (t0 < k_end) issue_tile(t0, krA, vrA);
    for (; t0 < k_end; t0 += 2 * STEP) {
      if (t0 + STEP < k_end) issue_tile(t0 + STEP, krB, vrB);
      compute_tile(t0, krA, vrA);
      if (t0 + 2 * STEP < k_end) issue_tile(t0 + 2 * STEP, krA, vrA);
      if (t0 + STEP < k_end) compute_tile(t0 + STEP, krB, vrB);
    }
  }

  // ---- combine: lanes of a row quad, then the warps of the CTA through shared memory ----
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
  }
  __shared__ float sm_m[GQA_WARPS * 16];
  __shared__ float sm_l[GQA_WARPS * 16];
  __shared__ float sm_acc[GQA_WARPS * 16 * D];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int row = g + 8 * r;
    if (row < G) {
      if (t == 0) { sm_m[warp * 16 + row] = m_run[r]; sm_l[warp * 16 + row] = l_run[r]; }
#pragma unroll
      for (int n = 0; n < VW; ++n) {
        sm_acc[(warp * 16 + row) * D + VW * (2 * t) + n] = o[n][2 * r];
        sm_acc[(warp * 16 + row) * D + VW * (2 * t + 1) + n] = o[n][2 * r + 1];
      }
    }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < G * D; idx += GQA_WARPS * 32) {
    const int row = idx / D, d = idx - row * D;
    float m = -INFINITY;
#pragma unroll
    for (int w = 0; w < GQA_WARPS; ++w) m = fmaxf(m, sm_m[w * 16 + row]);
    const float m_safe = (m == -INFINITY) ? 0.f : m;
    float l = 0.f, acc = 0.f;
#pragma unroll
    for (int w = 0; w < GQA_WARPS; ++w) {
      const float c = fast_exp2(sm_m[w * 16 + row] - m_safe);
      l = fmaf(sm_l[w * 16 + row], c, l);
      acc = fmaf(sm_acc[(w * 16 + row) * D + d], c, acc);
    }
    const float out = l > 0.f ? acc / l * v_scale : 0.f;
    const float lse = l > 0.f ? (m + log2f(l)) * kLn2 : -INFINITY;
    const int h = kvh * G + row;
    if (p.splits == 1) {
      T* op = reinterpret_cast<T*>(p.o) + (static_cast<int64_t>(b) * p.Hq + h) * D + d;
      if constexpr (Pack2<T>::kIsBf16) *op = __float2bfloat16_rn(out);
      else *op = __float2half_rn(out);
      if (d == 0 && p.lse != nullptr) p.lse[static_cast<int64_t>(b) * p.Hq + h] = lse;
    } else {
      const int64_t prow = (static_cast<int64_t>(b) * p.Hq + h) * p.splits + split;
      p.part_o[prow * D + d] = out;
      if (d == 0) p.part_lse[prow] = lse;
    }
  }
}

template <int D, typename T>
int launch_decode(int G, const Params& p, float v_scale, cudaStream_t stream) {
  dim3 grid(p.splits, p.Hkv, p.B);
  if (G >= 3) {
    decode_gqa_mma_kernel<D, T><<<grid, GQA_WARPS * 32, 0, stream>>>(p, G, v_scale);
    B200_CUDA_OK(cudaGetLastError());
    note_launch("fp8_decode_gqa_mma_kernel");
  } else {
    if (G == 1) decode_kernel<D, 1, T><<<grid, NUM_THREADS, 0, stream>>>(p, v_scale);
    else decode_kernel<D, 2, T><<<grid, NUM_THREADS, 0, stream>>>(p, v_scale);
    B200_CUDA_OK(cudaGetLastError());
    note_launch("fp8_decode_kernel");
  }
  if (p.splits > 1) {
    decode_reduce_kernel<D, T><<<p.B * p.Hq, D, 0, stream>>>(p.part_o, p.part_lse, p.o, p.lse, p.splits);
    B200_CUDA_OK(cudaGetLastError());
    note_launch("decode_reduce_kernel");
  }
  return B200_OK;
}

inline bool scale_ok(float s) { return s > 0.f && s <= 3.402823466e38f; }  // false for NaN, +-inf, 0 and negatives

}  // namespace fp8
}  // namespace decode
}  // namespace b200

extern "C" {

int b200_fa_decode_num_splits(int B, int Hq, int Hkv, int D, int max_context_len) {
  if (B <= 0 || Hq <= 0 || Hkv <= 0 || D <= 0 || max_context_len <= 0) return 1;
  const int sms = b200::sm_count();
  const int64_t ctas = static_cast<int64_t>(B) * Hkv;   // CTAs per split
  const int G = Hq / Hkv;
  // resident CTAs: 2 per SM for the MHA kernel and the D = 128 tensor-core GQA kernel, 3 for the D = 64 GQA kernel
  const int64_t resident = static_cast<int64_t>(sms) * ((G >= 3 && G <= 16 && D == 64) ? 3 : 2);
  // Measured (tests/decode_split_probe.py, profiles/r2_decode_splits.jsonl): a problem that fits in one wave is fastest
  // with ONE nearly full wave and a power-of-two split count (even key ranges) — MQA B=32 8K: 8 splits 46 us vs the 32 of
  // the old ">= 4 waves" rule 79 us; GQA B=8: 4 -> 64 us vs 28 -> 81 us (5 splits = 1.08 waves: 89 us); GQA B=1 32K: 32 ->
  // 40 us vs 128 -> 56 us. If the largest such wave leaves more than a fifth of the slots empty and the problem is large
  // enough to be bandwidth-bound (>= 256 MB of K/V), several waves win instead (D = 64 GQA B=64: 8 splits 108 us vs 1
  // split 127 us). One to four waves: 1, 2 or 4 splits by how full the last wave is. Four waves and more: not split.
  int splits = 1;
  if (ctas < resident) {
    int s1 = 1;
    while (ctas * (s1 * 2) <= resident) s1 *= 2;
    splits = s1;
    const double fill = static_cast<double>(ctas * s1) / static_cast<double>(resident);
    const double kv_bytes = 2.0 * static_cast<double>(ctas) * max_context_len * D * 2.0;
    if (fill < 0.8 && kv_bytes >= 256.0e6) {
      int s4 = s1;
      while (ctas * s4 < 4 * resident) s4 *= 2;
      splits = s4;
    }
  } else if (ctas < 4 * resident) {
    double best_eff = 0.0;
    for (int s = 1; s <= 4; s *= 2) {
      const double waves = static_cast<double>(ctas * s) / static_cast<double>(resident);
      const double eff = waves / static_cast<double>(static_cast<int64_t>(waves + 0.999999));
      if (eff > best_eff * 1.02) { best_eff = eff; splits = s; }
    }
  }
  const int max_by_len = (max_context_len + 255) / 256;  // keep >= 256 keys per split
  if (splits > max_by_len) splits = max_by_len;
  if (splits < 1) splits = 1;
  if (splits > 128) splits = 128;
  return splits;
}

int64_t b200_fa_decode_workspace_bytes(int B, int Hq, int Hkv, int D, int max_context_len, int num_splits) {
  int splits = num_splits > 0 ? num_splits : b200_fa_decode_num_splits(B, Hq, Hkv, D, max_context_len);
  if (splits <= 1) return 0;
  return static_cast<int64_t>(B) * Hq * splits * (D + 1) * static_cast<int64_t>(sizeof(float));
}

int b200_fa_decode(const void* q, const void* k_cache, const void* v_cache, void* o, float* lse, int B, int Hq, int Hkv,
                   int D, const int32_t* context_lens, int max_context_len, float softmax_scale, int layout,
                   int64_t kv_batch_stride, int64_t kv_token_stride, const int32_t* block_table,
                   int max_blocks_per_seq, int block_size, int num_layers, int layer_idx, int num_splits,
                   void* workspace, int64_t workspace_bytes, int dtype, void* stream) {
  using namespace b200;
  B200_CHECK_ARG(q && k_cache && v_cache && o && context_lens, "decode: NULL pointer argument");
  B200_CHECK_ARG(B > 0 && Hq > 0 && Hkv > 0 && Hq % Hkv == 0, "decode: bad B/Hq/Hkv = %d/%d/%d", B, Hq, Hkv);
  B200_CHECK_ARG(D == 64 || D == 128, "decode: head_dim %d unsupported (64, 128)", D);
  B200_CHECK_ARG(dtype == B200_DTYPE_BF16 || dtype == B200_DTYPE_FP16, "decode: dtype must be bf16 or fp16");
  B200_CHECK_ARG(layout == B200_KV_CONTIGUOUS || layout == B200_KV_PAGED, "decode: unknown KV layout %d", layout);
  B200_CHECK_ARG(max_context_len > 0, "decode: max_context_len must be positive");
  B200_CHECK_ARG(((uintptr_t)q & 15) == 0 && ((uintptr_t)k_cache & 15) == 0 && ((uintptr_t)v_cache & 15) == 0 &&
                     ((uintptr_t)o & 15) == 0,
                 "decode: pointers must be 16-byte aligned");
  if (layout == B200_KV_PAGED) {
    B200_CHECK_ARG(block_table != nullptr && block_size > 0 && max_blocks_per_seq > 0 && num_layers > 0 &&
                       layer_idx >= 0 && layer_idx < num_layers,
                   "decode: bad paged-cache arguments");
  } else {
    B200_CHECK_ARG(kv_token_stride >= static_cast<int64_t>(Hkv) * D && kv_token_stride % 8 == 0 &&
                       kv_batch_stride % 8 == 0,
                   "decode: bad contiguous-cache strides");
  }
  int splits = num_splits > 0 ? num_splits : b200_fa_decode_num_splits(B, Hq, Hkv, D, max_context_len);
  decode::Params p;
  p.q = q; p.k_cache = k_cache; p.v_cache = v_cache; p.o = o; p.lse = lse;
  p.part_o = nullptr; p.part_lse = nullptr;
  if (splits > 1) {
    const int64_t need = b200_fa_decode_workspace_bytes(B, Hq, Hkv, D, max_context_len, splits);
    if (workspace == nullptr || workspace_bytes < need)
      return set_error(B200_ERR_WORKSPACE, "decode workspace too small: need %lld bytes, got %lld", (long long)need,
                       (long long)workspace_bytes);
    p.part_o = static_cast<float*>(workspace);
    p.part_lse = p.part_o + static_cast<int64_t>(B) * Hq * splits * D;
  }
  p.context_lens = context_lens; p.block_table = block_table;
  p.B = B; p.Hq = Hq; p.Hkv = Hkv; p.splits = splits;
  p.scale_log2 = softmax_scale * decode::kLog2e;
  p.kv_batch_stride = kv_batch_stride; p.kv_token_stride = kv_token_stride;
  p.max_blocks_per_seq = max_blocks_per_seq; p.block_size = block_size; p.num_layers = num_layers;
  p.layer_idx = layer_idx;
  // paged: what the block table can address; contiguous: the caller's bound on the lengths (ops.py passes S_max)
  p.capacity = layout == B200_KV_PAGED ? (max_context_len < max_blocks_per_seq * block_size ? max_context_len : max_blocks_per_seq * block_size)
                                       : max_context_len;
  const int G = Hq / Hkv;
  const bool paged = layout == B200_KV_PAGED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (D == 128) {
    return dtype == B200_DTYPE_BF16 ? decode::dispatch_group<128, __nv_bfloat16>(G, p, paged, s)
                                    : decode::dispatch_group<128, __half>(G, p, paged, s);
  }
  return dtype == B200_DTYPE_BF16 ? decode::dispatch_group<64, __nv_bfloat16>(G, p, paged, s)
                                  : decode::dispatch_group<64, __half>(G, p, paged, s);
}

int b200_kv_append(const void* key, const void* value, void* k_cache, void* v_cache, int B, int Hkv, int D,
                   const int32_t* context_lens, int layout, int64_t kv_batch_stride, int64_t kv_token_stride,
                   const int32_t* block_table, int max_blocks_per_seq, int block_size, int num_layers, int layer_idx,
                   int dtype, void* stream) {
  using namespace b200;
  B200_CHECK_ARG(key && value && k_cache && v_cache && context_lens, "kv_append: NULL pointer argument");
  B200_CHECK_ARG(B > 0 && Hkv > 0 && D > 0 && (Hkv * D) % 8 == 0, "kv_append: bad sizes");
  B200_CHECK_ARG(layout == B200_KV_CONTIGUOUS || layout == B200_KV_PAGED, "kv_append: unknown KV layout %d", layout);
  if (layout == B200_KV_PAGED)
    B200_CHECK_ARG(block_table != nullptr && block_size > 0 && max_blocks_per_seq > 0 && num_layers > 0 &&
                       layer_idx >= 0 && layer_idx < num_layers,
                   "kv_append: bad paged-cache arguments");
  (void)dtype;  // a 16-bit copy: the element type does not matter
  // capacity in tokens: paged = what the block table addresses; contiguous = max_blocks_per_seq when the caller passes the
  // cache's S_max there (block_size == 0 marks that use), else unchecked
  const int capacity = layout == B200_KV_PAGED ? max_blocks_per_seq * block_size
                                               : (max_blocks_per_seq > 0 ? max_blocks_per_seq : 0x7fffffff);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  decode::kv_append_kernel<uint16_t><<<B, 128, 0, s>>>(
      static_cast<const uint16_t*>(key), static_cast<const uint16_t*>(value), static_cast<uint16_t*>(k_cache),
      static_cast<uint16_t*>(v_cache), context_lens, Hkv * D, layout, kv_batch_stride, kv_token_stride, block_table,
      max_blocks_per_seq, block_size, num_layers, layer_idx, capacity);
  B200_CUDA_OK(cudaGetLastError());
  note_launch("kv_append_kernel");
  return B200_OK;
}

int b200_fa_decode_fp8(const void* q, const void* k_cache, const void* v_cache, void* o, float* lse, int B, int Hq, int Hkv,
                       int D, const int32_t* context_lens, int max_context_len, float softmax_scale, int layout,
                       const int32_t* block_table, int max_blocks_per_seq, int block_size, int num_layers, int layer_idx,
                       int num_splits, void* workspace, int64_t workspace_bytes, float k_scale, float v_scale, int dtype,
                       void* stream) {
  using namespace b200;
  B200_CHECK_ARG(q && k_cache && v_cache && o && context_lens, "decode_fp8: NULL pointer argument");
  B200_CHECK_ARG(B > 0 && Hq > 0 && Hkv > 0 && Hq % Hkv == 0 && Hq / Hkv <= 16,
                 "decode_fp8: bad B/Hq/Hkv = %d/%d/%d (Hq/Hkv must be 1 .. 16)", B, Hq, Hkv);
  B200_CHECK_ARG(D == 64 || D == 128, "decode_fp8: head_dim %d unsupported (64, 128)", D);
  B200_CHECK_ARG(dtype == B200_DTYPE_BF16 || dtype == B200_DTYPE_FP16, "decode_fp8: q dtype must be bf16 or fp16");
  B200_CHECK_ARG(layout == B200_KV_CONTIGUOUS || layout == B200_KV_PAGED, "decode_fp8: unknown KV layout %d", layout);
  if (layout != B200_KV_PAGED)
    return set_error(B200_ERR_UNSUPPORTED, "decode_fp8: an FP8 cache exists in the paged layout only");
  B200_CHECK_ARG(max_context_len > 0, "decode_fp8: max_context_len must be positive");
  B200_CHECK_ARG(((uintptr_t)q & 15) == 0 && ((uintptr_t)k_cache & 15) == 0 && ((uintptr_t)v_cache & 15) == 0 &&
                     ((uintptr_t)o & 15) == 0,
                 "decode_fp8: pointers must be 16-byte aligned");
  B200_CHECK_ARG(block_table != nullptr && block_size > 0 && max_blocks_per_seq > 0 && num_layers > 0 && layer_idx >= 0 &&
                     layer_idx < num_layers,
                 "decode_fp8: bad paged-cache arguments");
  B200_CHECK_ARG(decode::fp8::scale_ok(k_scale) && decode::fp8::scale_ok(v_scale),
                 "decode_fp8: k_scale and v_scale must be positive and finite (got %g, %g)", k_scale, v_scale);
  const int splits = num_splits > 0 ? num_splits : b200_fa_decode_num_splits(B, Hq, Hkv, D, max_context_len);
  decode::Params p;
  p.q = q; p.k_cache = k_cache; p.v_cache = v_cache; p.o = o; p.lse = lse;
  p.part_o = nullptr; p.part_lse = nullptr;
  if (splits > 1) {
    const int64_t need = b200_fa_decode_workspace_bytes(B, Hq, Hkv, D, max_context_len, splits);
    if (workspace == nullptr || workspace_bytes < need)
      return set_error(B200_ERR_WORKSPACE, "decode_fp8 workspace too small: need %lld bytes, got %lld", (long long)need,
                       (long long)workspace_bytes);
    p.part_o = static_cast<float*>(workspace);
    p.part_lse = p.part_o + static_cast<int64_t>(B) * Hq * splits * D;
  }
  p.context_lens = context_lens; p.block_table = block_table;
  p.B = B; p.Hq = Hq; p.Hkv = Hkv; p.splits = splits;
  p.scale_log2 = softmax_scale * k_scale * decode::kLog2e;   // q . (byte * k_scale) = (q . byte) * k_scale
  p.kv_batch_stride = 0; p.kv_token_stride = 0;
  p.max_blocks_per_seq = max_blocks_per_seq; p.block_size = block_size; p.num_layers = num_layers;
  p.layer_idx = layer_idx;
  p.capacity = max_context_len < max_blocks_per_seq * block_size ? max_context_len : max_blocks_per_seq * block_size;
  const int G = Hq / Hkv;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (D == 128) {
    return dtype == B200_DTYPE_BF16 ? decode::fp8::launch_decode<128, __nv_bfloat16>(G, p, v_scale, s)
                                    : decode::fp8::launch_decode<128, __half>(G, p, v_scale, s);
  }
  return dtype == B200_DTYPE_BF16 ? decode::fp8::launch_decode<64, __nv_bfloat16>(G, p, v_scale, s)
                                  : decode::fp8::launch_decode<64, __half>(G, p, v_scale, s);
}

int b200_kv_append_fp8(const void* key, const void* value, void* k_cache, void* v_cache, int B, int n_tokens, int Hkv, int D,
                       const int32_t* context_lens, const int32_t* block_table, int max_blocks_per_seq, int block_size,
                       int num_layers, int layer_idx, float k_scale, float v_scale, int dtype, void* stream) {
  using namespace b200;
  B200_CHECK_ARG(key && value && k_cache && v_cache && context_lens, "kv_append_fp8: NULL pointer argument");
  B200_CHECK_ARG(B > 0 && B <= 65535 && n_tokens > 0 && Hkv > 0, "kv_append_fp8: bad sizes B/n_tokens/Hkv = %d/%d/%d", B,
                 n_tokens, Hkv);
  B200_CHECK_ARG(D == 64 || D == 128, "kv_append_fp8: head_dim %d unsupported (64, 128)", D);
  B200_CHECK_ARG(dtype == B200_DTYPE_BF16 || dtype == B200_DTYPE_FP16, "kv_append_fp8: key dtype must be bf16 or fp16");
  B200_CHECK_ARG(((uintptr_t)key & 15) == 0 && ((uintptr_t)value & 15) == 0 && ((uintptr_t)k_cache & 15) == 0 &&
                     ((uintptr_t)v_cache & 15) == 0,
                 "kv_append_fp8: pointers must be 16-byte aligned");
  B200_CHECK_ARG(block_table != nullptr && block_size > 0 && max_blocks_per_seq > 0 && num_layers > 0 && layer_idx >= 0 &&
                     layer_idx < num_layers,
                 "kv_append_fp8: bad paged-cache arguments");
  B200_CHECK_ARG(decode::fp8::scale_ok(k_scale) && decode::fp8::scale_ok(v_scale),
                 "kv_append_fp8: k_scale and v_scale must be positive and finite (got %g, %g)", k_scale, v_scale);
  const dim3 grid(n_tokens, B);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint8_t* kd = static_cast<uint8_t*>(k_cache);
  uint8_t* vd = static_cast<uint8_t*>(v_cache);
  if (dtype == B200_DTYPE_BF16)
    decode::fp8::kv_append_kernel<__nv_bfloat16><<<grid, 128, 0, s>>>(
        static_cast<const __nv_bfloat16*>(key), static_cast<const __nv_bfloat16*>(value), kd, vd, context_lens, n_tokens,
        Hkv * D, block_table, max_blocks_per_seq, block_size, num_layers, layer_idx, k_scale, v_scale);
  else
    decode::fp8::kv_append_kernel<__half><<<grid, 128, 0, s>>>(
        static_cast<const __half*>(key), static_cast<const __half*>(value), kd, vd, context_lens, n_tokens, Hkv * D,
        block_table, max_blocks_per_seq, block_size, num_layers, layer_idx, k_scale, v_scale);
  B200_CUDA_OK(cudaGetLastError());
  note_launch("fp8_kv_append_kernel");
  return B200_OK;
}

int b200_lse_merge(float* o_acc, float* lse_acc, const void* o_b, const float* lse_b, int B, int Sq, int Hq, int D,
                   const int64_t ob_strides[3], int dtype, void* stream) {
  using namespace b200;
  B200_CHECK_ARG(o_acc && lse_acc && o_b && lse_b && ob_strides, "lse_merge: NULL pointer argument");
  B200_CHECK_ARG(B > 0 && Sq > 0 && Hq > 0 && D > 0 && D % 8 == 0, "lse_merge: bad sizes");
  B200_CHECK_ARG(ob_strides[0] % 8 == 0 && ob_strides[1] % 8 == 0 && ob_strides[2] % 8 == 0 &&
                     ((uintptr_t)o_b & 15) == 0 && ((uintptr_t)o_acc & 15) == 0,
                 "lse_merge: o_b strides must be multiples of 8 elements and pointers 16-byte aligned");
  B200_CHECK_ARG(dtype == B200_DTYPE_BF16 || dtype == B200_DTYPE_FP16, "lse_merge: dtype must be bf16 or fp16");
  const int64_t total = static_cast<int64_t>(B) * Sq * Hq * (D / 8);
  const int threads = 256;
  const int64_t blocks = (total + threads - 1) / threads;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == B200_DTYPE_BF16)
    decode::lse_merge_kernel<__nv_bfloat16><<<static_cast<unsigned>(blocks), threads, 0, s>>>(
        o_acc, lse_acc, static_cast<const __nv_bfloat16*>(o_b), lse_b, B, Sq, Hq, D, ob_strides[0], ob_strides[1],
        ob_strides[2]);
  else
    decode::lse_merge_kernel<__half><<<static_cast<unsigned>(blocks), threads, 0, s>>>(
        o_acc, lse_acc, static_cast<const __half*>(o_b), lse_b, B, Sq, Hq, D, ob_strides[0], ob_strides[1],
        ob_strides[2]);
  B200_CUDA_OK(cudaGetLastError());
  note_launch("lse_merge_kernel");
  return B200_OK;
}

int b200_cast_out(const float* o_acc, void* o, int B, int Sq, int Hq, int D, const int64_t o_strides[3], int dtype,
                  void* stream) {
  using namespace b200;
  B200_CHECK_ARG(o_acc && o && o_strides, "cast_out: NULL pointer argument");
  B200_CHECK_ARG(B > 0 && Sq > 0 && Hq > 0 && D > 0 && D % 8 == 0, "cast_out: bad sizes");
  B200_CHECK_ARG(o_strides[0] % 8 == 0 && o_strides[1] % 8 == 0 && o_strides[2] % 8 == 0 && ((uintptr_t)o & 15) == 0,
                 "cast_out: strides must be multiples of 8 elements and o 16-byte aligned");
  const int64_t total = static_cast<int64_t>(B) * Sq * Hq * (D / 8);
  const int threads = 256;
  const int64_t blocks = (total + threads - 1) / threads;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == B200_DTYPE_BF16)
    decode::cast_out_kernel<__nv_bfloat16><<<static_cast<unsigned>(blocks), threads, 0, s>>>(
        o_acc, static_cast<__nv_bfloat16*>(o), B, Sq, Hq, D, o_strides[0], o_strides[1], o_strides[2]);
  else if (dtype == B200_DTYPE_FP16)
    decode::cast_out_kernel<__half><<<static_cast<unsigned>(blocks), threads, 0, s>>>(
        o_acc, static_cast<__half*>(o), B, Sq, Hq, D, o_strides[0], o_strides[1], o_strides[2]);
  else
    return set_error(B200_ERR_INVALID_ARGUMENT, "cast_out: dtype must be bf16 or fp16");
  B200_CUDA_OK(cudaGetLastError());
  note_launch("cast_out_kernel");
  return B200_OK;
}

}  // extern "C"
