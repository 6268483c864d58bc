// K1 — tiled online-softmax attention forward (prefill) for sm_100a.
//
// Replaces _flash_attention_forward_kernel / triton_flash_attention
// (kernels/triton/flash_attention_kernels.py:38-325, :1150-1358) and, per ring step,
// triton_ring_attention_forward (kernels/triton/attention_kernels.py:909-998).
//
// One work item = two 128-row query tiles of one (batch, head), walked over the KV sequence in 128-key tiles:
//   warp 0      TMA producer   : Q tiles, then K(j), V(j) through an mbarrier ring (128-byte swizzle)
//   warp 1      MMA issuer     : S_t = Q_t K^T  (tcgen05.mma SS, 128x128xD, fp32 accumulators in TMEM)
//                                O_t += P_t V   (tcgen05.mma TS: P read from TMEM, V MN-major from smem)
//   warp 2      TMEM allocator : 512 columns = [S0 | S1 | O0 | O1]; P_t (16-bit) overlays the upper half of S_t
//   warp 3      work scheduler : cluster launch control — asks the hardware for the block index of a CTA of this
//                                grid that has not started yet; the CTA then processes that block as well
//   warps 4-7   softmax of tile 0, warps 8-11 softmax of tile 1: one thread per query row — tcgen05.ld the
//               row of S, running max / sum in fp32 registers (no shuffles), exp2 with the scale folded in,
//               P written back to TMEM with tcgen05.st, lazy O rescale (only when the row max grew by > 2^8),
//               final O / l -> 16-bit -> global (one 2*D-byte row per thread), LSE -> global.
// The two query tiles ping-pong: while the softmax warps of tile 0 work on S_0(j+1), the tensor core runs
// P_1(j) V(j) and Q_1 K(j+1)^T. Causal tiles above the diagonal are never loaded or computed. CTAs are persistent
// over the launch grid: barrier phases, the KV ring and TMEM carry over from item to item, so the loads and the first
// Q K^T of the next item overlap the tail of the current one.

#include "common.cuh"
#include "host_common.h"

namespace b200 {
namespace fa {

#ifdef B200_FA_TRACE
// developer instrumentation (never compiled into the product library): per-iteration clock64 stamps of one CTA
__device__ long long* g_trace = nullptr;
#define FA_TRACE_ON (g_trace != nullptr && blockIdx.x == gridDim.x / 2 && blockIdx.y == 0 && blockIdx.z == 0)
#define FA_STAMP(slot, j, k) do { if (FA_TRACE_ON && (j) < 64) g_trace[((slot) * 64 + (j)) * 8 + (k)] = clock64(); } while (0)
#else
#define FA_STAMP(slot, j, k) do {} while (0)
#endif

constexpr int BLOCK_M = 128;
constexpr int BLOCK_N = 128;
constexpr int NUM_THREADS = 384;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr bool kPairDefault = false;  // B200_FA_PAIR=1 selects the CTA-pair kernel (generation 3)
constexpr float kRescaleThreshold = 8.0f;  // log2 units: P stays <= 2^8, safe for bf16/fp16 P and fp32 sums

template <int D>
struct Cfg {
  static constexpr int TILE_BYTES = 128 * D * 2;            // one Q / K / V tile
  static constexpr int BOXES = D / 64;                      // 64-column (128-byte) TMA boxes per tile
  static constexpr int KV_STAGES = (D == 128) ? 4 : 6;
  static constexpr int SMEM_Q_OFF = 0;
  static constexpr int SMEM_KV_OFF = 2 * TILE_BYTES;
  static constexpr int SMEM_BAR_OFF = SMEM_KV_OFF + KV_STAGES * TILE_BYTES;
  static constexpr int SMEM_BYTES = SMEM_BAR_OFF + 512 + 1024;
  // TMEM (512 columns): [S0 | S1 | O0 | O1]; P_t (16 bit) overlays the upper half of S_t, so Q_t K(j+1)^T is ordered
  // behind P_t(j) V(j) on the tensor pipe. (Separate P buffers for D = 64 were measured slower: both tiles then run
  // in lockstep and share the MUFU pipe, 606 vs 701 TFLOP/s.)
  static constexpr uint32_t TMEM_S = 0;    // + t * 128
  static constexpr uint32_t TMEM_P = 64;   // + t * 128
  static constexpr uint32_t TMEM_O = 256;  // + t * D
};

struct Params {
  void* o;                  // output, addressed by element strides (batch, seq, head); head dim contiguous
  int64_t o_sb, o_ss, o_sh;
  float* lse;               // [B, Hq, Sq] or nullptr
  const int32_t* kv_lens;   // [B] or nullptr
  int B, Sq, Sk, Hq, Hkv;
  int d_real;               // head_dim of the tensors (a multiple of 8, <= the kernel's D): the TMA loads zero-fill the columns
                            // [d_real, D) of Q / K / V (exact: they add 0 to every score and produce 0 outputs) and the
                            // epilogue does not store them
  float scale_log2;         // softmax_scale * log2(e)
  int causal;
  int64_t causal_offset;    // key j visible to query i iff j <= i + causal_offset
  int num_pairs;            // ceil(Sq / 256)
  int persistent;           // 1: a CTA that finished its block steals further blocks (cluster launch control)
  // accumulate mode (ring steps): the result is merged into a running fp32 output + LSE instead of being written as 16 bit
  float* o_acc;             // fp32, element strides (batch, seq, head) in acc_s*, head dim contiguous
  int64_t acc_sb, acc_ss, acc_sh;
  float* lse_acc;           // fp32, rows contiguous, element strides (batch, head)
  int64_t lse_sb, lse_sh;
  int acc_init;             // 1: overwrite the accumulator (first ring step), 0: log-sum-exp merge into it
  // paged K/V (chunked prefill against the cache, q_len > 1): the KV tile of 128 keys is assembled from 128 / block_size
  // physical blocks named by the block table (one TMA box per block); kv_lens holds the context lengths
  const int32_t* block_table;  // [B, max_blocks] or nullptr (K/V addressed by strides)
  int max_blocks, block_size;
  int causal_bottom;        // 1: the causal diagonal ends at each sequence's LAST key (offset = kv_len - Sq per sequence)
};

// number of KV tiles a query tile [row0, row0+128) needs
__device__ __forceinline__ int num_kv_tiles(const Params& p, int row0, int kv_len, int64_t coff) {
  if (row0 >= p.Sq) return 0;
  int64_t visible = kv_len;
  if (p.causal) {
    const int last_row = min(row0 + BLOCK_M - 1, p.Sq - 1);
    const int64_t lim = static_cast<int64_t>(last_row) + coff + 1;
    if (lim < visible) visible = lim;
  }
  if (visible <= 0) return 0;
  return static_cast<int>((visible + BLOCK_N - 1) / BLOCK_N);
}

// Zero rows [first, BLOCK_N) of a K/V tile in shared memory: the V rows at or past kv_len of the one tile per item that
// straddles it. Those keys are masked (P = 0, or 2^-125 on the exp2_poly2 path), but 0 * NaN / Inf in P V is still NaN,
// so padding that holds non-finite values (stale paged blocks, an uninitialised cache) would poison whole output rows.
// Whole 128-byte rows can be zeroed as they are: the 128-byte swizzle permutes 16-byte chunks inside a row, never across
// rows. Called by a whole warp; the proxy fence orders the stores before the tensor core reads the tile. Out of line: it
// runs at most once per item, and inlined into the MMA issuer it added spills to the kernel.
template <int BOXES>
__device__ __noinline__ void zero_tile_rows(uint8_t* tile, int first, int lane) {
  const int chunks = (BLOCK_N - first) * 8;  // 16-byte chunks per 64-column box
#pragma unroll
  for (int c = 0; c < BOXES; ++c) {
    uint4* rows = reinterpret_cast<uint4*>(tile + c * 16384 + first * 128);
    for (int i = lane; i < chunks; i += 32) rows[i] = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async_smem();
  __syncwarp();
}

// One work item = one block index of the launch grid: a pair of 128-row query tiles of one (batch, head).
struct Work {
  int head, batch, kv_head, q_row0, kv_len, n0, n1, n_max;
  int coff;  // causal offset of this item: key j visible to query i iff j <= i + coff
  __device__ __forceinline__ void set(const Params& p, int bx, int by, int bz) {
    // heavy (late) query tiles first under a causal mask
    const int pair = p.causal ? (p.num_pairs - 1 - bx) : bx;
    head = by;
    batch = bz;
    kv_head = head / (p.Hq / p.Hkv);
    q_row0 = pair * 2 * BLOCK_M;
    kv_len = p.Sk;
    if (p.kv_lens != nullptr) kv_len = max(0, min(p.Sk, p.kv_lens[batch]));
    coff = p.causal_bottom ? kv_len - p.Sq : static_cast<int>(p.causal_offset);
    n0 = num_kv_tiles(p, q_row0, kv_len, coff);
    n1 = num_kv_tiles(p, q_row0 + BLOCK_M, kv_len, coff);
    n_max = max(n0, n1);
  }
  // Every lane holds the same values, but the compiler cannot know that for fields derived from a launch-control
  // response or a global load; broadcasting from lane 0 lets it keep loop counters, ring stages and MMA descriptors
  // in uniform registers (otherwise each tcgen05.mma is preceded by vector-to-uniform moves).
  __device__ __forceinline__ void make_warp_uniform() {
    head = __shfl_sync(0xffffffffu, head, 0);
    batch = __shfl_sync(0xffffffffu, batch, 0);
    kv_head = __shfl_sync(0xffffffffu, kv_head, 0);
    q_row0 = __shfl_sync(0xffffffffu, q_row0, 0);
    kv_len = __shfl_sync(0xffffffffu, kv_len, 0);
    coff = __shfl_sync(0xffffffffu, coff, 0);
    n0 = __shfl_sync(0xffffffffu, n0, 0);
    n1 = __shfl_sync(0xffffffffu, n1, 0);
    n_max = max(n0, n1);
  }
};

// The kernel is persistent over the launch grid: every CTA starts on its own block index and, when a role has finished
// an item, it reads the next block index the scheduler warp obtained through cluster launch control — the hardware
// hands out the pending blocks in launch order (heavy-first, heads sharing K/V adjacent), there is no global counter.
// Barrier phases, the KV ring and TMEM carry over from item to item, so the loads (Q, K, V) and the first Q K^T of
// item i+1 overlap the last P V, the normalisation and the stores of item i.
template <int D, typename T, bool ACCUM>
__global__ void __launch_bounds__(NUM_THREADS, 1)
fa_fwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
              const __grid_constant__ CUtensorMap tmap_v, const Params p) {
  using C = Cfg<D>;
  constexpr int NS = C::KV_STAGES;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  uint64_t* q_full = reinterpret_cast<uint64_t*>(smem + C::SMEM_BAR_OFF);  // [2]  TMA -> MMA
  uint64_t* q_free = q_full + 2;                                           // [2]  softmax -> TMA: last Q_t K^T of the item retired
  uint64_t* kv_full = q_free + 2;                                          // [NS]
  uint64_t* kv_empty = kv_full + NS;                                       // [NS]
  uint64_t* s_full = kv_empty + NS;                                        // [2]  MMA -> softmax
  uint64_t* p_half = s_full + 2;                                           // [2][2] softmax -> MMA: P columns [0,64) / [64,128) stored (one arrival per warp)
  uint64_t* pv_done = p_half + 4;                                          // [2]  MMA -> softmax (O_t updated)
  uint64_t* clc_full = pv_done + 2;                                        // [1]  launch-control response landed
  uint64_t* clc_empty = clc_full + 1;                                      // [1]  all 10 reader warps have decoded it
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(clc_empty + 1);
  uint8_t* clc_resp = reinterpret_cast<uint8_t*>(tmem_ptr_smem + 4);       // 16 bytes, 16-byte aligned
  constexpr int kClcReaders = 10;  // producer lane + MMA warp + 8 softmax warps

  const int warp_idx = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);  // warp-uniform
  const int lane = threadIdx.x & 31;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
  }
  if (warp_idx == 1 && lane == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_free[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_half[2 * i], 4);
      mbar_init(&p_half[2 * i + 1], 4);
      mbar_init(&pv_done[i], 1);
    }
    for (int i = 0; i < NS; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    mbar_init(clc_full, 1);
    mbar_init(clc_empty, kClcReaders);
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    tmem_alloc(tmem_ptr_smem, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // Item k >= 1 of this CTA is launch-control response k-1. `whole_warp`: all 32 lanes of the calling warp read it.
  auto next_work = [&](Work& w, int k, bool whole_warp) -> bool {
    if (!p.persistent) return false;
    mbar_wait_long(clc_full, static_cast<uint32_t>((k - 1) & 1));
    int bx, by, bz;
    bool ok = clc_query(clc_resp, bx, by, bz);
    fence_proxy_async_smem();  // our generic-proxy read is ordered before the next async-proxy write of the response
    if (whole_warp) {
      __syncwarp();
      ok = __shfl_sync(0xffffffffu, static_cast<int>(ok), 0) != 0;
    }
    if (lane == 0) mbar_arrive(clc_empty);
    if (ok) {
      w.set(p, bx, by, bz);
      if (whole_warp) w.make_warp_uniform();
    }
    return ok;
  };

  Work w;
  w.set(p, blockIdx.x, blockIdx.y, blockIdx.z);
  if (warp_idx != 0) w.make_warp_uniform();  // (the producer runs on one lane)

  // register budget: 384 threads x 168 at launch; the producer warpgroup gives 96 per thread to the softmax
  // warpgroups (128 x 72 + 256 x 216 = 64512)
  if (warp_idx < 4) {
    setmaxnreg_dec<72>();
  }
  if (warp_idx == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int q_loads[2] = {0, 0};
      for (int k = 0;; ++k) {
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          if ((t == 0 ? w.n0 : w.n1) > 0) {
            // the previous item's last Q_t K^T must have retired before its Q tile is overwritten
            if (q_loads[t] > 0) mbar_wait(&q_free[t], static_cast<uint32_t>((q_loads[t] - 1) & 1));
            ++q_loads[t];
            mbar_arrive_expect_tx(&q_full[t], C::TILE_BYTES);
            uint8_t* sq = smem + C::SMEM_Q_OFF + t * C::TILE_BYTES;
#pragma unroll
            for (int c = 0; c < C::BOXES; ++c)
              tma_load_4d(sq + c * 16384, &tmap_q, &q_full[t], c * 64, w.head, w.q_row0 + t * BLOCK_M, w.batch);
          }
        }
        for (int j = 0; j < w.n_max; ++j) {
#pragma unroll
          for (int kv = 0; kv < 2; ++kv) {  // 0: K(j), 1: V(j)
            mbar_wait(&kv_empty[stage], phase ^ 1);
            mbar_arrive_expect_tx(&kv_full[stage], C::TILE_BYTES);
            uint8_t* dst = smem + C::SMEM_KV_OFF + stage * C::TILE_BYTES;
            const CUtensorMap* tm = kv == 0 ? &tmap_k : &tmap_v;
            if (p.block_table != nullptr) {
              // paged cache, tensor map dims (D, Hkv, block_size, num_blocks): one box of block_size keys per physical
              // block, placed at its row offset inside the swizzled tile (block_size % 8 == 0 keeps the 1024-byte swizzle
              // atoms aligned). Blocks past the sequence's last one re-load the last block: finite data, masked by kv_len.
              const int bs = p.block_size, nblk = (w.kv_len + bs - 1) / bs;
              const int32_t* bt = p.block_table + static_cast<int64_t>(w.batch) * p.max_blocks;
              for (int b = 0, lb = j * (BLOCK_N / bs); b < BLOCK_N / bs; ++b, ++lb) {
                const int phys = __ldg(bt + min(lb, nblk - 1));
#pragma unroll
                for (int c = 0; c < C::BOXES; ++c)
                  tma_load_4d(dst + c * 16384 + b * bs * 128, tm, &kv_full[stage], c * 64, w.kv_head, 0, phys);
              }
            } else {
#pragma unroll
              for (int c = 0; c < C::BOXES; ++c)
                tma_load_4d(dst + c * 16384, tm, &kv_full[stage], c * 64, w.kv_head, j * BLOCK_N, w.batch);
            }
            if (++stage == NS) { stage = 0; phase ^= 1; }
          }
        }
        if (!next_work(w, k + 1, false)) break;
      }
    }
  } else if (warp_idx == 1) {
    // ============================== MMA issuer ==============================
    // The whole warp runs the (warp-uniform) control flow so descriptors live in uniform registers; one elected
    // lane issues the tcgen05 instructions.
    constexpr uint32_t idesc_qk = make_idesc_f16(BLOCK_M, BLOCK_N, Pack2<T>::kIsBf16, false, false);
    constexpr uint32_t idesc_pv = make_idesc_f16(BLOCK_M, D, Pack2<T>::kIsBf16, false, true);
    const uint32_t sq_addr = smem_u32(smem + C::SMEM_Q_OFF);
    const uint32_t skv_addr = smem_u32(smem + C::SMEM_KV_OFF);
    // descriptor templates; the start-address field (bits 0-13, 16-byte units) is advanced by plain adds
    const uint64_t qdesc0 = make_smem_desc_sw128(sq_addr, 16, 1024);
    const uint64_t kdesc0 = make_smem_desc_sw128(skv_addr, 16, 1024);
    const uint64_t vdesc0 = make_smem_desc_sw128(skv_addr, 16384, 1024);
    constexpr uint32_t TILE16 = C::TILE_BYTES >> 4;

    // S_t = Q_t K^T
    auto issue_qk = [&](int t, int k_stage) {
      const uint64_t qd = qdesc0 + static_cast<uint64_t>(t * TILE16);
      const uint64_t kd = kdesc0 + static_cast<uint64_t>(k_stage * TILE16);
      const uint32_t d_tmem = tmem_base + C::TMEM_S + static_cast<uint32_t>(t * 128);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < D / 16; ++ks) {
          const uint32_t off = (ks >> 2) * 1024 + (ks & 3) * 2;  // 16-byte units: next 64-col box / next 32 bytes
          umma_ss(d_tmem, qd + off, kd + off, idesc_qk, ks > 0 ? 1u : 0u);
        }
        umma_commit(&s_full[t]);
      }
      __syncwarp();
    };
    // P V for keys [64*part, 64*part+64) of the tile: issued as soon as that half of P is in TMEM, so the tensor
    // pipe works on the first half while the softmax warps still exponentiate the second
    auto issue_pv = [&](int t, int v_stage, int part, bool accumulate) {
      const uint64_t vd = vdesc0 + static_cast<uint64_t>(v_stage * TILE16);
      const uint32_t d_tmem = tmem_base + C::TMEM_O + static_cast<uint32_t>(t * D);
      const uint32_t p_tmem = tmem_base + C::TMEM_P + static_cast<uint32_t>(t * 128);
      if (elect_one()) {
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          const int ks = part * 4 + k4;
          umma_ts(d_tmem, p_tmem + ks * 8, vd + static_cast<uint64_t>(ks * 128), idesc_pv,
                  (accumulate || ks > 0) ? 1u : 0u);
        }
        if (part == 1) umma_commit(&pv_done[t]);
      }
      __syncwarp();
    };
    auto release = [&](int stage) {
      if (elect_one()) umma_commit(&kv_empty[stage]);
      __syncwarp();
    };

    // ring bookkeeping: the KV ring carries K(0),V(0),K(1),V(1),... of item after item; (stage, phase) advance by one
    // per tile. k_stage = stage of the next K tile to consume.
    int k_stage = 0;
    uint32_t k_phase = 0;
    uint32_t it_par[2] = {0, 0};  // parity of the KV iterations completed per query tile over all items
    uint32_t q_par[2] = {0, 0};   // parity of the Q tiles consumed per query tile
    for (int k = 0;; ++k) {
      if (w.n_max > 0) {
        const int nt[2] = {w.n0, w.n1};
#pragma unroll
        for (int t = 0; t < 2; ++t)
          if (nt[t] > 0) { mbar_wait(&q_full[t], q_par[t]); q_par[t] ^= 1; }
        mbar_wait(&kv_full[k_stage], k_phase);
        tc_fence_after();
#pragma unroll
        for (int t = 0; t < 2; ++t)
          if (nt[t] > 0) issue_qk(t, k_stage);
        release(k_stage);  // K(0) is free once both S MMAs retire

        for (int j = 0; j < w.n_max; ++j) {
          int v_stage = k_stage + 1;
          uint32_t v_phase = k_phase;
          if (v_stage == NS) { v_stage = 0; v_phase ^= 1; }
          k_stage = v_stage + 1;
          k_phase = v_phase;
          if (k_stage == NS) { k_stage = 0; k_phase ^= 1; }
          const bool has_next = (j + 1 < w.n_max);
          mbar_wait(&kv_full[v_stage], v_phase);
          if (w.kv_len - j * BLOCK_N < BLOCK_N)  // V(j) straddles kv_len: its rows past the end must read as zeros
            zero_tile_rows<C::BOXES>(smem + C::SMEM_KV_OFF + v_stage * C::TILE_BYTES, w.kv_len - j * BLOCK_N, lane);
          bool next_k_ready = false;
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            if (j < nt[t]) {
              const uint32_t par = (it_par[t] + static_cast<uint32_t>(j)) & 1;
              if (lane == 0) FA_STAMP(2 + t, j, 0);
              mbar_wait(&p_half[2 * t], par);
              tc_fence_after();
              if (lane == 0) FA_STAMP(2 + t, j, 1);
              issue_pv(t, v_stage, 0, j > 0);
              mbar_wait(&p_half[2 * t + 1], par);
              tc_fence_after();
              issue_pv(t, v_stage, 1, true);
              if (lane == 0) FA_STAMP(2 + t, j, 2);
            }
            if (j + 1 < nt[t]) {
              if (!next_k_ready) {
                mbar_wait(&kv_full[k_stage], k_phase);
                tc_fence_after();
                next_k_ready = true;
              }
              issue_qk(t, k_stage);
              if (lane == 0) FA_STAMP(2 + t, j, 3);
            }
          }
          release(v_stage);
          if (has_next) {
            if (!next_k_ready) mbar_wait(&kv_full[k_stage], k_phase);
            release(k_stage);
          }
        }
        it_par[0] = (it_par[0] + static_cast<uint32_t>(w.n0)) & 1;
        it_par[1] = (it_par[1] + static_cast<uint32_t>(w.n1)) & 1;
      }
      if (!next_work(w, k + 1, true)) break;
    }
  } else if (warp_idx == 3) {
    // ============================== work scheduler ==============================
    // Request k asks for the block that becomes item k+1 of this CTA; it is issued once every reader has decoded
    // response k-1 (= has started item k), so one item is prefetched and none is hoarded.
    if (p.persistent && lane == 0) {
      for (int k = 0;; ++k) {
        if (k > 0) mbar_wait_long(clc_empty, static_cast<uint32_t>((k - 1) & 1));
        mbar_arrive_expect_tx(clc_full, 16);
        clc_try_cancel(clc_resp, clc_full);
        mbar_wait_long(clc_full, static_cast<uint32_t>(k & 1));
        int bx, by, bz;
        if (!clc_query(clc_resp, bx, by, bz)) break;  // grid exhausted: a failed request must not be repeated
      }
    }
  } else if (warp_idx >= 4) {
    // ============================== softmax / correction / epilogue ==============================
    setmaxnreg_inc<216>();
    const int t = (warp_idx - 4) >> 2;           // query tile of this warpgroup
    const int quad = warp_idx & 3;               // TMEM lane quadrant
    const int row = quad * 32 + lane;            // row inside the tile
    const int wg_tid = threadIdx.x - 128 - t * 128;
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t tS = tmem_base + lane_addr + C::TMEM_S + static_cast<uint32_t>(t * 128);
    const uint32_t tP = tmem_base + lane_addr + C::TMEM_P + static_cast<uint32_t>(t * 128);
    const uint32_t tO = tmem_base + lane_addr + C::TMEM_O + static_cast<uint32_t>(t * D);
    uint32_t iters = 0;  // KV iterations of this query tile over all items (barrier parities)
    // barrier addresses of this warpgroup as one opaque base register + constant offsets (see smem_addr_opaque)
    const uint32_t bar_base = smem_addr_opaque(q_full) + static_cast<uint32_t>(t) * 8u;
    auto bar_off = [&](const uint64_t* b0) { return static_cast<uint32_t>((b0 - q_full) * 8); };
    const uint32_t a_s_full = bar_base + bar_off(s_full);
    const uint32_t a_pv_done = bar_base + bar_off(pv_done);
    const uint32_t a_q_free = bar_base + bar_off(q_free);
    const uint32_t a_p_half = bar_base + static_cast<uint32_t>(t) * 8u + bar_off(p_half);  // [2 * t + half]

    for (int k = 0;; ++k) {
      const int tile_row0 = w.q_row0 + t * BLOCK_M;
      const int q_row = tile_row0 + row;
      const int nt = t == 0 ? w.n0 : w.n1;
      const int kv_len = w.kv_len;
      float m_used = -INFINITY;  // reference max (log2 units) the stored P / O / l are relative to
      float l_run = 0.f;
      const int64_t q_pos_plus = static_cast<int64_t>(q_row) + w.coff;  // last visible key under causal

      for (int j = 0; j < nt; ++j) {
        const uint32_t par = (iters + static_cast<uint32_t>(j)) & 1;
        mbar_wait_addr(a_s_full, par);
        tc_fence_after();
        // the commit behind s_full covers every earlier MMA: once the item's last S tile is visible, Q_t is free
        if (j + 1 == nt && wg_tid == 0) mbar_arrive_addr(a_q_free);
        if (wg_tid == 0) FA_STAMP(t, j, 0);
        uint32_t s[128];
        tmem_ld_x32(tS + 0, s + 0);
        tmem_ld_x32(tS + 32, s + 32);
        tmem_ld_x32(tS + 64, s + 64);
        tmem_ld_x32(tS + 96, s + 96);
        tmem_wait_ld();
        if (wg_tid == 0) FA_STAMP(t, j, 1);
        // ---- masking: keys >= limit (relative to the tile) are invisible ----
        const int kv0 = j * BLOCK_N;
        int limit = kv_len - kv0;
        if (p.causal) {
          const int64_t cl = q_pos_plus - kv0 + 1;
          if (cl < limit) limit = static_cast<int>(cl < 0 ? 0 : cl);
        }
        if (limit < BLOCK_N) {
#pragma unroll
          for (int c = 0; c < 128; ++c)
            if (c >= limit) s[c] = 0xFF800000u;  // -inf
        }
        const float2 sc2 = make_float2(p.scale_log2, p.scale_log2);
        float2 nm2, sum2;
        uint32_t pk0[32], pk1[32];
        // columns c, c+1: packed fp32x2 FMA / ADD halve the issue slots of the scale-subtract and the row sum
#ifndef B200_FA_POLY_MOD
#define B200_FA_POLY_MOD 4
#endif
        // One pair in B200_FA_POLY_MOD takes the exponential on the FMA pipe (exp2_poly2) instead of the MUFU pipe,
        // which is the busier of the two in this loop (0 = MUFU only).
        auto exp_pair = [&](int c) -> uint32_t {
          const float2 x = __ffma2_rn(make_float2(__uint_as_float(s[c]), __uint_as_float(s[c + 1])), sc2, nm2);
          const bool poly = B200_FA_POLY_MOD > 0 && ((c >> 1) % (B200_FA_POLY_MOD > 0 ? B200_FA_POLY_MOD : 1)) == 1;
          const float2 e = poly ? exp2_poly2(x) : make_float2(fast_exp2(x.x), fast_exp2(x.y));
          sum2 = __fadd2_rn(sum2, e);
          return Pack2<T>::pack(e.x, e.y);
        };
        auto set_reference = [&]() {
          const float m_ref = (m_used == -INFINITY) ? 0.f : m_used;
          nm2 = make_float2(-m_ref, -m_ref);
          sum2 = make_float2(0.f, 0.f);
        };
        auto publish = [&](int half) {
          tmem_wait_st();
          __syncwarp();
          if (lane == 0) mbar_arrive_addr(a_p_half + static_cast<uint32_t>(half) * 8u);
        };
        // ---- speculative first half: P = exp2(s * scale - m_used) against the reference max of the PREVIOUS tiles ----
        // With lazy rescaling the reference only changes when the row max grows by more than 2^8, which is rare after
        // the first tiles, so the exponentials (MUFU pipe) need not wait for this tile's row max (ALU pipe): both run
        // concurrently and the max leaves the critical path. If the reference does change (always for the first tile of
        // an item) the first half is recomputed. (Skipping the speculation for j == 0 instead was measured: the second
        // conditional copy of the exponentials makes ptxas spill in this loop, +40 % cycles.)
        set_reference();
#pragma unroll
        for (int i = 0; i < 32; ++i) pk0[i] = exp_pair(2 * i);
        if (wg_tid == 0) FA_STAMP(t, j, 3);
        // ---- row max ----
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int c = 0; c < 128; c += 4) {
          mx0 = fmaxf(mx0, __uint_as_float(s[c + 0]));
          mx1 = fmaxf(mx1, __uint_as_float(s[c + 1]));
          mx2 = fmaxf(mx2, __uint_as_float(s[c + 2]));
          mx3 = fmaxf(mx3, __uint_as_float(s[c + 3]));
        }
        const float m_tile = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * p.scale_log2;
        if (wg_tid == 0) FA_STAMP(t, j, 2);
        // ---- lazy rescale decision ----
        float alpha = 1.0f;
        bool rescale = false;
        if (m_tile > m_used + kRescaleThreshold) {  // (m_used = -inf until the first visible key)
          alpha = fast_exp2(m_used - m_tile);       // m_used = -inf -> 0
          m_used = m_tile;
          l_run *= alpha;
          rescale = true;
        }
        if (__any_sync(0xffffffffu, rescale)) {
          if (j > 0) {
            // O_t must contain P(j-1) V(j-1) before it is rescaled
            mbar_wait_addr(a_pv_done, par ^ 1);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < D / 32; ++c) {
              uint32_t o[32];
              tmem_ld_x32(tO + c * 32, o);
              tmem_wait_ld();
#pragma unroll
              for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
              tmem_st_x32(tO + c * 32, o);
            }
          }
          // the speculation failed for at least one row of this warp: redo the first half against the new reference
          set_reference();
#pragma unroll
          for (int i = 0; i < 32; ++i) pk0[i] = exp_pair(2 * i);
        }
        // ---- store P (16 bit) to TMEM in two halves of 64 keys; second half of the exponentials ----
        tmem_st_x32(tP, pk0);
#pragma unroll
        for (int i = 0; i < 16; ++i) pk1[i] = exp_pair(64 + 2 * i);
        publish(0);  // the first half of P has landed by now: its P V MMAs start while we finish the row
        if (wg_tid == 0) FA_STAMP(t, j, 4);
#pragma unroll
        for (int i = 16; i < 32; ++i) pk1[i] = exp_pair(64 + 2 * i);
        tmem_st_x32(tP + 32, pk1);
        l_run += sum2.x + sum2.y;
        if (wg_tid == 0) FA_STAMP(t, j, 6);
        publish(1);
        if (wg_tid == 0) FA_STAMP(t, j, 7);
      }

      // ---- epilogue: O / l -> 16 bit -> global (each thread owns one 2*D-byte output row); LSE -> global ----
      // No shared-memory staging: the Q buffers stay free for the next item's loads, and O_t is back in registers
      // before this warp publishes the next item's first P (which is what lets the MMA warp overwrite O_t).
      if (tile_row0 < p.Sq) {
        float inv_l = 0.f;
        float lse_val = -INFINITY;
        if (nt > 0) {
          mbar_wait_addr(a_pv_done, (iters + static_cast<uint32_t>(nt - 1)) & 1);
          tc_fence_after();
          if (l_run > 0.f && m_used != -INFINITY) {  // (a row without a visible key keeps m_used = -inf)
            inv_l = 1.0f / l_run;
            lse_val = (m_used + log2f(l_run)) * kLn2;
          }
        }
        const bool row_ok = q_row < p.Sq;
        if constexpr (!ACCUM) {
          if (p.lse != nullptr && row_ok) p.lse[(static_cast<int64_t>(w.batch) * p.Hq + w.head) * p.Sq + q_row] = lse_val;
          T* orow = reinterpret_cast<T*>(p.o) + static_cast<int64_t>(w.batch) * p.o_sb + static_cast<int64_t>(q_row) * p.o_ss +
                    static_cast<int64_t>(w.head) * p.o_sh;
#pragma unroll
          for (int c = 0; c < D / 32; ++c) {
            uint32_t o[32];
            if (nt > 0) {
              tmem_ld_x32(tO + c * 32, o);
              tmem_wait_ld();
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) o[i] = 0u;
            }
            if (row_ok) {
#pragma unroll
              for (int q4 = 0; q4 < 4; ++q4) {
                uint4 pk;
                pk.x = Pack2<T>::pack(__uint_as_float(o[q4 * 8 + 0]) * inv_l, __uint_as_float(o[q4 * 8 + 1]) * inv_l);
                pk.y = Pack2<T>::pack(__uint_as_float(o[q4 * 8 + 2]) * inv_l, __uint_as_float(o[q4 * 8 + 3]) * inv_l);
                pk.z = Pack2<T>::pack(__uint_as_float(o[q4 * 8 + 4]) * inv_l, __uint_as_float(o[q4 * 8 + 5]) * inv_l);
                pk.w = Pack2<T>::pack(__uint_as_float(o[q4 * 8 + 6]) * inv_l, __uint_as_float(o[q4 * 8 + 7]) * inv_l);
                if (c * 32 + q4 * 8 < p.d_real) *reinterpret_cast<uint4*>(orow + c * 32 + q4 * 8) = pk;
              }
            }
          }
        } else {
          // ---- accumulate mode: (O / l, LSE) of this key block is merged into the running fp32 (O, LSE) in place:
          //   lse = logaddexp(lse_acc, lse_new);  o_acc = o_acc * exp(lse_acc - lse) + (O / l) * exp(lse_new - lse)
          // (kernels/triton/attention_kernels.py:1567-1585). A side with LSE = -inf contributes nothing. ----
          float* lrow = p.lse_acc + static_cast<int64_t>(w.batch) * p.lse_sb + static_cast<int64_t>(w.head) * p.lse_sh + q_row;
          float* arow = p.o_acc + static_cast<int64_t>(w.batch) * p.acc_sb + static_cast<int64_t>(q_row) * p.acc_ss +
                        static_cast<int64_t>(w.head) * p.acc_sh;
          float w_old = 0.f, w_new = inv_l, lse_out = lse_val;
          if (!p.acc_init && row_ok) {
            const float lse_old = *lrow;
            const float mx = fmaxf(lse_old, lse_val);
            if (mx == -INFINITY) {
              w_old = 0.f;
              w_new = 0.f;
              lse_out = -INFINITY;
            } else {
              const float e_old = fast_exp2((lse_old - mx) * kLog2e);
              const float e_new = fast_exp2((lse_val - mx) * kLog2e);
              const float den = e_old + e_new;
              lse_out = mx + log2f(den) * kLn2;
              w_old = e_old / den;
              w_new = e_new / den * inv_l;
            }
          }
          // a merge with a block that has no visible key for this row leaves the accumulator untouched
          const bool touch = row_ok && (p.acc_init || lse_val != -INFINITY);
          if (touch) *lrow = lse_out;
#pragma unroll
          for (int c = 0; c < D / 32; ++c) {
            uint32_t o[32];
            if (nt > 0) {
              tmem_ld_x32(tO + c * 32, o);
              tmem_wait_ld();
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) o[i] = 0u;
            }
            if (touch) {
#pragma unroll
              for (int q4 = 0; q4 < 8; ++q4) {
                if (c * 32 + q4 * 4 >= p.d_real) continue;
                float4* dst = reinterpret_cast<float4*>(arow + c * 32 + q4 * 4);
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
                if (!p.acc_init) a = *dst;
                a.x = a.x * w_old + __uint_as_float(o[q4 * 4 + 0]) * w_new;
                a.y = a.y * w_old + __uint_as_float(o[q4 * 4 + 1]) * w_new;
                a.z = a.z * w_old + __uint_as_float(o[q4 * 4 + 2]) * w_new;
                a.w = a.w * w_old + __uint_as_float(o[q4 * 4 + 3]) * w_new;
                *dst = a;
              }
            }
          }
        }
      }
      iters += static_cast<uint32_t>(nt);
      if (!next_work(w, k + 1, true)) break;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int D, typename T, bool ACCUM>
int launch(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const Params& p, cudaStream_t stream) {
  auto kern = fa_fwd_kernel<D, T, ACCUM>;
  static bool attr_set[64] = {};  // per device
  B200_CUDA_OK(set_max_dynamic_smem(reinterpret_cast<const void*>(kern), Cfg<D>::SMEM_BYTES, attr_set));
  dim3 grid(p.num_pairs, p.Hq, p.B);
  kern<<<grid, NUM_THREADS, Cfg<D>::SMEM_BYTES, stream>>>(tq, tk, tv, p);
  B200_CUDA_OK(cudaGetLastError());
  note_launch("fa_fwd_kernel");
  return B200_OK;
}

// =====================================================================================================================
// K1 generation 3 — CTA PAIR kernel (cluster of 2): each CTA owns ONE 128-row query tile of a 256-row pair.
//
// Why (DESIGN.md §3 K1, round-2 measurements): with two query tiles per CTA the 512 TMEM columns are exactly
// [S0 | S1 | O0 | O1]; P_t has to overlay S_t, which orders Q_t K(j+1)^T behind P_t(j) V(j) and makes each tile's
// S -> softmax -> P V -> next S chain (2 mbarrier hops + ~1700 cycles of softmax + 768 cycles of MMA) the period: 2850-2960
// cycles per KV iteration against 2048 of tensor work. With ONE tile per CTA the columns are [S_a | S_b | P_a | P_b | O]:
// scores and probabilities are double buffered, the MMA warp issues Q K(j+2)^T while P(j) is still being computed, and two
// softmax warpgroups take alternate KV blocks (even / odd), so neither the tensor pipe nor the softmax warps wait for
// each other in steady state. One tile per CTA would double the K/V fill per FLOP (L2 -> SM traffic above what the L2
// delivers), so the two CTAs of a cluster load HALF of every K/V tile each and TMA-multicast it into both CTAs' shared
// memory: the K/V traffic per 256 query rows is what it was.
//
//   warp 0      TMA producer   : own Q tile; keys [64c, 64c+64) of every K / V tile (c = CTA rank), multicast to both CTAs
//   warp 1      MMA issuer     : step s: S_[s&1] = Q K(s)^T, then O += P_[s&1](s-2) V(s-2)   (tcgen05 cta_group::1)
//   warp 2      TMEM allocator
//   warps 4-7   softmax of the even KV blocks, warps 8-11 of the odd ones (one thread per query row each)
// The two warpgroups share the row state through the reference maximum: block j's group reads the reference block j-1
// left in shared memory (`ref_bar`), rescales its own partial row sum if it moved, decides (lazily, threshold 2^8)
// whether to raise it — rescaling O after P(j-1) V(j-1) retired — and publishes the result for block j+1. The row sum is
// the sum of the two groups' partial sums once both are relative to the final reference.
// K/V ring order (producer and consumer walk the same list): step s holds K(s) then V(s-2).
// =====================================================================================================================
template <int D>
struct Cfg2 {
  static constexpr int TILE_BYTES = 128 * D * 2;            // one Q / K / V tile
  static constexpr int BOXES = D / 64;                      // 64-column (128-byte) TMA boxes per tile
  static constexpr int KV_STAGES = (D == 128) ? 5 : 8;
  static constexpr int SMEM_Q_OFF = 0;
  static constexpr int SMEM_KV_OFF = TILE_BYTES;
  static constexpr int SMEM_BAR_OFF = SMEM_KV_OFF + KV_STAGES * TILE_BYTES;
  static constexpr int SMEM_XCH_OFF = SMEM_BAR_OFF + 512;   // mref[128], lsum[2][128] (fp32)
  static constexpr int SMEM_BYTES = SMEM_XCH_OFF + 3 * 128 * 4 + 1024;
  static constexpr uint32_t TMEM_S = 0;    // + buf * 128
  static constexpr uint32_t TMEM_P = 256;  // + buf * 64
  static constexpr uint32_t TMEM_O = 384;  // D columns
};

template <int D, typename T, bool ACCUM>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
fa_fwd_pair_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                   const __grid_constant__ CUtensorMap tmap_v, const Params p) {
  using C = Cfg2<D>;
  constexpr int NS = C::KV_STAGES;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  uint64_t* q_full = reinterpret_cast<uint64_t*>(smem + C::SMEM_BAR_OFF);  // [1]  TMA -> MMA
  uint64_t* kv_full = q_full + 1;                                          // [NS] TMA (both CTAs' halves) -> MMA
  uint64_t* kv_empty = kv_full + NS;                                       // [NS] MMA warps of BOTH CTAs -> TMA
  uint64_t* s_full = kv_empty + NS;                                        // [2]  MMA -> softmax group buf
  uint64_t* s_free = s_full + 2;                                           // [2]  softmax -> MMA: scores are in registers (4 warps)
  uint64_t* p_half = s_free + 2;                                           // [half][group] softmax -> MMA: half of P stored (4 warps)
  uint64_t* pv_done = p_half + 4;                                          // [2]  MMA -> softmax: P_buf consumed, O updated
  uint64_t* ref_bar = pv_done + 2;                                         // [2]  softmax group -> the other group: reference published (4 warps)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(ref_bar + 2);
  float* mref = reinterpret_cast<float*>(smem + C::SMEM_XCH_OFF);          // [128] reference max after the latest block
  float* lsum = mref + 128;                                                // [2][128] partial row sums at the end

  const int warp_idx = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);  // warp-uniform
  const int lane = threadIdx.x & 31;
  const uint32_t cta = cluster_ctarank();  // which 128-row tile of the pair, and which half of every K/V tile we load

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
  }
  if (warp_idx == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < NS; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 2);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 4);
      mbar_init(&p_half[2 * i], 4);
      mbar_init(&p_half[2 * i + 1], 4);
      mbar_init(&pv_done[i], 1);
      mbar_init(&ref_bar[i], 4);
    }
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    tmem_alloc(tmem_ptr_smem, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer's barriers are initialised before any multicast load or commit can reach them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // ---- work item: cluster = one 256-row pair of one (batch, head); heavy pairs first under a causal mask ----
  const int pair_idx = p.causal ? (p.num_pairs - 1 - static_cast<int>(blockIdx.x >> 1)) : static_cast<int>(blockIdx.x >> 1);
  const int head = blockIdx.y, batch = blockIdx.z;
  const int kv_head = head / (p.Hq / p.Hkv);
  int kv_len = p.Sk;
  if (p.kv_lens != nullptr) kv_len = max(0, min(p.Sk, p.kv_lens[batch]));
  const int coff = p.causal_bottom ? kv_len - p.Sq : static_cast<int>(p.causal_offset);
  const int pair_row0 = pair_idx * 2 * BLOCK_M;
  const int n_t0 = num_kv_tiles(p, pair_row0, kv_len, coff), n_t1 = num_kv_tiles(p, pair_row0 + BLOCK_M, kv_len, coff);
  const int n_mine = __shfl_sync(0xffffffffu, cta == 0 ? n_t0 : n_t1, 0);
  const int n_max = __shfl_sync(0xffffffffu, max(n_t0, n_t1), 0);   // the ring carries the K/V tiles either CTA needs
  const int tile_row0 = pair_row0 + static_cast<int>(cta) * BLOCK_M;

  if (warp_idx < 4) {
    setmaxnreg_dec<72>();
  }
  if (warp_idx == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      if (n_mine > 0) {
        mbar_arrive_expect_tx(q_full, C::TILE_BYTES);
        uint8_t* sq = smem + C::SMEM_Q_OFF;
#pragma unroll
        for (int c = 0; c < C::BOXES; ++c) tma_load_4d(sq + c * 16384, &tmap_q, q_full, c * 64, head, tile_row0, batch);
      }
      int stage = 0;
      uint32_t phase = 0;
      auto load_half = [&](const CUtensorMap* tm, int j) {
        mbar_wait(&kv_empty[stage], phase ^ 1);  // both CTAs have released this stage
        mbar_arrive_expect_tx(&kv_full[stage], C::TILE_BYTES);  // (our half + the peer's half land here)
        uint8_t* dst = smem + C::SMEM_KV_OFF + stage * C::TILE_BYTES + cta * (64 * 128);  // rows [64c, 64c+64) of every box
#pragma unroll
        for (int c = 0; c < C::BOXES; ++c)
          tma_load_4d_mcast(dst + c * 16384, tm, &kv_full[stage], c * 64, kv_head, j * BLOCK_N + static_cast<int>(cta) * 64, batch, 3);
        if (++stage == NS) { stage = 0; phase ^= 1; }
      };
      for (int s = 0; s < n_max + 2; ++s) {
        if (s < n_max) load_half(&tmap_k, s);
        if (s >= 2) load_half(&tmap_v, s - 2);
      }
    }
  } else if (warp_idx == 1) {
    // ============================== MMA issuer ==============================
    constexpr uint32_t idesc_qk = make_idesc_f16(BLOCK_M, BLOCK_N, Pack2<T>::kIsBf16, false, false);
    constexpr uint32_t idesc_pv = make_idesc_f16(BLOCK_M, D, Pack2<T>::kIsBf16, false, true);
    const uint32_t sq_addr = smem_u32(smem + C::SMEM_Q_OFF);
    const uint32_t skv_addr = smem_u32(smem + C::SMEM_KV_OFF);
    const uint64_t qdesc0 = make_smem_desc_sw128(sq_addr, 16, 1024);
    const uint64_t kdesc0 = make_smem_desc_sw128(skv_addr, 16, 1024);
    const uint64_t vdesc0 = make_smem_desc_sw128(skv_addr, 16384, 1024);
    constexpr uint32_t TILE16 = C::TILE_BYTES >> 4;
    auto issue_qk = [&](int buf, int k_stage) {
      const uint64_t kd = kdesc0 + static_cast<uint64_t>(k_stage * TILE16);
      const uint32_t d_tmem = tmem_base + C::TMEM_S + static_cast<uint32_t>(buf * 128);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < D / 16; ++ks) {
          const uint32_t off = (ks >> 2) * 1024 + (ks & 3) * 2;  // 16-byte units: next 64-col box / next 32 bytes
          umma_ss(d_tmem, qdesc0 + off, kd + off, idesc_qk, ks > 0 ? 1u : 0u);
        }
        umma_commit(&s_full[buf]);
      }
      __syncwarp();
    };
    auto issue_pv = [&](int buf, int v_stage, int part, bool accumulate) {
      const uint64_t vd = vdesc0 + static_cast<uint64_t>(v_stage * TILE16);
      const uint32_t d_tmem = tmem_base + C::TMEM_O;
      const uint32_t p_tmem = tmem_base + C::TMEM_P + static_cast<uint32_t>(buf * 64);
      if (elect_one()) {
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          const int ks = part * 4 + k4;
          umma_ts(d_tmem, p_tmem + ks * 8, vd + static_cast<uint64_t>(ks * 128), idesc_pv, (accumulate || ks > 0) ? 1u : 0u);
        }
        if (part == 1) umma_commit(&pv_done[buf]);
      }
      __syncwarp();
    };
    // the stage is free for the NEXT multicast load once the MMA warps of both CTAs have released it
    auto release = [&](int stage) {
      if (elect_one()) umma_commit_mcast(&kv_empty[stage], 3);
      __syncwarp();
    };
    if (n_mine > 0) mbar_wait(q_full, 0);
    int stage = 0;
    uint32_t phase = 0;
    auto advance = [&]() { if (++stage == NS) { stage = 0; phase ^= 1; } };
    for (int s = 0; s < n_max + 2; ++s) {
      if (s < n_max) {  // K(s)
        mbar_wait(&kv_full[stage], phase);
        if (s < n_mine) {
          const int buf = s & 1;
          if (s >= 2) mbar_wait(&s_free[buf], static_cast<uint32_t>(((s - 2) >> 1) & 1));  // S(s-2) is in registers
          tc_fence_after();
          issue_qk(buf, stage);
        }
        release(stage);
        advance();
      }
      if (s >= 2) {     // V(s-2)
        const int j = s - 2;
        mbar_wait(&kv_full[stage], phase);
        if (j < n_mine) {
          // V(j) straddles kv_len: this CTA zeroes its own copy of the multicast tile (the stage is refilled only once both
          // CTAs have released it)
          if (kv_len - j * BLOCK_N < BLOCK_N)
            zero_tile_rows<C::BOXES>(smem + C::SMEM_KV_OFF + stage * C::TILE_BYTES, kv_len - j * BLOCK_N, lane);
          const int buf = j & 1;
          const uint32_t par = static_cast<uint32_t>((j >> 1) & 1);
          mbar_wait(&p_half[buf], par);        // (p_half[half][group])
          tc_fence_after();
          issue_pv(buf, stage, 0, j > 0);
          mbar_wait(&p_half[2 + buf], par);
          tc_fence_after();
          issue_pv(buf, stage, 1, true);
        }
        release(stage);
        advance();
      }
    }
  } else if (warp_idx >= 4) {
    // ============================== softmax / correction / epilogue ==============================
    setmaxnreg_inc<216>();
    const int w = (warp_idx - 4) >> 2;           // 0: even KV blocks, 1: odd KV blocks
    const int quad = warp_idx & 3;               // TMEM lane quadrant
    const int row = quad * 32 + lane;            // row inside the tile
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t tS = tmem_base + lane_addr + C::TMEM_S + static_cast<uint32_t>(w * 128);
    const uint32_t tP = tmem_base + lane_addr + C::TMEM_P + static_cast<uint32_t>(w * 64);
    const uint32_t tO = tmem_base + lane_addr + C::TMEM_O;
    // barrier addresses as two opaque base registers (this group's / the other group's slot) + constant offsets
    // (see smem_addr_opaque); p_half is laid out [half][group] so that it follows the same rule
    const uint32_t base_w = smem_addr_opaque(q_full) + static_cast<uint32_t>(w) * 8u;
    const uint32_t base_o = base_w + 8u - static_cast<uint32_t>(w) * 16u;   // (w ^ 1) * 8
    auto bar_off = [&](const uint64_t* b0) { return static_cast<uint32_t>((b0 - q_full) * 8); };
    const uint32_t a_s_full = base_w + bar_off(s_full);
    const uint32_t a_s_free = base_w + bar_off(s_free);
    const uint32_t a_p_half = base_w + bar_off(p_half);   // + half * 16
    const uint32_t a_pv_mine = base_w + bar_off(pv_done);
    const uint32_t a_pv_other = base_o + bar_off(pv_done);
    const uint32_t a_ref_mine = base_w + bar_off(ref_bar);
    const uint32_t a_ref_other = base_o + bar_off(ref_bar);

    const int q_row = tile_row0 + row;
    float m_own = -INFINITY;  // reference max (log2 units) this group's l_run (and the P it stored last) are relative to
    float l_run = 0.f;        // this group's share of the row sum
    const int64_t q_pos_plus = static_cast<int64_t>(q_row) + coff;  // last visible key under causal
    // exp2(a - b) with the convention exp2(-inf - x) = 0, also for x = -inf
    auto ratio = [](float a, float b) { return a == -INFINITY ? 0.f : fast_exp2(a - b); };

    for (int j = w; j < n_mine; j += 2) {
      const uint32_t par = static_cast<uint32_t>((j >> 1) & 1);
      mbar_wait_addr(a_s_full, par);
      tc_fence_after();
      uint32_t s[128];
      tmem_ld_x32(tS + 0, s + 0);
      tmem_ld_x32(tS + 32, s + 32);
      tmem_ld_x32(tS + 64, s + 64);
      tmem_ld_x32(tS + 96, s + 96);
      tmem_wait_ld();
      // the scores are in registers: the buffer goes back to the MMA warp for Q K(j+2)^T
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_addr(a_s_free);
      // ---- masking: keys >= limit (relative to the tile) are invisible ----
      const int kv0 = j * BLOCK_N;
      int limit = kv_len - kv0;
      if (p.causal) {
        const int64_t cl = q_pos_plus - kv0 + 1;
        if (cl < limit) limit = static_cast<int>(cl < 0 ? 0 : cl);
      }
      if (limit < BLOCK_N) {
#pragma unroll
        for (int c = 0; c < 128; ++c)
          if (c >= limit) s[c] = 0xFF800000u;  // -inf
      }
      const float2 sc2 = make_float2(p.scale_log2, p.scale_log2);
      float2 nm2, sum2;
      uint32_t pk0[32], pk1[32];
#ifndef B200_FA_PAIR_POLY_MOD
#define B200_FA_PAIR_POLY_MOD 4
#endif
      auto exp_pair = [&](int c) -> uint32_t {
        const float2 x = __ffma2_rn(make_float2(__uint_as_float(s[c]), __uint_as_float(s[c + 1])), sc2, nm2);
        const bool poly = B200_FA_PAIR_POLY_MOD > 0 && ((c >> 1) % (B200_FA_PAIR_POLY_MOD > 0 ? B200_FA_PAIR_POLY_MOD : 1)) == 1;
        const float2 e = poly ? exp2_poly2(x) : make_float2(fast_exp2(x.x), fast_exp2(x.y));
        sum2 = __fadd2_rn(sum2, e);
        return Pack2<T>::pack(e.x, e.y);
      };
      auto set_reference = [&](float m) {
        const float m_ref = (m == -INFINITY) ? 0.f : m;
        nm2 = make_float2(-m_ref, -m_ref);
        sum2 = make_float2(0.f, 0.f);
      };
      auto publish = [&](int half) {
        tmem_wait_st();
        __syncwarp();
        if (lane == 0) mbar_arrive_addr(a_p_half + static_cast<uint32_t>(half) * 16u);
      };
      // ---- speculative first half against the reference this group used last (it rarely moves, see K1 notes) ----
      const float m_spec = m_own;
      set_reference(m_spec);
#pragma unroll
      for (int i = 0; i < 32; ++i) pk0[i] = exp_pair(2 * i);
      // ---- row max of this block ----
      float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
      for (int c = 0; c < 128; c += 4) {
        mx0 = fmaxf(mx0, __uint_as_float(s[c + 0]));
        mx1 = fmaxf(mx1, __uint_as_float(s[c + 1]));
        mx2 = fmaxf(mx2, __uint_as_float(s[c + 2]));
        mx3 = fmaxf(mx3, __uint_as_float(s[c + 3]));
      }
      const float m_tile = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * p.scale_log2;
      // ---- the reference block j-1 (other group) left behind ----
      float m_in = -INFINITY;
      if (j >= 1) {
        mbar_wait_addr(a_ref_other, static_cast<uint32_t>(((j - 1) >> 1) & 1));
        m_in = mref[row];
      }
      if (m_in != m_own) l_run *= ratio(m_own, m_in);  // our partial sum follows the reference the other group moved
      // ---- lazy rescale decision for block j ----
      float m_out = m_in, alpha = 1.0f;
      bool rescale = false;
      if (m_tile > m_in + kRescaleThreshold) {  // (m_in = -inf until the first visible key)
        m_out = m_tile;
        alpha = ratio(m_in, m_out);
        l_run *= alpha;
        rescale = true;
      }
      if (__any_sync(0xffffffffu, rescale) && j > 0) {
        // O must contain P(j-1) V(j-1) (other group's buffer) before it is rescaled
        mbar_wait_addr(a_pv_other, static_cast<uint32_t>(((j - 1) >> 1) & 1));
        tc_fence_after();
        // (rare path, rolled loop of 16-column pieces: a 32-register block here makes ptxas route the S registers of
        // the hot path through local memory)
#pragma unroll 1
        for (int c = 0; c < D / 16; ++c) {
          uint32_t o[16];
          tmem_ld_x16(tO + c * 16, o);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
          tmem_st_x16(tO + c * 16, o);
        }
        tmem_wait_st();
      }
      // ---- publish the reference (and the rescaled O) for block j+1 ----
      mref[row] = m_out;
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_addr(a_ref_mine);
      m_own = m_out;
      if (__any_sync(0xffffffffu, m_out != m_spec)) {
        // the speculation failed for at least one row of this warp: redo the first half against the reference in force
        set_reference(m_out);
#pragma unroll
        for (int i = 0; i < 32; ++i) pk0[i] = exp_pair(2 * i);
      }
      // ---- our P buffer is free once P(j-2) V(j-2) retired ----
      if (j >= 2) {
        mbar_wait_addr(a_pv_mine, static_cast<uint32_t>(((j - 2) >> 1) & 1));
        tc_fence_after();
      }
      tmem_st_x32(tP, pk0);
#pragma unroll
      for (int i = 0; i < 16; ++i) pk1[i] = exp_pair(64 + 2 * i);
      publish(0);
#pragma unroll
      for (int i = 16; i < 32; ++i) pk1[i] = exp_pair(64 + 2 * i);
      tmem_st_x32(tP + 32, pk1);
      l_run += sum2.x + sum2.y;
      publish(1);
    }

    // ---- epilogue: both groups agree on the final reference, add their partial sums, and write half of the columns each ----
    if (tile_row0 < p.Sq) {
      const bool row_ok = q_row < p.Sq;
      float m_fin = m_own;
      if (n_mine > 0) {
        const int wl = (n_mine - 1) & 1;  // the group that processed the last block holds the final reference
        if (w != wl) {
          mbar_wait_addr(a_ref_other, static_cast<uint32_t>(((n_mine - 1) >> 1) & 1));
          m_fin = mref[row];
          if (m_fin != m_own) l_run *= ratio(m_own, m_fin);
        }
      }
      [[maybe_unused]] float lse_old = -INFINITY;
      if constexpr (ACCUM) {
        if (!p.acc_init && row_ok)
          lse_old = p.lse_acc[static_cast<int64_t>(batch) * p.lse_sb + static_cast<int64_t>(head) * p.lse_sh + q_row];
      }
      lsum[w * 128 + row] = l_run;
      named_bar_sync(1, 256);
      const float l_tot = lsum[row] + lsum[128 + row];
      float inv_l = 0.f;
      float lse_val = -INFINITY;
      if (n_mine > 0) {
        const int wl = (n_mine - 1) & 1;
        mbar_wait_addr(wl == w ? a_pv_mine : a_pv_other, static_cast<uint32_t>(((n_mine - 1) >> 1) & 1));
        tc_fence_after();
        if (l_tot > 0.f && m_fin != -INFINITY) {  // (a row without a visible key keeps the reference at -inf)
          inv_l = 1.0f / l_tot;
          lse_val = (m_fin + log2f(l_tot)) * kLn2;
        }
      }
      const uint32_t tOh = tO + static_cast<uint32_t>(w * (D / 2));
      if constexpr (!ACCUM) {
        if (p.lse != nullptr && row_ok && w == 0) p.lse[(static_cast<int64_t>(batch) * p.Hq + head) * p.Sq + q_row] = lse_val;
        T* orow = reinterpret_cast<T*>(p.o) + static_cast<int64_t>(batch) * p.o_sb + static_cast<int64_t>(q_row) * p.o_ss +
                  static_cast<int64_t>(head) * p.o_sh + w * (D / 2);
#pragma unroll
        for (int c = 0; c < D / 64; ++c) {
          uint32_t o[32];
          if (n_mine > 0) {
            tmem_ld_x32(tOh + c * 32, o);
            tmem_wait_ld();
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = 0u;
          }
          if (row_ok) {
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              uint4 pk;
              pk.x = Pack2<T>::pack(__uint_as_float(o[q4 * 8 + 0]) * inv_l, __uint_as_float(o[q4 * 8 + 1]) * inv_l);
              pk.y = Pack2<T>::pack(__uint_as_float(o[q4 * 8 + 2]) * inv_l, __uint_as_float(o[q4 * 8 + 3]) * inv_l);
              pk.z = Pack2<T>::pack(__uint_as_float(o[q4 * 8 + 4]) * inv_l, __uint_as_float(o[q4 * 8 + 5]) * inv_l);
              pk.w = Pack2<T>::pack(__uint_as_float(o[q4 * 8 + 6]) * inv_l, __uint_as_float(o[q4 * 8 + 7]) * inv_l);
              if (w * (D / 2) + c * 32 + q4 * 8 < p.d_real) *reinterpret_cast<uint4*>(orow + c * 32 + q4 * 8) = pk;
            }
          }
        }
      } else {
        float* lrow = p.lse_acc + static_cast<int64_t>(batch) * p.lse_sb + static_cast<int64_t>(head) * p.lse_sh + q_row;
        float* arow = p.o_acc + static_cast<int64_t>(batch) * p.acc_sb + static_cast<int64_t>(q_row) * p.acc_ss +
                      static_cast<int64_t>(head) * p.acc_sh + w * (D / 2);
        float w_old = 0.f, w_new = inv_l, lse_out = lse_val;
        if (!p.acc_init && row_ok) {
          const float mx = fmaxf(lse_old, lse_val);
          if (mx == -INFINITY) {
            w_old = 0.f;
            w_new = 0.f;
            lse_out = -INFINITY;
          } else {
            const float e_old = fast_exp2((lse_old - mx) * kLog2e);
            const float e_new = fast_exp2((lse_val - mx) * kLog2e);
            const float den = e_old + e_new;
            lse_out = mx + log2f(den) * kLn2;
            w_old = e_old / den;
            w_new = e_new / den * inv_l;
          }
        }
        const bool touch = row_ok && (p.acc_init || lse_val != -INFINITY);
        if (touch && w == 0) *lrow = lse_out;
#pragma unroll
        for (int c = 0; c < D / 64; ++c) {
          uint32_t o[32];
          if (n_mine > 0) {
            tmem_ld_x32(tOh + c * 32, o);
            tmem_wait_ld();
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = 0u;
          }
          if (touch) {
#pragma unroll
            for (int q4 = 0; q4 < 8; ++q4) {
              if (w * (D / 2) + c * 32 + q4 * 4 >= p.d_real) continue;
              float4* dst = reinterpret_cast<float4*>(arow + c * 32 + q4 * 4);
              float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
              if (!p.acc_init) a = *dst;
              a.x = a.x * w_old + __uint_as_float(o[q4 * 4 + 0]) * w_new;
              a.y = a.y * w_old + __uint_as_float(o[q4 * 4 + 1]) * w_new;
              a.z = a.z * w_old + __uint_as_float(o[q4 * 4 + 2]) * w_new;
              a.w = a.w * w_old + __uint_as_float(o[q4 * 4 + 3]) * w_new;
              *dst = a;
            }
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer may still multicast into / arrive on this CTA's shared memory until it is done too
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int D, typename T, bool ACCUM>
int launch_pair(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const Params& p, cudaStream_t stream) {
  auto kern = fa_fwd_pair_kernel<D, T, ACCUM>;
  static bool attr_set[64] = {};  // per device
  B200_CUDA_OK(set_max_dynamic_smem(reinterpret_cast<const void*>(kern), Cfg2<D>::SMEM_BYTES, attr_set));
  dim3 grid(2 * p.num_pairs, p.Hq, p.B);  // clusters of 2 along x: the two 128-row tiles of a pair
  kern<<<grid, NUM_THREADS, Cfg2<D>::SMEM_BYTES, stream>>>(tq, tk, tv, p);
  B200_CUDA_OK(cudaGetLastError());
  note_launch("fa_fwd_pair_kernel");
  return B200_OK;
}

static int make_bshd_tmap(CUtensorMap* out, const void* base, int B, int S, int H, int D, const int64_t strides[3],
                          const char* name, uint32_t box_rows = 128) {
  // tensor addressed as [b][s][h][d] with element strides (b, s, h); TMA dims innermost-first: (d, h, s, b)
  for (int i = 0; i < 3; ++i)
    if (strides[i] <= 0 || strides[i] % 8 != 0)
      return set_error(B200_ERR_INVALID_ARGUMENT, "%s stride %d = %lld must be a positive multiple of 8 elements", name,
                       i, (long long)strides[i]);
  uint64_t dims[4] = {static_cast<uint64_t>(D), static_cast<uint64_t>(H), static_cast<uint64_t>(S),
                      static_cast<uint64_t>(B)};
  uint64_t str[3] = {static_cast<uint64_t>(strides[2]) * 2, static_cast<uint64_t>(strides[1]) * 2,
                     static_cast<uint64_t>(strides[0]) * 2};
  uint32_t box[4] = {64, 1, box_rows, 1};
  return encode_tmap_sw128_16b(out, base, 4, dims, str, box);
}

}  // namespace fa
}  // namespace b200

#ifdef B200_FA_TRACE
extern "C" int b200_debug_fa_trace(long long* dev_buf) {
  return cudaMemcpyToSymbol(b200::fa::g_trace, &dev_buf, sizeof(dev_buf)) == cudaSuccess ? 0 : -3;
}
#endif

namespace b200 {
namespace fa {

// shared host path of b200_fa_fwd (16-bit output) and b200_fa_fwd_accum (merge into an fp32 accumulator)
static int run(const void* q, const void* k, const void* v, int B, int Sq, int Sk, int Hq, int Hkv, int D,
               const int64_t q_strides[3], const int64_t k_strides[3], const int64_t v_strides[3], float softmax_scale,
               int causal, int64_t causal_offset, const int32_t* kv_lens, int dtype, void* stream, Params p, bool accum) {
  B200_CHECK_ARG(q && k && v && q_strides && k_strides && v_strides, "fa_fwd: NULL pointer argument");
  B200_CHECK_ARG(B > 0 && Sq > 0 && Sk > 0 && Hq > 0 && Hkv > 0, "fa_fwd: bad sizes B=%d Sq=%d Sk=%d Hq=%d Hkv=%d", B, Sq,
                 Sk, Hq, Hkv);
  B200_CHECK_ARG(Hq % Hkv == 0, "fa_fwd: Hq (%d) must be a multiple of Hkv (%d)", Hq, Hkv);
  // head_dim: any multiple of 8 up to 128 (reference: hidden_size // num_heads, unconstrained). The kernels are built for
  // 64 and 128 columns; a narrower head runs in the next wider build with its missing columns zero-filled by TMA.
  B200_CHECK_ARG(D >= 8 && D <= 128 && D % 8 == 0, "fa_fwd: head_dim %d unsupported (a multiple of 8, at most 128)", D);
  p.d_real = D;
  const int KD = D <= 64 ? 64 : 128;  // the kernel build
  B200_CHECK_ARG(dtype == B200_DTYPE_BF16 || dtype == B200_DTYPE_FP16, "fa_fwd: dtype must be bf16 or fp16");
  B200_CHECK_ARG(softmax_scale > 0.f, "fa_fwd: softmax_scale must be positive");
  B200_CHECK_ARG(B <= 65535 && Hq <= 65535, "fa_fwd: B and Hq must be <= 65535");
  CUtensorMap tq, tk, tv;
  int rc;
  // CTA-pair kernel (one 128-row tile per CTA, K/V multicast across the pair): B200_FA_PAIR=1/0 forces it on/off
  // (read per call: tests flip it inside one process). It does not read the paged cache.
  const char* pair_env = getenv("B200_FA_PAIR");
  const bool use_pair = p.block_table == nullptr && (pair_env != nullptr ? pair_env[0] == '1' : kPairDefault);
  if ((rc = make_bshd_tmap(&tq, q, B, Sq, Hq, D, q_strides, "q"))) return rc;
  if (p.block_table != nullptr) {
    // paged: k / v point at the layer's slice of the cache; k_strides = (block, token, head) element strides, box = one block
    for (int which = 0; which < 2; ++which) {
      const int64_t* st = which == 0 ? k_strides : v_strides;
      // (for the paged call `Sk` carries the number of PHYSICAL blocks of the cache: the extent of the tensor map)
      uint64_t dims[4] = {static_cast<uint64_t>(D), static_cast<uint64_t>(Hkv), static_cast<uint64_t>(p.block_size),
                          static_cast<uint64_t>(Sk)};
      uint64_t str[3] = {static_cast<uint64_t>(st[2]) * 2, static_cast<uint64_t>(st[1]) * 2, static_cast<uint64_t>(st[0]) * 2};
      uint32_t box[4] = {64, 1, static_cast<uint32_t>(p.block_size), 1};
      if ((rc = encode_tmap_sw128_16b(which == 0 ? &tk : &tv, which == 0 ? k : v, 4, dims, str, box))) return rc;
    }
    Sk = p.max_blocks * p.block_size;  // the key range the kernel walks is bounded by the block table
  } else {
    if ((rc = make_bshd_tmap(&tk, k, B, Sk, Hkv, D, k_strides, "k", use_pair ? 64 : 128))) return rc;
    if ((rc = make_bshd_tmap(&tv, v, B, Sk, Hkv, D, v_strides, "v", use_pair ? 64 : 128))) return rc;
  }
  // B200_FA_PERSISTENT=0 in the environment: every CTA handles only its own block (no work stealing)
  static const bool persistent = [] { const char* e = getenv("B200_FA_PERSISTENT"); return !(e && e[0] == '0'); }();
  p.persistent = persistent ? 1 : 0;
  p.kv_lens = kv_lens;
  p.B = B; p.Sq = Sq; p.Sk = Sk; p.Hq = Hq; p.Hkv = Hkv;
  p.scale_log2 = softmax_scale * kLog2e;
  p.causal = causal ? 1 : 0;
  p.causal_offset = causal_offset;
  p.num_pairs = (Sq + 2 * BLOCK_M - 1) / (2 * BLOCK_M);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool bf = dtype == B200_DTYPE_BF16;
  if (use_pair) {
    if (accum) {
      if (KD == 128) return bf ? launch_pair<128, __nv_bfloat16, true>(tq, tk, tv, p, s) : launch_pair<128, __half, true>(tq, tk, tv, p, s);
      return bf ? launch_pair<64, __nv_bfloat16, true>(tq, tk, tv, p, s) : launch_pair<64, __half, true>(tq, tk, tv, p, s);
    }
    if (KD == 128) return bf ? launch_pair<128, __nv_bfloat16, false>(tq, tk, tv, p, s) : launch_pair<128, __half, false>(tq, tk, tv, p, s);
    return bf ? launch_pair<64, __nv_bfloat16, false>(tq, tk, tv, p, s) : launch_pair<64, __half, false>(tq, tk, tv, p, s);
  }
  if (accum) {
    if (KD == 128) return bf ? launch<128, __nv_bfloat16, true>(tq, tk, tv, p, s) : launch<128, __half, true>(tq, tk, tv, p, s);
    return bf ? launch<64, __nv_bfloat16, true>(tq, tk, tv, p, s) : launch<64, __half, true>(tq, tk, tv, p, s);
  }
  if (KD == 128) return bf ? launch<128, __nv_bfloat16, false>(tq, tk, tv, p, s) : launch<128, __half, false>(tq, tk, tv, p, s);
  return bf ? launch<64, __nv_bfloat16, false>(tq, tk, tv, p, s) : launch<64, __half, false>(tq, tk, tv, p, s);
}

}  // namespace fa
}  // namespace b200

extern "C" int b200_fa_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int B, int Sq, int Sk,
                           int Hq, int Hkv, int D, const int64_t q_strides[3], const int64_t k_strides[3],
                           const int64_t v_strides[3], const int64_t o_strides[3], float softmax_scale, int causal,
                           int64_t causal_offset, const int32_t* kv_lens, int dtype, void* stream) {
  using namespace b200;
  B200_CHECK_ARG(o && o_strides, "fa_fwd: NULL output argument");
  for (int i = 0; i < 3; ++i)
    B200_CHECK_ARG(o_strides[i] > 0 && o_strides[i] % 8 == 0, "fa_fwd: o stride %d = %lld must be a positive multiple of 8 elements",
                   i, (long long)o_strides[i]);
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(o) & 15) == 0, "fa_fwd: o must be 16-byte aligned");
  fa::Params p{};
  p.o = o;
  p.o_sb = o_strides[0]; p.o_sh = o_strides[2]; p.o_ss = o_strides[1];
  p.lse = lse;
  return fa::run(q, k, v, B, Sq, Sk, Hq, Hkv, D, q_strides, k_strides, v_strides, softmax_scale, causal, causal_offset, kv_lens,
                 dtype, stream, p, false);
}

extern "C" int b200_fa_fwd_accum(const void* q, const void* k, const void* v, float* o_acc, float* lse_acc, int B, int Sq,
                                 int Sk, int Hq, int Hkv, int D, const int64_t q_strides[3], const int64_t k_strides[3],
                                 const int64_t v_strides[3], const int64_t acc_strides[3], const int64_t lse_strides[2],
                                 float softmax_scale, int causal, int64_t causal_offset, const int32_t* kv_lens, int init,
                                 int dtype, void* stream) {
  using namespace b200;
  B200_CHECK_ARG(o_acc && lse_acc && acc_strides && lse_strides, "fa_fwd_accum: NULL accumulator argument");
  for (int i = 0; i < 3; ++i)
    B200_CHECK_ARG(acc_strides[i] > 0 && acc_strides[i] % 4 == 0,
                   "fa_fwd_accum: accumulator stride %d = %lld must be a positive multiple of 4 elements", i,
                   (long long)acc_strides[i]);
  B200_CHECK_ARG(lse_strides[0] > 0 && lse_strides[1] >= Sq, "fa_fwd_accum: bad LSE strides");
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(o_acc) & 15) == 0, "fa_fwd_accum: o_acc must be 16-byte aligned");
  fa::Params p{};
  p.o_acc = o_acc;
  p.acc_sb = acc_strides[0]; p.acc_ss = acc_strides[1]; p.acc_sh = acc_strides[2];
  p.lse_acc = lse_acc;
  p.lse_sb = lse_strides[0]; p.lse_sh = lse_strides[1];
  p.acc_init = init ? 1 : 0;
  return fa::run(q, k, v, B, Sq, Sk, Hq, Hkv, D, q_strides, k_strides, v_strides, softmax_scale, causal, causal_offset, kv_lens,
                 dtype, stream, p, true);
}

extern "C" int b200_fa_fwd_paged(const void* q, const void* k_cache, const void* v_cache, void* o, float* lse, int B, int Sq,
                                 int Hq, int Hkv, int D, const int64_t q_strides[3], const int64_t o_strides[3],
                                 const int32_t* block_tables, int max_blocks_per_seq, int block_size, int num_blocks,
                                 int num_layers, int layer_idx, const int32_t* context_lens, float softmax_scale, int causal,
                                 int dtype, void* stream) {
  using namespace b200;
  B200_CHECK_ARG(o && o_strides && k_cache && v_cache && block_tables && context_lens, "fa_fwd_paged: NULL pointer argument");
  B200_CHECK_ARG(block_size >= 8 && block_size <= 128 && (block_size & (block_size - 1)) == 0,
                 "fa_fwd_paged: block_size %d must be a power of two in [8, 128]", block_size);
  B200_CHECK_ARG(max_blocks_per_seq > 0 && num_blocks > 0 && num_layers > 0 && layer_idx >= 0 && layer_idx < num_layers,
                 "fa_fwd_paged: bad paged-cache arguments");
  B200_CHECK_ARG(D == 64 || D == 128, "fa_fwd_paged: head_dim %d unsupported (the paged cache holds 64 or 128)", D);
  for (int i = 0; i < 3; ++i)
    B200_CHECK_ARG(o_strides[i] > 0 && o_strides[i] % 8 == 0, "fa_fwd_paged: o stride %d = %lld must be a positive multiple of 8 elements",
                   i, (long long)o_strides[i]);
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(o) & 15) == 0, "fa_fwd_paged: o must be 16-byte aligned");
  fa::Params p{};
  p.o = o;
  p.o_sb = o_strides[0]; p.o_sh = o_strides[2]; p.o_ss = o_strides[1];
  p.lse = lse;
  p.block_table = block_tables;
  p.max_blocks = max_blocks_per_seq;
  p.block_size = block_size;
  p.causal_bottom = causal ? 1 : 0;
  // cache layout [num_blocks, L, block_size, Hkv, D] (baseline/inference.py:1077-1084): element strides (block, token, head)
  const int64_t tok = static_cast<int64_t>(Hkv) * D;
  const int64_t cs[3] = {static_cast<int64_t>(num_layers) * block_size * tok, tok, static_cast<int64_t>(D)};
  const char* kb = static_cast<const char*>(k_cache) + static_cast<int64_t>(layer_idx) * block_size * tok * 2;
  const char* vb = static_cast<const char*>(v_cache) + static_cast<int64_t>(layer_idx) * block_size * tok * 2;
  return fa::run(q, kb, vb, B, Sq, /*Sk: physical blocks for the tensor map*/ num_blocks, Hq, Hkv, D, q_strides, cs, cs, softmax_scale,
                 causal, 0, context_lens, dtype, stream, p, false);
}
