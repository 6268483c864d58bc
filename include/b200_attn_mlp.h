/*
 * b200_attn_mlp.h — C-ABI of the B200 (sm_100a) attention + FusedMLP hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b). The reference has no FFI of its own: its seam is the Python
 * function layer in kernels/triton/*.py. Every entry point below names the reference function it replaces
 * (file:line under the reference tree). INTEGRATION.md shows the ctypes binding a reference maintainer adds.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types. Returns 0 (B200_OK) or a negative error
 *     code; b200_last_error() returns a thread-local description. Never throws, never allocates or frees
 *     caller memory, never synchronises the device.
 *   - All data pointers are DEVICE pointers. Strides are in ELEMENTS. `stream` is a cudaStream_t passed as
 *     void* (NULL = legacy default stream).
 *   - dtype: B200_DTYPE_BF16 or B200_DTYPE_FP16 for q/k/v/o/x/weights; statistics (LSE) and split-K partials
 *     are fp32. Accumulation and softmax are always fp32.
 *   - There is no CPU fallback: on a machine without an sm_100 GPU every compute call returns
 *     B200_ERR_NO_DEVICE / B200_ERR_CUDA.
 */
#ifndef B200_ATTN_MLP_H_
#define B200_ATTN_MLP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ERR_INVALID_ARGUMENT (-1)
#define B200_ERR_UNSUPPORTED (-2)
#define B200_ERR_CUDA (-3)
#define B200_ERR_NO_DEVICE (-4)
#define B200_ERR_WORKSPACE (-5)

#define B200_DTYPE_BF16 0
#define B200_DTYPE_FP16 1

/* Activation selector of the FusedMLP path.
 *   GELU_TANH : kernels/triton/mlp_kernels.py:144-161 (Triton kernel) == kernels/mlp/fused_mlp.py:223-237
 *   GELU_ERF  : kernels/mlp/fused_mlp.py:162-163, kernels/triton/mlp_kernels.py:783 (exact F.gelu)
 *   RELU      : kernels/triton/mlp_kernels.py:233-414, kernels/mlp/fused_mlp.py:299-315
 *   SWIGLU    : silu(gate) * up, kernels/triton/mlp_kernels.py:567-572, kernels/mlp/fused_mlp.py:262-275
 *   NONE      : plain Linear (+bias), used for the down projection alone                                  */
#define B200_ACT_NONE 0
#define B200_ACT_GELU_TANH 1
#define B200_ACT_GELU_ERF 2
#define B200_ACT_RELU 3
#define B200_ACT_SWIGLU 4

/* KV-cache layouts of the decode path */
#define B200_KV_CONTIGUOUS 0 /* [B, S_max, Hkv, D]                      baseline/inference.py:866-874   */
#define B200_KV_PAGED 1      /* [num_blocks, L, block_size, Hkv, D]     baseline/inference.py:1077-1084 */

/* ---- library / device -------------------------------------------------------------------------------- */
const char* b200_version(void);
const char* b200_last_error(void);
/* 1 if the current CUDA device is compute capability 10.x, 0 if not, negative error if no device. */
int b200_arch_ok(void);

/* Process-wide cap on the CTAs of the persistent GEMM kernels (0 = all SMs). The tensor-parallel MLP lowers it while an
 * NCCL all-reduce of the previous token chunk is in flight so that the collective finds free SMs (overlap instead of
 * serialisation, parallelism/tensor_parallel.py:302 rebuilt). */
int b200_set_sm_limit(int max_ctas);

/* L2 rasterisation of the persistent GEMM kernels: output tiles are visited in groups that cover `rows` rows of the
 * activation: the group's activation panel stays L2-resident while the weight is streamed once per group, so DRAM reads
 * ~ x + W * ceil(T / rows). rows = 0 (default) picks the largest group whose per-wave footprint fits a 48 MB L2 budget
 * (measured, csrc/gemm_mlp.cu choose_group_m); otherwise rows >= 256. (The reference's Triton kernels have no such
 * control: kernels/triton/mlp_kernels.py uses a plain 2-D grid, :690-705.) */
int b200_set_gemm_group_rows(int rows);

/* Measurement hooks (the reference's BenchmarkRunner counts nothing, benchmarks/runners.py:185-248): number of kernel
 * launches this library has issued in the process so far, the name of the GEMM kernel the last linear / FusedMLP
 * call dispatched to and the name of the kernel launched last, whatever it was (static strings). */
int64_t b200_launch_count(void);
const char* b200_last_gemm_kernel(void);
const char* b200_last_kernel(void);

/* ---- K1: tiled online-softmax attention forward (prefill) -------------------------------------------
 * Replaces triton_flash_attention / _flash_attention_forward_kernel
 *   (kernels/triton/flash_attention_kernels.py:1150-1358, :38-325), the attention inside
 *   FlashAttention3.forward (kernels/attention/flash_attention.py:145-225), and — called once per ring step —
 *   triton_ring_attention_forward (kernels/triton/attention_kernels.py:909-998).
 *
 *   O[b,i,h,:] = softmax_j( scale * <Q[b,i,h,:], K[b,j,h/g,:]> + mask ) V[b,j,h/g,:],   g = Hq/Hkv
 *   LSE[b,h,i] = log sum_j exp(scale * s_ij)          (fp32, natural log; -inf for a fully masked row, O = 0)
 *
 *   mask: key j is visible to query i iff  j < kv_len(b)  and (not causal or  j <= i + causal_offset).
 *         causal_offset = (global position of query row 0) - (global position of key row 0); 0 for
 *         self-attention prefill (reference: triu(diagonal=1), flash_attention.py:1221-1225), Sk - Sq for
 *         bottom-right alignment, arbitrary for ring steps / chunked prefill.
 *   kv_lens: optional int32[B] (device) per-batch key count (right-padding masks); NULL = Sk for all.
 *
 *   q [B,Sq,Hq,D], k/v [B,Sk,Hkv,D], o [B,Sq,Hq,D] addressed through (batch, seq, head) element strides,
 *   D contiguous; D = any multiple of 8 up to 128 (the reference takes hidden_size // num_heads as it comes,
 *   flash_attention.py:176; kernels are built for 64 and 128 columns, a narrower head runs in the next wider build with
 *   the missing columns zero-filled by the TMA loads and never stored); pointers 16-byte aligned and strides multiples
 *   of 8 elements. (The decode kernels and the caches take D in {64, 128}; the Python layer stores narrower heads in the
 *   next wider cache with zero columns behind them.)
 *   lse: fp32 [B,Hq,Sq] contiguous, may be NULL.                                                          */
int b200_fa_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int B, int Sq, int Sk, int Hq,
                int Hkv, int D, const int64_t q_strides[3], const int64_t k_strides[3], const int64_t v_strides[3],
                const int64_t o_strides[3], float softmax_scale, int causal, int64_t causal_offset,
                const int32_t* kv_lens, int dtype, void* stream);

/* ---- K1 in accumulate mode: one ring step --------------------------------------------------------------
 * Same computation as b200_fa_fwd, but the result of this key block is merged in the kernel epilogue into a running
 * fp32 output + LSE (the step of SequenceParallelAttention._ring_attention, parallelism/sequence_parallel.py:519-585,
 * rebuilt exact with the merge algebra of kernels/triton/attention_kernels.py:1567-1585):
 *   init != 0 : o_acc = O, lse_acc = LSE                       (first step)
 *   init == 0 : lse = logaddexp(lse_acc, LSE); o_acc = o_acc*exp(lse_acc-lse) + O*exp(LSE-lse); lse_acc = lse
 * Rows for which this block has no visible key leave the accumulator untouched (init: O = 0, LSE = -inf).
 *   o_acc  : fp32, addressed by element strides acc_strides = (batch, seq, head), head dim contiguous, 16-byte aligned
 *   lse_acc: fp32, rows of Sq contiguous, element strides lse_strides = (batch, head)
 * No 16-bit output tensor and no separate merge pass: b200_cast_out converts the accumulator at the end.   */
int b200_fa_fwd_accum(const void* q, const void* k, const void* v, float* o_acc, float* lse_acc, int B, int Sq, int Sk,
                      int Hq, int Hkv, int D, const int64_t q_strides[3], const int64_t k_strides[3],
                      const int64_t v_strides[3], const int64_t acc_strides[3], const int64_t lse_strides[2],
                      float softmax_scale, int causal, int64_t causal_offset, const int32_t* kv_lens, int init, int dtype,
                      void* stream);

/* ---- LSE merge: combine two partial attention results over disjoint key sets ---------------------------
 * The online-softmax merge algebra of kernels/triton/attention_kernels.py:1567-1585, used by the ring
 * (parallelism/sequence_parallel.py:519-585 rebuilt exact):
 *   lse = logaddexp(lse_a, lse_b);  o = o_a * exp(lse_a - lse) + o_b * exp(lse_b - lse)
 * In place on (o_acc fp32 [B,Sq,Hq,D] contiguous, lse_acc fp32 [B,Hq,Sq]); the incoming block is (o_b 16-bit
 * with strides, lse_b fp32 [B,Hq,Sq]). A side with lse = -inf contributes nothing.                        */
int b200_lse_merge(float* o_acc, float* lse_acc, const void* o_b, const float* lse_b, int B, int Sq, int Hq, int D,
                   const int64_t ob_strides[3], int dtype, void* stream);

/* Convert the fp32 ring accumulator to the 16-bit output tensor (strided). */
int b200_cast_out(const float* o_acc, void* o, int B, int Sq, int Hq, int D, const int64_t o_strides[3], int dtype,
                  void* stream);

/* ---- K2: single-token decode attention against a KV cache (HBM-bound, split-K) -------------------------
 * Replaces triton_paged_attention_forward / _paged_attention_fwd_kernel
 *   (kernels/triton/attention_kernels.py:1206-1311, :628-808).  No causal mask, keys j < context_len(b)
 *   (attention_kernels.py:771-777).  GQA: query head h reads kv head h / (Hq/Hkv).
 *
 *   q, o      : [B, Hq, D] (the reference's [B,Hq,1,D] with the unit axis dropped), contiguous
 *   k_cache, v_cache :
 *       B200_KV_CONTIGUOUS  [B, S_max, Hkv, D]   (kv_batch_stride / kv_token_stride in elements)
 *       B200_KV_PAGED       [num_blocks, L, block_size, Hkv, D] contiguous, addressed through
 *                           block_table int32 [B, max_blocks_per_seq] and layer_idx
 *   context_lens : int32 [B] (device), number of valid keys per sequence (includes the appended token)
 *   lse       : optional fp32 [B, Hq]
 *   num_splits: >= 1 splits of the key axis per (batch, kv head); 0 = choose so the grid fills the SMs.
 *   workspace : device scratch of at least b200_fa_decode_workspace_bytes(...) bytes (may be NULL when the
 *               resolved num_splits == 1).                                                               */
int64_t b200_fa_decode_workspace_bytes(int B, int Hq, int Hkv, int D, int max_context_len, int num_splits);
int b200_fa_decode_num_splits(int B, int Hq, int Hkv, int D, int max_context_len);
int b200_fa_decode(const void* q, const void* k_cache, const void* v_cache, void* o, float* lse, int B, int Hq,
                   int Hkv, int D, const int32_t* context_lens, int max_context_len, float softmax_scale, int layout,
                   int64_t kv_batch_stride, int64_t kv_token_stride, const int32_t* block_table,
                   int max_blocks_per_seq, int block_size, int num_layers, int layer_idx, int num_splits,
                   void* workspace, int64_t workspace_bytes, int dtype, void* stream);

/* ---- KV append: write the new token's K,V into the cache at position context_len-1 --------------------
 * Replaces triton_reshape_and_cache / _reshape_and_cache_kernel (attention_kernels.py:1314-1407, :811-905).
 *   key, value: [B, Hkv, D] contiguous (the reference's [B,1,Hkv,D]).
 *   Bounds: a position >= the cache capacity is DROPPED (never written into another sequence's rows): capacity =
 *   max_blocks_per_seq * block_size for the paged layout; for the contiguous layout pass S_max as max_blocks_per_seq
 *   (block_size = 0), 0 = unchecked. b200_fa_decode clamps context_lens to min(max_context_len, capacity) likewise.  */
int b200_kv_append(const void* key, const void* value, void* k_cache, void* v_cache, int B, int Hkv, int D,
                   const int32_t* context_lens, int layout, int64_t kv_batch_stride, int64_t kv_token_stride,
                   const int32_t* block_table, int max_blocks_per_seq, int block_size, int num_layers,
                   int layer_idx, int dtype, void* stream);

/* ---- FP8 (e4m3) paged KV cache: quantizing append and decode ------------------------------------------------
 * Format (the same for every writer and reader): element torch.float8_e4m3fn, one fp32 k_scale and one v_scale per
 * layer (> 0 and finite). Stored byte = cvt.rn.satfinite.e4m3(x / scale) with a correctly rounded fp32 division:
 * |x / scale| past 448 and +-inf saturate to +-448, NaN stays NaN. Value read = byte * scale. Paged layout only:
 * [num_blocks, L, block_size, Hkv, D] bytes, D in {64, 128}.
 *
 * b200_kv_append_fp8: key, value [B, n_tokens, Hkv, D] contiguous, bf16 or fp16 (dtype). Row i of sequence b goes to
 *   position context_lens[b] - n_tokens + i: n_tokens = 1 is the decode append, n_tokens = S the prompt of prefill.
 *   Positions below 0 or >= max_blocks_per_seq * block_size are dropped, as in b200_kv_append.
 * b200_fa_decode_fp8: the contract of b200_fa_decode for the paged layout, over an FP8 cache; q / o bf16 or fp16, lse
 *   optional, same split rule (b200_fa_decode_num_splits) and workspace size (b200_fa_decode_workspace_bytes).
 *   k_scale is folded into softmax_scale, v_scale multiplies each output row. B200_KV_CONTIGUOUS returns
 *   B200_ERR_UNSUPPORTED. Cache bytes at or past context_lens[b] are never read.                                */
int b200_kv_append_fp8(const void* key, const void* value, void* k_cache, void* v_cache, int B, int n_tokens, int Hkv,
                       int D, const int32_t* context_lens, const int32_t* block_table, int max_blocks_per_seq,
                       int block_size, int num_layers, int layer_idx, float k_scale, float v_scale, int dtype,
                       void* stream);
int b200_fa_decode_fp8(const void* q, const void* k_cache, const void* v_cache, void* o, float* lse, int B, int Hq,
                       int Hkv, int D, const int32_t* context_lens, int max_context_len, float softmax_scale, int layout,
                       const int32_t* block_table, int max_blocks_per_seq, int block_size, int num_layers,
                       int layer_idx, int num_splits, void* workspace, int64_t workspace_bytes, float k_scale,
                       float v_scale, int dtype, void* stream);

/* ---- K3: FusedMLP ---------------------------------------------------------------------------------------
 * Replaces triton_fused_mlp (kernels/triton/mlp_kernels.py:648-756) and FusedMLP*._forward_*
 *   (kernels/mlp/fused_mlp.py:59-72, :159-178, :223-237, :262-275):
 *      y = act(x W_up^T + b_up) W_down^T + b_down                        (GELU_TANH / GELU_ERF / RELU)
 *      y = (silu(x W_gate^T + b_gate) * (x W_up^T + b_up)) W_down^T + b_down          (SWIGLU)
 *   x [T, h] (row stride ldx), w_up / w_gate [i, h], w_down [h_out, i] in nn.Linear layout ([out, in], row
 *   contiguous), biases [i] / [h_out] or NULL, y [T, h_out] (row stride ldy). h, i, h_out multiples of 8.
 *   workspace: b200_fused_mlp_workspace_bytes(T, h, i) bytes: the activated 16-bit intermediate [T, i] (written once,
 *   consumed by the down projection) plus split-K partials for decode-sized T; see DESIGN.md.           */
int64_t b200_fused_mlp_workspace_bytes(int64_t T, int h, int i);
int b200_fused_mlp(const void* x, int64_t ldx, const void* w_up, const void* b_up, const void* w_gate,
                   const void* b_gate, const void* w_down, const void* b_down, void* y, int64_t ldy, int64_t T,
                   int h, int i, int h_out, int act, void* workspace, int64_t workspace_bytes, int dtype,
                   void* stream);

/* One tcgen05 GEMM with a fused epilogue: y = act(x W^T + b) (or the SwiGLU pair form when w_gate != NULL).
 * This is ColumnParallelLinear/RowParallelLinear's F.linear (parallelism/tensor_parallel.py:173, :299) and
 * the building block of b200_fused_mlp. x [T,K] (ldx), w [N,K], y [T,N] (ldy).                          */
/* workspace: optional device scratch of b200_linear_act_workspace_bytes(...) bytes; when present, skinny problems
 * (few output tiles, long K: decode-sized T) run split-K across the SMs with an fp32 reduce pass. NULL = never split. */
int64_t b200_linear_act_workspace_bytes(int64_t T, int K, int N, int act);
int b200_linear_act(const void* x, int64_t ldx, const void* w, const void* b, const void* w_gate,
                    const void* b_gate, void* y, int64_t ldy, int64_t T, int K, int N, int act, void* workspace,
                    int64_t workspace_bytes, int dtype, void* stream);

/* ---- LayerNorm (+ residual) — the op feeding the attention / MLP blocks (SURVEY.md §8 f3) --------------------
 * Replaces triton_layernorm / _layernorm_fwd_kernel / _layernorm_residual_fwd_kernel
 *   (kernels/triton/layernorm_kernels.py:191-277, :36-190):
 *     y = LayerNorm(x + residual_alpha * residual) * weight + bias      (residual, bias may be NULL)
 *   mean / biased variance over the last dimension in fp32 (two-pass), eps inside the sqrt (:305-308).
 *   x, residual, y: [rows, cols] with row strides ldx/ldr/ldy (elements); cols % 8 == 0, cols <= 8192.            */
int b200_layernorm(const void* x, const void* residual, const void* weight, const void* bias, void* y, int64_t rows,
                   int cols, int64_t ldx, int64_t ldr, int64_t ldy, float eps, float residual_alpha, int dtype,
                   void* stream);

/* ---- K1 over the paged cache: short-q / chunked-prefill attention (q_len > 1) --------------------------
 * Replaces triton_paged_attention_forward for q_seq_len > 1 (kernels/triton/attention_kernels.py:1206-1311, which picks
 * BLOCK_SIZE_M = 64 for it, :1251) and FlashAttentionLayer's paged branch (kernels/attention/flash_attention.py:572-621).
 *   q, o        : [B, Sq, Hq, D] by element strides (batch, seq, head); the Sq new tokens of every sequence, whose K/V
 *                 have ALREADY been written to the cache
 *   k/v_cache   : [num_blocks, L, block_size, Hkv, D] contiguous; block_size a power of two in [8, 128]
 *   block_tables: int32 [B, max_blocks_per_seq]; context_lens int32 [B] = keys of each sequence INCLUDING the Sq new ones
 *   causal != 0 : query i of sequence b sees keys [0, context_lens[b] - Sq + i] (the diagonal ends at the sequence's last
 *                 key). The reference kernel leaves its causal mask commented out (:774-777), i.e. every new token would
 *                 see the later ones; causal = 0 reproduces that literally.
 * The KV tiles are gathered block by block with TMA through the block table inside the prefill kernel (tcgen05 path);
 * the cache must hold finite values in every slot of a block that is in use (PagedKVCache zero-fills).           */
int b200_fa_fwd_paged(const void* q, const void* k_cache, const void* v_cache, void* o, float* lse, int B, int Sq, int Hq,
                      int Hkv, int D, const int64_t q_strides[3], const int64_t o_strides[3], const int32_t* block_tables,
                      int max_blocks_per_seq, int block_size, int num_blocks, int num_layers, int layer_idx,
                      const int32_t* context_lens, float softmax_scale, int causal, int dtype, void* stream);

/* ---- K6: tensor-parallel all-reduce over NVSwitch multicast / peer memory -------------------------------
 * Replaces torch.distributed.all_reduce(output_parallel) + the bias add of RowParallelLinear.forward
 * (parallelism/tensor_parallel.py:296-308) and comm.all_reduce (parallelism/communication.py:37-209) for the
 * row-parallel down projection of the FusedMLP.
 *
 * In-place two-shot all-reduce (sum) of the byte range [data_offset, data_offset + nbytes) of a SYMMETRIC buffer:
 * a buffer of identical size on every rank, mapped into this process once per peer (`peer_bases[world]`, HOST array of
 * device pointers, own rank included) and — when the fabric supports it — once as a multicast address
 * (`multicast_base`, NULL selects the unicast peer load/store path). Rank r reduces slice r with
 * multimem.ld_reduce (fp32 accumulation inside the switch), optionally adds `bias` ([ncols], region = whole rows of
 * ncols elements) and broadcasts it with multimem.st. `flag_offset` names b200_tp_allreduce_flag_bytes() bytes inside
 * the symmetric buffer, zeroed once at creation; `epoch` must advance by 2 per call on that buffer, identically on all
 * ranks (the first call uses 1). All ranks must pass identical sizes and `max_ctas` (0 = one per SM; <= 160). Spins are bounded:
 * on a timeout (a peer never arrived) *error_flag (device int) is set to 1 and the kernel returns.            */
int64_t b200_tp_allreduce_flag_bytes(void);
int b200_tp_allreduce(void* multicast_base, void* const* peer_bases, int world, int rank, int64_t data_offset,
                      int64_t nbytes, int64_t flag_offset, uint32_t epoch, const void* bias, int ncols, int dtype,
                      int max_ctas, int* error_flag, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_ATTN_MLP_H_ */
