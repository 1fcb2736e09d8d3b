/*
 * deva_b200 - C ABI of the B200-native temporal-propagation kernels behind DEVA's
 * DEVAInferenceCore.step / MemoryManager API.
 *
 * The reference (hkchengrex/Tracking-Anything-with-DEVA @ 404a112) is pure Python/PyTorch and has no
 * FFI of its own; the boundary it exposes for this path is the set of Python call sites cited on each
 * entry point below.  A maintainer binds this library with ctypes (see INTEGRATION.md); the shipped
 * drop-in package does exactly that (tracking-anything-with-deva_b200/deva/_native.py).
 *
 * Conventions
 *  - every pointer is a CUDA device pointer unless marked HOST; fp16 buffers are passed as void*;
 *  - `stream` is a cudaStream_t (0 = legacy default stream); calls only enqueue work and never
 *    synchronise; inputs are borrowed until the enqueued work completes, outputs are caller-allocated;
 *  - return 0 on success; otherwise a non-zero code, with text available from deva_b200_last_error()
 *    (thread-local).  The Python side raises RuntimeError, mirroring the reference's exceptions;
 *  - "window" = the contiguous run of valid memory slots of one bucket's bank; slot indices in the
 *    outputs are relative to the window start.  The first `n_lead` (< 8) slots of a window are
 *    alignment padding and are masked out.
 */
#ifndef DEVA_B200_H_
#define DEVA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* v12: deva_b200_resize_rgb8, deva_b200_resize_rgb8_workspace_bytes, deva_b200_resize_aa_weights and
 * deva_b200_resize_labels (frames and first-frame masks resized to the evaluation size on the device).
 * v11: deva_b200_cbam / deva_b200_cbam_split take a larger scratch buffer (64 pooling slices) and require c = 8 x a divisor
 * of 256; deva_b200_conv2d requires cout_pad <= 2048 (<= 1024 with a rank-1 input): the layer's bias lives in shared memory. */
#define DEVA_B200_ABI_VERSION 12
#define DEVA_B200_LIST_PITCH 32 /* row pitch of top-k outputs == max supported top_k */
#define DEVA_B200_MAX_GROUPS 256 /* objects per deva_b200_readout call */

typedef void* deva_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define DEVA_B200_API __attribute__((visibility("default")))
#else
#define DEVA_B200_API
#endif

DEVA_B200_API int deva_b200_abi_version(void);
DEVA_B200_API const char* deva_b200_last_error(void);
/* Number of kernels this library has launched in the calling process (bench.py reports it). */
DEVA_B200_API uint64_t deva_b200_launch_count(void);
/* 0 when the current CUDA device can run the sm_100a kernels. */
DEVA_B200_API int deva_b200_device_check(void);

/* ---- query side ------------------------------------------------------------------------------------
 * Packs the per-frame query operand of get_similarity (deva/model/memory_utils.py:24-32):
 * row q = [ -qe[:,q] | 2*qk[:,q]*qe[:,q] ] split into fp16 (hi, lo), and bsq[q] = sum_c qe*qk^2.
 * Element (c, q) of qk/qe is read at c*stride_c + q*stride_q (channel-major [CK,Q]: stride_c=Q, stride_q=1).
 * q_hi/q_lo: [q, 2*ck] fp16;  bsq: [q] fp32.  ck in {32, 64}. */
DEVA_B200_API int deva_b200_pack_query(const float* qk, const float* qe, int64_t stride_c, int64_t stride_q, int ck, int q,
                         void* q_hi, void* q_lo, float* bsq, deva_stream_t stream);

/* ---- bank append -----------------------------------------------------------------------------------
 * Replaces the torch.cat growth of KeyValueMemoryStore.add (deva/inference/kv_memory_store.py:97-116):
 * writes `n` new tokens at the destination pointers (already offset to the first new slot).
 * key/selection element (c, t) at c*stride_c + t*stride_t; shrinkage [n].  selection/raw_sel may be NULL.
 * k_hi/k_lo: [n, 2*ck] fp16 rows [ s*k^2 | s*k ], s = shrinkage/sqrt(ck);  neg_s: [n] = -s;
 * raw_key/raw_sel: [n, ck] fp32 token-major copies;  raw_shr: [n]. */
DEVA_B200_API int deva_b200_pack_keys(const float* key, const float* selection, int64_t stride_c, int64_t stride_t,
                        const float* shrinkage, int ck, int n, void* k_hi, void* k_lo, float* neg_s, float* raw_key,
                        float* raw_sel, float* raw_shr, deva_stream_t stream);
/* Value rows fp32 src[r, j] (ld_src) -> fp16 dst[r, j] (ld_dst), r < rows, j < n
 * (MemoryManager.add_memory, deva/inference/memory_manager.py:199-205). */
DEVA_B200_API int deva_b200_append_values(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int rows, int n,
                            deva_stream_t stream);

/* ---- memory read -----------------------------------------------------------------------------------
 * get_similarity + do_softmax(top_k, inplace, return_usage) (deva/model/memory_utils.py:6-76) and the
 * usage bookkeeping of MemoryManager.match_memory / update_bucket_usage
 * (deva/inference/memory_manager.py:115-150, kv_memory_store.py:118-125), fused.
 *   workspace: deva_b200_simtopk_workspace_bytes(q) bytes of scratch;
 *   out_idx/out_w: [q, 32] int32 / fp32, entries sorted by descending similarity, zero beyond top_k;
 *   affinity (optional): [q, ld_affinity] fp16 dense rows (zero-filled, top_k non-zeros per row) for
 *                        deva_b200_readout;
 *   use_cnt/life_cnt (optional): [n_window] fp32 counters; slots < n_long are long-term memory;
 *   count_long/count_work: which region(s) receive usage (+= affinity row sums) and life (+= 1). */
DEVA_B200_API size_t deva_b200_simtopk_workspace_bytes(int q);
DEVA_B200_API int deva_b200_sim_topk(const void* k_hi, const void* k_lo, const float* neg_s, int n_window, int n_lead,
                       const void* q_hi, const void* q_lo, const float* bsq, int q, int ck, int top_k,
                       void* workspace, int32_t* out_idx, float* out_w, void* affinity, int64_t ld_affinity,
                       float* use_cnt, float* life_cnt, int n_long, int count_long, int count_work, float* out_sim,
                       const int32_t* prev_idx, float* thr_ws, deva_stream_t stream);
/* prev_idx (optional, with thr_ws: [q] fp32 scratch): out_idx of the PREVIOUS read of the same window (same slot numbering;
 * may alias out_idx).  Temporal warm start: the similarities of those top_k slots to the current queries bound every
 * query's k-th best from below, so the streaming top-k inserts only the few candidates above that bound - the result
 * is unchanged (exact), the epilogue work drops several-fold.  Pass NULL after any compaction / re-numbering. */
/* out_sim (optional): fp32 [q, 32] raw similarities of the selected slots (descending; -inf beyond top_k) - what a
 * bank-sharded read exchanges between ranks.
 *
 * deva_b200_merge_lists: global top-k + softmax over n_lists (<= 16) candidate lists per query, layout
 * part_val/part_idx [n_lists][32][q_pitch] (query index fastest; idx < 0 = empty entry).  It is the cross-rank merge of a
 * memory bank sharded along the slot axis (SURVEY section 8e): every rank all-gathers the (similarity, global slot) lists
 * of all ranks and obtains the identical global top-k set and softmax weights. */
DEVA_B200_API int deva_b200_merge_lists(const float* part_val, const int32_t* part_idx, int n_lists, int top_k, int q,
                                        int q_pitch, int32_t* out_idx, float* out_w, float* out_sim,
                                        deva_stream_t stream);
/* get_similarity + do_softmax without top-k (max-subtracted branch, memory_utils.py:66-71) as used by
 * MemoryManager.consolidation (memory_manager.py:262-273).  sim_ws: [q, ld_sim] fp32 scratch;
 * affinity: [q, ld_affinity] fp16;  shr_out[q] = sum_n affinity[q,n]*shrinkage[n] (optional). */
DEVA_B200_API int deva_b200_sim_dense_softmax(const void* k_hi, const void* k_lo, const float* neg_s, const float* shrinkage,
                                int n_window, int n_lead, const void* q_hi, const void* q_lo, const float* bsq,
                                int q, int ck, float* sim_ws, int64_t ld_sim, void* affinity, int64_t ld_affinity,
                                float* shr_out, deva_stream_t stream);
/* MemoryManager._readout (deva/inference/memory_manager.py:64-75):
 * out[out_row[g] + r, j] = sum_n values[val_row[g] + r, n] * affinity[j, n]
 * for g < n_groups, r < rows_per_group (multiple of 128), j < q, n < n_window.
 * values: fp16 [values_rows, values_ld] already offset to the window start; val_row/out_row: HOST int32 arrays. */
DEVA_B200_API int deva_b200_readout(const void* values, int64_t values_ld, int64_t values_rows, const int32_t* val_row,
                      const int32_t* out_row, int n_groups, int rows_per_group, const void* affinity,
                      int64_t ld_affinity, int n_window, int q, float* out, int64_t ld_out, void* out_tok, deva_stream_t stream);
/* out_tok (optional; when non-NULL it replaces `out`): fp16 token-major result
 * out_tok[(object*q + j)*rows_per_group + r] with object = out_row[g] / rows_per_group - the layout the NHWC
 * decoder kernels consume. */

/* Same read-out with the affinity operand generated on chip: instead of a dense [q, n_window] fp16 matrix the
 * kernel takes the top-k lists written by deva_b200_sim_topk (idx/w: [q, 32]) and builds each 256-query x 64-slot
 * affinity tile in shared memory (zeroed stage buffers + scatter of the ~top_k*256*64/n_window non-zeros), so the
 * dense affinity never exists in HBM and only the value operand streams through TMA.
 * workspace: deva_b200_readout_sparse_workspace_bytes(q, n_window) bytes (per-tile bucket offsets + entries). */
DEVA_B200_API size_t deva_b200_readout_sparse_workspace_bytes(int q, int n_window);
DEVA_B200_API int deva_b200_readout_sparse(const void* values, int64_t values_ld, int64_t values_rows,
                                           const int32_t* val_row, const int32_t* out_row, int n_groups,
                                           int rows_per_group, const int32_t* idx, const float* w, int top_k,
                                           int n_window, int q, void* workspace, float* out, int64_t ld_out,
                                           void* out_tok, deva_stream_t stream);
/* Bank-sharded read (one video, slots split over the ranks of an NVLink box; SURVEY 8e): readout GEMM fused with the
 * reduce-scatter by object.  Each rank multiplies ITS slots; the tile of group g is added (red.add.f32, system scope)
 * straight from the GEMM epilogue into rank_dst[owner[g]] + out_row[g] * ld_out, the fp32 [objects_owned * cv, q]
 * buffer of the rank that owns object g - peer memory mapped through CUDA IPC, or local.  rank_dst: HOST array of
 * n_ranks (<= 8) device pointers.  The caller zeroes the buffers beforehand and fences the ranks afterwards. */
DEVA_B200_API int deva_b200_readout_sparse_scatter(const void* values, int64_t values_ld, int64_t values_rows,
                                                   const int32_t* val_row, const int32_t* out_row,
                                                   const int32_t* owner, int n_groups, int rows_per_group,
                                                   const int32_t* idx, const float* w, int top_k, int n_window, int q,
                                                   void* workspace, float* const* rank_dst, int n_ranks,
                                                   int64_t ld_out, deva_stream_t stream);
/* Let kernels launched on `device` dereference memory of `peer_device` (cudaDeviceEnablePeerAccess; already-enabled
 * is not an error).  Needed once per peer before deva_b200_readout_sparse_scatter is given IPC-mapped pointers. */
DEVA_B200_API int deva_b200_enable_peer_access(int device, int peer_device);
/* Peer-visible buffers for the scatter read-out.  peer_alloc: cudaMalloc (zeroed) on `device` + its 64-byte CUDA IPC
 * handle, to be sent to the other ranks; peer_open: map a peer's handle INTO `device`'s address space
 * (cudaIpcOpenMemHandle with lazy peer access - an IPC mapping opened under the exporter's device is not reachable
 * from other devices); peer_close / peer_free undo them. */
DEVA_B200_API int deva_b200_peer_alloc(int device, int64_t bytes, void** ptr, uint8_t handle[64]);
DEVA_B200_API int deva_b200_peer_open(int device, const uint8_t handle[64], void** ptr);
DEVA_B200_API int deva_b200_peer_close(int device, void* ptr);
DEVA_B200_API int deva_b200_peer_free(int device, void* ptr);

/* ---- bank compaction (sieve_by_range / remove_obsolete_features, kv_memory_store.py:127-185) ----------
 * dst must not alias src.  idx: device int32 [n]. */
DEVA_B200_API int deva_b200_gather_rows(void* dst, const void* src, const int32_t* idx, int n, int row_bytes, deva_stream_t stream);
DEVA_B200_API int deva_b200_gather_f32(float* dst, const float* src, const int32_t* idx, int n, deva_stream_t stream);
DEVA_B200_API int deva_b200_gather_cols_f16(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const int32_t* idx,
                              int rows, int n, deva_stream_t stream);
/* usage[i] = use_cnt[i] / life_cnt[i]  (KeyValueMemoryStore.get_usage, kv_memory_store.py:187-193) */
DEVA_B200_API int deva_b200_usage(float* out, const float* use_cnt, const float* life_cnt, int n, deva_stream_t stream);

/* ==== network path: NHWC fp16 implicit-GEMM convolution + helper kernels ===================================
 * Activations are fp16 NHWC [batch, h, w, c] with c a multiple of 64 (8 for the helpers); weights are packed
 * fp16 [cout_pad, kh*kw*cin_pad] (filter tap major, input channel minor), bias fp32 [cout_pad] with the
 * eval-mode BatchNorm already folded in. */
typedef struct deva_b200_conv_desc {
  const void* x;        /* fp16 NHWC input [batch, h, w, cin_pad] */
  const void* x2;       /* optional second input of the same shape: the convolution sees cat[x, x2] along channels
                         * (weights packed [cout_pad, 2, kh*kw, cin_pad]); stride 1 only */
  const void* x_lo;     /* optional fp16 low-order part of x (x_true = x + x_lo): split-precision mode
                         * D = Xh.Wh + Xl.Wh + Xh.Wl with weights packed [cout_pad, 2 (hi, lo), kh*kw, cin_pad];
                         * ~fp32 accuracy at 3x the MMA work.  Exclusive with x2. */
  int32_t split_mode;   /* 0: as described above (x_lo => three passes);  1: x_lo with SINGLE fp16 weights,
                         * D = Xh.W + Xl.W (removes the activation-operand rounding, 2x the MMA work);  2: no x_lo,
                         * weights packed (hi, lo) as for mode 0, D = X.Wh + X.Wl (removes the weight rounding) */
  int32_t batch, h, w, cin_pad;
  const void* w_packed; /* fp16 [cout_pad, kh*kw*cin_pad] */
  int32_t kh, kw, stride; /* 1x1 or 3x3, stride 1 or 2, padding kh/2 (nn.Conv2d semantics) */
  int32_t cout, cout_pad, nt; /* real / padded output channels, channel tile (multiple of 32, <= 256, divides cout_pad) */
  int32_t th, tw;       /* spatial tile of the implicit GEMM, th*tw == 128 */
  const float* bias;
  const void* res;      /* optional fp16 NHWC residual added before the activation (shape of the output) */
  const void* res_lo;   /* optional low-order part of the residual */
  int32_t res_broadcast; /* 1: `res` is ONE image broadcast over the batch */
  const float* rank1_w; /* optional fp32 [cout_pad]: weight of an extra 1-channel input ... */
  const float* rank1_x; /* ... whose fp32 plane is [batch, ho*wo]  (out += rank1_w[c] * rank1_x[b, pixel]) */
  void* out_raw;        /* optional fp16 NHWC output */
  void* out_relu;       /* optional fp16 NHWC output, ReLU applied */
  float* out_f32;       /* optional fp32 NHWC output */
  void* out_raw_lo;     /* optional fp16 remainders (value - fp16(value)) of out_raw / out_relu */
  void* out_relu_lo;
  const float* head_w;  /* optional fused 1x1 head on the ReLU'd fp32 result (needs cout_pad == nt): fp32 [head_n, cout] */
  float* head_out;      /* fp32 [batch*ho*wo, head_n]: head_out[p, t] = sum_c relu(out[p, c]) * head_w[t, c] */
  int32_t head_n;       /* <= 9.  Folds MaskDecoder.pred (big_modules.py:189-190) into the last decoder conv. */
  /* optional fused gate epilogue (SensoryUpdater / SensoryDeepUpdater, modules.py:145-149,163-167): the conv output is
   * never written; with C = cout/3 hidden channels the channel tile (nt must be 192) holds [forget | update | new] x 64
   * for hidden channels 64*tile .. +63 (weight rows / bias packed in that order) and the epilogue writes
   * gate_out = sigmoid(f) * gate_h * (1 - sigmoid(u)) + sigmoid(u) * tanh(n), evaluated on the fp32 accumulators. */
  const void* gate_h;   /* fp16 NHWC [batch, ho, wo, cout/3] previous hidden state */
  void* gate_out;       /* fp16 NHWC [batch, ho, wo, cout/3] new hidden state */
  /* split_mode 3: the low-order activation pass on the fp8 tensor-core path (half the cost of split_mode 1):
   * D = (X . W16 + Xlo8 . W8) * acc_scale, W16 = fp16(W * 2^S) in w_packed, W8 = e4m3(W * 2^(S-12)) in w8_packed,
   * Xlo8 = e4m3((x - fp16(x)) * 4096) in x_lo8, acc_scale = 2^-S.  Stride 1, cin_pad % 128 == 0. */
  const void* x_lo8;    /* u8 NHWC [batch, h, w, cin_pad] */
  const void* w8_packed; /* u8 [cout_pad, kh*kw*cin_pad] */
  float acc_scale;      /* 0 = 1 */
  void* out_relu_lo8;   /* optional u8 NHWC: e4m3 low-order part (x 4096) of the ReLU'd output */
  int32_t ksplit;       /* > 1: split the K loop into that many chains (fp32 output only): out_f32 then holds
                         * ceil(k_iters / ceil(k_iters / ksplit)) partial sums [part, batch, ho, wo, cout] (bias in part 0)
                         * for the consumer to add in fp32.  The tensor core's accumulator rounds toward zero at every
                         * accumulation step; short chains keep a split-precision convolution at fp32 accuracy. */
} deva_b200_conv_desc;
/* nn.Conv2d + folded BatchNorm (+ residual, + ReLU) as in deva/model/resnet.py:46-114, group_modules.py:41-67,
 * modules.py:22-39; `desc` is a HOST struct. */
DEVA_B200_API int deva_b200_conv2d(const deva_b200_conv_desc* desc, deva_stream_t stream);
/* im2col of the 7x7 stride-2 pad-3 stems (resnet.py:120): src fp32 planes [b, c, h, w] -> fp16 [b, h/2, w/2, k_pad],
 * column (kh*7+kw)*c + ch, zero padded to k_pad (multiple of 64).  The stem then runs through deva_b200_conv2d as a
 * 1x1 convolution over k_pad channels.  dst_lo (optional) receives the fp16 remainders for split precision. */
DEVA_B200_API int deva_b200_stem_im2col(const float* src, void* dst, void* dst_lo, int b, int c, int h, int w, int k_pad,
                                        deva_stream_t stream);
DEVA_B200_API int deva_b200_nchw_to_nhwc(const float* src, void* dst, int b, int c, int h, int w, int c_pad,
                                         deva_stream_t stream);
DEVA_B200_API int deva_b200_nhwc_to_nchw(const void* src, float* dst, int b, int c, int h, int w, deva_stream_t stream);
/* 3x3 stride-2 max pool (resnet.py:123); x_lo / y_lo: optional low-order parts (pooling acts on x + x_lo) */
DEVA_B200_API int deva_b200_maxpool(const void* x, const void* x_lo, void* y, void* y_lo, int b, int h, int w, int c,
                                    deva_stream_t stream);
/* bilinear x2 (align_corners=False) + broadcast skip add -> raw and/or ReLU'd (modules.py:88-91) */
DEVA_B200_API int deva_b200_up2_add(const void* g, const void* skip, void* raw, void* relu, int b, int h, int w, int c,
                                    deva_stream_t stream);
/* F.interpolate(mode='area') by an integer ratio r (group_modules.py:33-38), fp16 NHWC and fp32 planes */
DEVA_B200_API int deva_b200_area_down(const void* x, void* y, int b, int h, int w, int c, int r, deva_stream_t stream);
DEVA_B200_API int deva_b200_area_down_plane(const float* x, float* y, int b, int h, int w, int r, deva_stream_t stream);
/* x + CBAM(x) (cbam.py:21-77 inside group_modules.py:146-150); scratch: fp32 [129*b*c + 2*b*h*w] (2 x 64 pooling slices + the gate, then the per-pixel statistics); c = 8 x a divisor of 256 */
DEVA_B200_API int deva_b200_cbam(const void* x, const float* w1, const float* b1, const float* w2, const float* b2,
                                 const float* ws, const float* bs, float* scratch, void* raw, void* relu, int b, int h,
                                 int w, int c, int r, deva_stream_t stream);
/* Split-precision twins for a residual stream carried as fp16 (hi, lo) pairs (the default "parity" precision plan): the
 * input is g + g_lo (x + x_lo) [+ skip_lo, optional], the raw result is written as (raw, raw_lo) (both NULL = not
 * wanted), the ReLU'd copy (an MMA operand) as hi, plus its remainder relu_lo when the consumer runs a second
 * activation pass (conv split_mode 1). */
DEVA_B200_API int deva_b200_up2_add_split(const void* g, const void* g_lo, const void* skip, const void* skip_lo,
                                          void* raw, void* raw_lo, void* relu, void* relu_lo, void* relu_lo8, int b, int h,
                                          int w, int c, deva_stream_t stream);
/* relu_lo8 (instead of relu_lo): u8 NHWC, e4m3 of (relu - fp16(relu)) * 4096 - the low-order operand of a conv with
 * split_mode 3. */
DEVA_B200_API int deva_b200_cbam_split(const void* x, const void* x_lo, const float* w1, const float* b1, const float* w2,
                                       const float* b2, const float* ws, const float* bs, float* scratch, void* raw,
                                       void* raw_lo, void* relu, void* relu_lo, int pool_lo, int b, int h, int w, int c,
                                       int r, deva_stream_t stream);
/* pool_lo: 1 = the gate statistics (channel pooling, per-pixel max / mean) are taken over x + x_lo, 0 = over x only. */
/* sensory GRU gates (modules.py:145-149): values fp16 [pixels, 3c], h fp16 [pixels, c] -> out fp16 */
DEVA_B200_API int deva_b200_gru(const void* values, const void* h, void* out, int64_t pixels, int c,
                                deva_stream_t stream);
/* Finish of a split-K convolution (deva_b200_conv2d with ksplit > 1): out = sum of the n_parts fp32 partial sums
 * (part_stride elements apart, bias in part 0) + optional fp16 residual (res + res_lo), written as fp16 raw / ReLU'd
 * tensors, each optionally as a (hi, lo) pair.  n = elements per part (multiple of 8). */
DEVA_B200_API int deva_b200_sum_parts(const float* parts, int n_parts, int64_t part_stride, const void* res,
                                      const void* res_lo, void* raw, void* raw_lo, void* relu, void* relu_lo, int64_t n,
                                      deva_stream_t stream);
/* key projection tail (modules.py:73-78): y fp32 [q, ld] = [key | d | e], given as n_parts partial sums part_stride
 * elements apart (deva_b200_conv2d's ksplit) -> key [q,ck], shrinkage [q] = d^2 + 1, selection [q,ck] = sigmoid(e) */
DEVA_B200_API int deva_b200_key_tail(const float* y, int ld, int q, int ck, int n_parts, int64_t part_stride, float* key,
                                     float* shrinkage, float* selection, deva_stream_t stream);
/* sigmoid -> aggregate -> bilinear x4 -> softmax (network.py:33-40,144-168): logits fp32 [k,h,w] ->
 * prob fp32 [(k+1),4h,4w] (and optionally the up-sampled logits); agg: fp32 scratch [(k+1),h,w] */
DEVA_B200_API int deva_b200_output_tail(const float* logits, float* agg, float* prob, float* logits_out, int k, int h,
                                        int w, deva_stream_t stream);
/* logits[b,y,x] = bias + sum_{dy,dx} z[b, y+dy, x+dx, (dy+1)*3+(dx+1)]: the 3x3 gather completing the fused head
 * (z fp32 [b,h,w,9] from deva_b200_conv2d's head_out) == nn.Conv2d(256, 1, 3, padding=1) on relu(p4) */
DEVA_B200_API int deva_b200_head_gather3x3(const float* z, float* out, float bias, int b, int h, int w,
                                           deva_stream_t stream);
/* fp16 token-major values [n, c] -> bank rows dst[c, j] (ld_dst): append from the NHWC value encoder */
DEVA_B200_API int deva_b200_transpose_append(const void* src, void* dst, int64_t ld_dst, int n, int c,
                                             deva_stream_t stream);

/* ---- frame ingest / egress (SURVEY 8f-3) ------------------------------------------------------------------------ */
/* Decoded frame u8 [h, w, 3] (RGB interleaved) -> fp32 [3, h, w], (x / 255 - mean[c]) / std[c]: torchvision's
 * ToTensor + Normalize (deva/inference/data/video_reader.py:146-150) after the upload instead of before it (4x fewer
 * PCIe bytes).  Bit-exact with the torch ops (IEEE divisions in the same order). */
DEVA_B200_API int deva_b200_ingest_rgb8(const uint8_t* src, float* dst, int h, int w, const float mean[3],
                                        const float std[3], deva_stream_t stream);
/* Driver post-step (evaluation/eval_vos.py:169-181) in one pass: optional bilinear resize (align_corners=False) of
 * prob fp32 [c, h, w] to [out_h, out_w], optional horizontal flip, argmax over channels (first maximum wins),
 * temporary-id -> object-id remap through lut int32 [c] (lut[0] = 0).  Writes out_u8 [out_h, out_w] and/or
 * out_i64 [out_h, out_w] (either may be NULL). */
DEVA_B200_API int deva_b200_prob_to_ids(const float* prob, int c, int h, int w, int out_h, int out_w, int flip,
                                        const int32_t* lut, uint8_t* out_u8, int64_t* out_i64, deva_stream_t stream);

/* Frame u8 [h, w, 3] (RGB interleaved) -> fp32 [3, out_h, out_w]: ToTensor + Normalize per source pixel as in
 * deva_b200_ingest_rgb8, then a resize to the evaluation size.
 *  - DEVA_B200_RESIZE_READER: torchvision Resize(bilinear, antialias=True) after the normalisation
 *    (deva/inference/data/video_reader.py:141-145): separable triangle filter, rows first into the fp32 workspace
 *    `ws` [3, h, out_w], then columns; the tap weights are bit-identical to torch's float32 CPU ones.
 *  - DEVA_B200_RESIZE_DEMO: F.interpolate(bilinear, align_corners=False) (deva/inference/demo_utils.py:10-19);
 *    `ws` is unused and may be NULL.
 * The caller picks out_h / out_w (torchvision's Resize(size) rule for the reader, int(h * size / min(h, w)) for the
 * demo) and, for the reader, skips the call when they equal h / w: torchvision returns such an image unresized. */
#define DEVA_B200_RESIZE_READER 0
#define DEVA_B200_RESIZE_DEMO 1
DEVA_B200_API size_t deva_b200_resize_rgb8_workspace_bytes(int h, int w, int out_h, int out_w, int mode);
DEVA_B200_API int deva_b200_resize_rgb8(const uint8_t* src, float* dst, float* ws, int h, int w, int out_h, int out_w,
                                        int mode, const float mean[3], const float std[3], deva_stream_t stream);
/* HOST: the antialiased tap tables deva_b200_resize_rgb8 computes on the fly for one axis n_in -> n_out: output i
 * reads x0[i] .. x0[i] + n[i] - 1 with weights w[i * max_taps + j] (zero past n[i]).  Fails when max_taps is below
 * 2 * ceil(max(n_in / n_out, 1)) + 1.  Needs no GPU. */
DEVA_B200_API int deva_b200_resize_aa_weights(int n_in, int n_out, int max_taps, int32_t* x0, int32_t* n, float* w);
/* Palette mask u8 [h, w] -> int64 [out_h, out_w], dst[y, x] = src[src_y[y], src_x[x]] (0 where either index is
 * negative).  With Pillow's NEAREST tables (INTEGRATION.md) this is transforms.Resize(size, NEAREST) on the 'P' image
 * followed by torch.LongTensor (video_reader.py:147-150, 211-214), bit for bit.  src_y int32 [out_h], src_x int32
 * [out_w]. */
DEVA_B200_API int deva_b200_resize_labels(const uint8_t* src, int64_t* dst, int h, int w, int out_h, int out_w,
                                          const int32_t* src_y, const int32_t* src_x, deva_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DEVA_B200_H_ */
