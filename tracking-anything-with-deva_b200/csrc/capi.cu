// extern "C" surface of libdeva_b200.so; declarations and reference citations live in include/deva_b200.h.
#include "../../include/deva_b200.h"

#include <cuda_fp16.h>

#include "bank_ops.h"
#include <string.h>

#include "common.h"
#include "conv.h"
#include "elementwise.h"
#include "readout.h"
#include "simtopk.h"

namespace b200 { const char* last_error(); unsigned long long launch_count(); }
using namespace b200;

static inline cudaStream_t S(deva_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline __half* H(void* p) { return reinterpret_cast<__half*>(p); }
static inline const __half* H(const void* p) { return reinterpret_cast<const __half*>(p); }

extern "C" {

DEVA_B200_API int deva_b200_abi_version(void) { return DEVA_B200_ABI_VERSION; }
DEVA_B200_API const char* deva_b200_last_error(void) { return last_error(); }
DEVA_B200_API uint64_t deva_b200_launch_count(void) { return launch_count(); }

DEVA_B200_API int deva_b200_device_check(void) {
  int dev = 0, major = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  B200_REQUIRE(major == 10, "deva_b200 kernels are built for sm_100a; device has compute capability major %d", major);
  return 0;
}

DEVA_B200_API int deva_b200_pack_query(const float* qk, const float* qe, int64_t stride_c, int64_t stride_q, int ck, int q,
                         void* q_hi, void* q_lo, float* bsq, deva_stream_t stream) {
  return launch_pack_query(qk, qe, stride_c, stride_q, ck, q, H(q_hi), H(q_lo), bsq, S(stream));
}
DEVA_B200_API int deva_b200_pack_keys(const float* key, const float* selection, int64_t stride_c, int64_t stride_t,
                        const float* shrinkage, int ck, int n, void* k_hi, void* k_lo, float* neg_s, float* raw_key,
                        float* raw_sel, float* raw_shr, deva_stream_t stream) {
  return launch_pack_keys(key, selection, stride_c, stride_t, shrinkage, ck, n, H(k_hi), H(k_lo), neg_s, raw_key,
                          raw_sel, raw_shr, S(stream));
}
DEVA_B200_API int deva_b200_append_values(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int rows, int n,
                            deva_stream_t stream) {
  return launch_append_values(src, ld_src, H(dst), ld_dst, rows, n, S(stream));
}
DEVA_B200_API size_t deva_b200_simtopk_workspace_bytes(int q) { return simtopk_workspace_bytes(q); }
DEVA_B200_API int deva_b200_sim_topk(const void* k_hi, const void* k_lo, const float* neg_s, int n_window, int n_lead,
                       const void* q_hi, const void* q_lo, const float* bsq, int q, int ck, int top_k,
                       void* workspace, int32_t* out_idx, float* out_w, void* affinity, int64_t ld_affinity,
                       float* use_cnt, float* life_cnt, int n_long, int count_long, int count_work, float* out_sim,
                       const int32_t* prev_idx, float* thr_ws, deva_stream_t stream) {
  return launch_sim_topk(H(k_hi), H(k_lo), neg_s, n_window, n_lead, H(q_hi), H(q_lo), bsq, q, ck, top_k, workspace,
                         out_idx, out_w, H(affinity), ld_affinity, use_cnt, life_cnt, n_long, count_long, count_work,
                         out_sim, prev_idx, thr_ws, S(stream));
}
DEVA_B200_API int deva_b200_merge_lists(const float* part_val, const int32_t* part_idx, int n_lists, int top_k, int q,
                                        int q_pitch, int32_t* out_idx, float* out_w, float* out_sim,
                                        deva_stream_t stream) {
  return launch_merge_lists(part_val, part_idx, n_lists, top_k, q, q_pitch, out_idx, out_w, out_sim, S(stream));
}
DEVA_B200_API int deva_b200_sim_dense_softmax(const void* k_hi, const void* k_lo, const float* neg_s, const float* shrinkage,
                                int n_window, int n_lead, const void* q_hi, const void* q_lo, const float* bsq,
                                int q, int ck, float* sim_ws, int64_t ld_sim, void* affinity, int64_t ld_affinity,
                                float* shr_out, deva_stream_t stream) {
  return launch_sim_dense_softmax(H(k_hi), H(k_lo), neg_s, shrinkage, n_window, n_lead, H(q_hi), H(q_lo), bsq, q, ck,
                                  sim_ws, ld_sim, H(affinity), ld_affinity, shr_out, S(stream));
}
DEVA_B200_API int deva_b200_readout(const void* values, int64_t values_ld, int64_t values_rows, const int32_t* val_row,
                      const int32_t* out_row, int n_groups, int rows_per_group, const void* affinity,
                      int64_t ld_affinity, int n_window, int q, float* out, int64_t ld_out, void* out_tok,
                      deva_stream_t stream) {
  return launch_readout(H(values), values_ld, values_rows, val_row, out_row, n_groups, rows_per_group, H(affinity),
                        ld_affinity, n_window, q, out, ld_out, H(out_tok), S(stream));
}
DEVA_B200_API size_t deva_b200_readout_sparse_workspace_bytes(int q, int n_window) {
  return readout_sparse_workspace_bytes(q, n_window);
}
DEVA_B200_API int deva_b200_readout_sparse(const void* values, int64_t values_ld, int64_t values_rows,
                                           const int32_t* val_row, const int32_t* out_row, int n_groups,
                                           int rows_per_group, const int32_t* idx, const float* w, int top_k,
                                           int n_window, int q, void* workspace, float* out, int64_t ld_out,
                                           void* out_tok, deva_stream_t stream) {
  return launch_readout_sparse(H(values), values_ld, values_rows, val_row, out_row, n_groups, rows_per_group, idx, w,
                               top_k, n_window, q, workspace, out, ld_out, H(out_tok), S(stream));
}
DEVA_B200_API int deva_b200_readout_sparse_scatter(const void* values, int64_t values_ld, int64_t values_rows,
                                                   const int32_t* val_row, const int32_t* out_row,
                                                   const int32_t* owner, int n_groups, int rows_per_group,
                                                   const int32_t* idx, const float* w, int top_k, int n_window, int q,
                                                   void* workspace, float* const* rank_dst, int n_ranks,
                                                   int64_t ld_out, deva_stream_t stream) {
  return launch_readout_sparse(H(values), values_ld, values_rows, val_row, out_row, n_groups, rows_per_group, idx, w,
                               top_k, n_window, q, workspace, nullptr, ld_out, nullptr, S(stream), owner, rank_dst, n_ranks);
}
DEVA_B200_API int deva_b200_enable_peer_access(int device, int peer_device) {
  int prev = 0, can = 0;
  B200_CUDA(cudaGetDevice(&prev));
  B200_CUDA(cudaDeviceCanAccessPeer(&can, device, peer_device));
  B200_REQUIRE(can, "device %d has no peer-to-peer path to device %d", device, peer_device);
  B200_CUDA(cudaSetDevice(device));
  cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { (void)cudaGetLastError(); e = cudaSuccess; }
  (void)cudaSetDevice(prev);
  B200_CUDA(e);
  return 0;
}
namespace {
struct DeviceScope {
  int prev = 0;
  explicit DeviceScope(int d) { cudaGetDevice(&prev); cudaSetDevice(d); }
  ~DeviceScope() { cudaSetDevice(prev); }
};
}  // namespace
DEVA_B200_API int deva_b200_peer_alloc(int device, int64_t bytes, void** ptr, uint8_t handle[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  B200_REQUIRE(bytes > 0 && ptr && handle, "peer_alloc: bad arguments");
  DeviceScope scope(device);
  B200_CUDA(cudaMalloc(ptr, (size_t)bytes));
  B200_CUDA(cudaMemset(*ptr, 0, (size_t)bytes));
  cudaIpcMemHandle_t h;
  B200_CUDA(cudaIpcGetMemHandle(&h, *ptr));
  memcpy(handle, &h, 64);
  return 0;
}
DEVA_B200_API int deva_b200_peer_open(int device, const uint8_t handle[64], void** ptr) {
  B200_REQUIRE(ptr && handle, "peer_open: bad arguments");
  DeviceScope scope(device);
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  B200_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}
DEVA_B200_API int deva_b200_peer_close(int device, void* ptr) {
  DeviceScope scope(device);
  B200_CUDA(cudaIpcCloseMemHandle(ptr));
  return 0;
}
DEVA_B200_API int deva_b200_peer_free(int device, void* ptr) {
  DeviceScope scope(device);
  B200_CUDA(cudaFree(ptr));
  return 0;
}
DEVA_B200_API int deva_b200_gather_rows(void* dst, const void* src, const int32_t* idx, int n, int row_bytes, deva_stream_t stream) {
  return launch_gather_rows(dst, src, idx, n, row_bytes, S(stream));
}
DEVA_B200_API int deva_b200_gather_f32(float* dst, const float* src, const int32_t* idx, int n, deva_stream_t stream) {
  return launch_gather_f32(dst, src, idx, n, S(stream));
}
DEVA_B200_API int deva_b200_gather_cols_f16(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const int32_t* idx,
                              int rows, int n, deva_stream_t stream) {
  return launch_gather_cols_f16(H(dst), ld_dst, H(src), ld_src, idx, rows, n, S(stream));
}
DEVA_B200_API int deva_b200_usage(float* out, const float* use_cnt, const float* life_cnt, int n, deva_stream_t stream) {
  return launch_usage(out, use_cnt, life_cnt, n, S(stream));
}

DEVA_B200_API int deva_b200_conv2d(const deva_b200_conv_desc* c, deva_stream_t stream) {
  ConvDesc d;
  d.x = c->x; d.x2 = c->x2; d.x_lo = c->x_lo; d.split_mode = c->split_mode; d.batch = c->batch; d.h = c->h; d.w = c->w; d.cin_pad = c->cin_pad;
  d.w_packed = c->w_packed; d.kh = c->kh; d.kw = c->kw; d.stride = c->stride;
  d.cout = c->cout; d.cout_pad = c->cout_pad; d.nt = c->nt; d.th = c->th; d.tw = c->tw;
  d.bias = c->bias; d.res = c->res; d.res_lo = c->res_lo; d.res_broadcast = c->res_broadcast;
  d.rank1_w = c->rank1_w; d.rank1_x = c->rank1_x;
  d.out_raw = c->out_raw; d.out_relu = c->out_relu; d.out_f32 = c->out_f32;
  d.out_raw_lo = c->out_raw_lo; d.out_relu_lo = c->out_relu_lo;
  d.head_w = c->head_w; d.head_out = c->head_out; d.head_n = c->head_n;
  d.gate_h = c->gate_h; d.gate_out = c->gate_out; d.ksplit = c->ksplit;
  d.x_lo8 = c->x_lo8; d.w8_packed = c->w8_packed; d.acc_scale = c->acc_scale; d.out_relu_lo8 = c->out_relu_lo8;
  return launch_conv(d, S(stream));
}
DEVA_B200_API int deva_b200_stem_im2col(const float* src, void* dst, void* dst_lo, int b, int c, int h, int w, int k_pad,
                                        deva_stream_t stream) {
  return ew_stem_im2col(src, H(dst), H(dst_lo), b, c, h, w, k_pad, S(stream));
}
DEVA_B200_API int deva_b200_nchw_to_nhwc(const float* src, void* dst, int b, int c, int h, int w, int c_pad,
                                         deva_stream_t stream) {
  return ew_nchw_to_nhwc(src, H(dst), b, c, h, w, c_pad, S(stream));
}
DEVA_B200_API int deva_b200_nhwc_to_nchw(const void* src, float* dst, int b, int c, int h, int w, deva_stream_t stream) {
  return ew_nhwc_to_nchw(H(src), dst, b, c, h, w, S(stream));
}
DEVA_B200_API int deva_b200_maxpool(const void* x, const void* x_lo, void* y, void* y_lo, int b, int h, int w, int c,
                                    deva_stream_t stream) {
  return ew_maxpool(H(x), H(x_lo), H(y), H(y_lo), b, h, w, c, S(stream));
}
DEVA_B200_API int deva_b200_up2_add(const void* g, const void* skip, void* raw, void* relu, int b, int h, int w, int c,
                                    deva_stream_t stream) {
  return ew_up2_add(H(g), H(skip), H(raw), H(relu), b, h, w, c, S(stream));
}
DEVA_B200_API int deva_b200_area_down(const void* x, void* y, int b, int h, int w, int c, int r, deva_stream_t stream) {
  return ew_area_down(H(x), H(y), b, h, w, c, r, S(stream));
}
DEVA_B200_API int deva_b200_area_down_plane(const float* x, float* y, int b, int h, int w, int r, deva_stream_t stream) {
  return ew_area_down_plane(x, y, b, h, w, r, S(stream));
}
DEVA_B200_API int deva_b200_cbam(const void* x, const float* w1, const float* b1, const float* w2, const float* b2,
                                 const float* ws, const float* bs, float* scratch, void* raw, void* relu, int b, int h,
                                 int w, int c, int r, deva_stream_t stream) {
  return ew_cbam(H(x), w1, b1, w2, b2, ws, bs, scratch, H(raw), H(relu), b, h, w, c, r, S(stream));
}
DEVA_B200_API int deva_b200_up2_add_split(const void* g, const void* g_lo, const void* skip, const void* skip_lo,
                                          void* raw, void* raw_lo, void* relu, void* relu_lo, void* relu_lo8, int b, int h,
                                          int w, int c, deva_stream_t stream) {
  return ew_up2_add_split(H(g), H(g_lo), H(skip), H(skip_lo), H(raw), H(raw_lo), H(relu), H(relu_lo),
                          reinterpret_cast<unsigned char*>(relu_lo8), b, h, w, c, S(stream));
}
DEVA_B200_API int deva_b200_cbam_split(const void* x, const void* x_lo, const float* w1, const float* b1, const float* w2,
                                       const float* b2, const float* ws, const float* bs, float* scratch, void* raw,
                                       void* raw_lo, void* relu, void* relu_lo, int pool_lo, int b, int h, int w, int c,
                                       int r, deva_stream_t stream) {
  return ew_cbam_split(H(x), H(x_lo), w1, b1, w2, b2, ws, bs, scratch, H(raw), H(raw_lo), H(relu), H(relu_lo), pool_lo, b, h,
                       w, c, r, S(stream));
}
DEVA_B200_API int deva_b200_gru(const void* values, const void* h, void* out, int64_t pixels, int c,
                                deva_stream_t stream) {
  return ew_gru(H(values), H(h), H(out), pixels, c, S(stream));
}
DEVA_B200_API int deva_b200_sum_parts(const float* parts, int n_parts, int64_t part_stride, const void* res,
                                      const void* res_lo, void* raw, void* raw_lo, void* relu, void* relu_lo, int64_t n,
                                      deva_stream_t stream) {
  return ew_sum_parts(parts, n_parts, part_stride, H(res), H(res_lo), H(raw), H(raw_lo), H(relu), H(relu_lo), n, S(stream));
}
DEVA_B200_API int deva_b200_key_tail(const float* y, int ld, int q, int ck, int n_parts, int64_t part_stride, float* key,
                                     float* shrinkage, float* selection, deva_stream_t stream) {
  return ew_key_tail(y, ld, q, ck, n_parts, part_stride, key, shrinkage, selection, S(stream));
}
DEVA_B200_API int deva_b200_output_tail(const float* logits, float* agg, float* prob, float* logits_out, int k, int h,
                                        int w, deva_stream_t stream) {
  return ew_output_tail(logits, agg, prob, logits_out, k, h, w, S(stream));
}
DEVA_B200_API int deva_b200_head_gather3x3(const float* z, float* out, float bias, int b, int h, int w,
                                           deva_stream_t stream) {
  return ew_head_gather3x3(z, out, bias, b, h, w, S(stream));
}
DEVA_B200_API int deva_b200_transpose_append(const void* src, void* dst, int64_t ld_dst, int n, int c,
                                             deva_stream_t stream) {
  return ew_transpose_append(H(src), H(dst), ld_dst, n, c, S(stream));
}
DEVA_B200_API int deva_b200_ingest_rgb8(const uint8_t* src, float* dst, int h, int w, const float mean[3],
                                        const float std[3], deva_stream_t stream) {
  return ew_ingest_rgb8(src, dst, h, w, mean, std, S(stream));
}
DEVA_B200_API int deva_b200_prob_to_ids(const float* prob, int c, int h, int w, int out_h, int out_w, int flip,
                                        const int32_t* lut, uint8_t* out_u8, int64_t* out_i64, deva_stream_t stream) {
  return ew_prob_to_ids(prob, c, h, w, out_h, out_w, flip, lut, out_u8, reinterpret_cast<long long*>(out_i64), S(stream));
}
static_assert(RESIZE_READER == DEVA_B200_RESIZE_READER && RESIZE_DEMO == DEVA_B200_RESIZE_DEMO, "resize modes");
DEVA_B200_API size_t deva_b200_resize_rgb8_workspace_bytes(int h, int w, int out_h, int out_w, int mode) {
  (void)w; (void)out_h;
  return ew_resize_rgb8_workspace_bytes(h, out_w, mode);
}
DEVA_B200_API int deva_b200_resize_rgb8(const uint8_t* src, float* dst, float* ws, int h, int w, int out_h, int out_w,
                                        int mode, const float mean[3], const float std[3], deva_stream_t stream) {
  return ew_resize_rgb8(src, dst, ws, h, w, out_h, out_w, mode, mean, std, S(stream));
}
DEVA_B200_API int deva_b200_resize_aa_weights(int n_in, int n_out, int max_taps, int32_t* x0, int32_t* n, float* w) {
  return ew_resize_aa_weights(n_in, n_out, max_taps, x0, n, w);
}
DEVA_B200_API int deva_b200_resize_labels(const uint8_t* src, int64_t* dst, int h, int w, int out_h, int out_w,
                                          const int32_t* src_y, const int32_t* src_x, deva_stream_t stream) {
  return ew_resize_labels(src, reinterpret_cast<long long*>(dst), h, w, out_h, out_w, src_y, src_x, S(stream));
}

}  // extern "C"
