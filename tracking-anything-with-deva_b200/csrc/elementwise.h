#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

namespace b200 {
int ew_nchw_to_nhwc(const float* src, __half* dst, int B, int C, int H, int W, int Cp, cudaStream_t s);
int ew_nhwc_to_nchw(const __half* src, float* dst, int B, int C, int H, int W, cudaStream_t s);
int ew_stem_im2col(const float* src, __half* dst, __half* dst_lo, int B, int C, int H, int W, int Kp, cudaStream_t s);
int ew_maxpool(const __half* x, const __half* x_lo, __half* y, __half* y_lo, int B, int H, int W, int C, cudaStream_t s);
int ew_up2_add(const __half* g, const __half* skip, __half* raw, __half* relu, int B, int h, int w, int C, cudaStream_t s);
int ew_up2_add_split(const __half* g, const __half* g_lo, const __half* skip, const __half* skip_lo, __half* raw,
                     __half* raw_lo, __half* relu, __half* relu_lo, unsigned char* relu_lo8, int B, int h, int w, int C,
                     cudaStream_t s);
int ew_cbam_split(const __half* x, const __half* x_lo, const float* w1, const float* b1, const float* w2, const float* b2,
                  const float* ws, const float* bs, float* scratch, __half* raw, __half* raw_lo, __half* relu, __half* relu_lo,
                  int pool_lo, int B, int H, int W, int C, int R, cudaStream_t s);
int ew_area_down(const __half* x, __half* y, int B, int H, int W, int C, int r, cudaStream_t s);
int ew_area_down_plane(const float* x, float* y, int B, int H, int W, int r, cudaStream_t s);
int ew_cbam(const __half* x, const float* w1, const float* b1, const float* w2, const float* b2, const float* ws,
            const float* bs, float* scratch, __half* raw, __half* relu, int B, int H, int W, int C, int R,
            cudaStream_t s);
int ew_gru(const __half* values, const __half* h, __half* out, long long pixels, int C, cudaStream_t s);
int ew_sum_parts(const float* parts, int n_parts, long long part_stride, const __half* res, const __half* res_lo,
                 __half* raw, __half* raw_lo, __half* relu, __half* relu_lo, long long n, cudaStream_t s);
int ew_key_tail(const float* y, int ld, int Q, int CK, int n_parts, long long part_stride, float* key, float* shr,
                float* sel, cudaStream_t s);
int ew_output_tail(const float* logits, float* agg, float* prob, float* logits_out, int K, int h, int w, cudaStream_t s);
int ew_head_gather3x3(const float* z, float* out, float bias, int B, int H, int W, cudaStream_t s);
int ew_transpose_append(const __half* src, __half* dst, long long ld_dst, int n, int C, cudaStream_t s);
int ew_ingest_rgb8(const unsigned char* src, float* dst, int h, int w, const float* mean, const float* stdv, cudaStream_t s);
int ew_prob_to_ids(const float* prob, int c, int h, int w, int out_h, int out_w, int flip, const int* lut,
                   unsigned char* out_u8, long long* out_i64, cudaStream_t s);
enum { RESIZE_READER = 0, RESIZE_DEMO = 1 };  // == DEVA_B200_RESIZE_READER / _DEMO
size_t ew_resize_rgb8_workspace_bytes(int h, int out_w, int mode);
int ew_resize_rgb8(const unsigned char* src, float* dst, float* ws, int h, int w, int out_h, int out_w, int mode,
                   const float* mean, const float* stdv, cudaStream_t s);
int ew_resize_aa_weights(int n_in, int n_out, int max_taps, int* x0, int* n, float* wt);
int ew_resize_labels(const unsigned char* src, long long* dst, int h, int w, int out_h, int out_w, const int* src_y,
                     const int* src_x, cudaStream_t s);
}  // namespace b200
