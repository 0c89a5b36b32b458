/*
 * lce_b200_builtins.h -- C-ABI of the float TFLite builtins the three model
 * families (QuickNet, QuickNetLarge, Bi-RealNet-18) use AROUND the binary path
 * (SURVEY 8f-1). In the reference these come from stock TFLite
 * (tensorflow/lite/kernels/internal/reference/{conv.h:27, depthwiseconv_float.h:25,
 * pooling.h:28,196, add.h, fully_connected.h:29, softmax.h:31, reduce.h}); here they
 * are plain fp32 CUDA kernels so the graph never leaves HBM between binary layers.
 * They are callers of the hot path, not part of it: no tensor cores, no tuning
 * beyond coalescing. All tensors NHWC fp32, device pointers, async on `stream`.
 */
#ifndef LCE_B200_BUILTINS_H_
#define LCE_B200_BUILTINS_H_

#include <stdint.h>

#include "lce_b200_types.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lce_f32_conv_desc {
  int32_t batch, in_h, in_w, in_c;
  int32_t filter_h, filter_w, out_c; /* filter OHWI [out_c, fh, fw, in_c] */
  int32_t stride_h, stride_w, dilation_h, dilation_w;
  int32_t padding;    /* LCE_PADDING_* (zero padding) */
  int32_t activation; /* LCE_ACT_* */
} lce_f32_conv_desc;

typedef struct lce_f32_pool_desc {
  int32_t batch, in_h, in_w, channels;
  int32_t filter_h, filter_w, stride_h, stride_w;
  int32_t padding;
  int32_t activation;
} lce_f32_pool_desc;

/* out = act(conv(in, filter) + bias); bias may be NULL. Also used for
 * FULLY_CONNECTED (1x1 conv on a [B,1,1,K] view). */
int lce_b200_f32_conv_out_shape(const lce_f32_conv_desc* d, int* out_h, int* out_w);
int lce_b200_f32_conv2d(const lce_f32_conv_desc* d, const float* in_dev, const float* filter_dev,
                        const float* bias_dev, float* out_dev, void* stream);
/* conv2d + LceQuantize of its output in one call: packed_out[pixel][ceil(out_c/32)] gets the sign
 * bits of `out` (bit = value < 0, tail bits 0), from the convolution's epilogue where the kernel
 * allows it, else by the stand-alone pack kernel. Identical to conv2d followed by lce_b200_quantize. */
int lce_b200_f32_conv2d_packed(const lce_f32_conv_desc* d, const float* in_dev,
                               const float* filter_dev, const float* bias_dev, float* out_dev,
                               int32_t* packed_out_dev, void* stream);
/* Diagnostics: successful launches so far of each convolution kernel conv2d(_packed) chooses from:
 * [0] tcgen05 tf32 pointwise, [1] tcgen05 tf32 7x7 stem, [2] direct (K <= 32), [3] small-M GEMM,
 * [4] 128x128 GEMM, [5] implicit GEMM 8x8, [6] implicit GEMM 8x4 (LCE_B200_IGEMM_8X4=1),
 * [7] implicit GEMM for K > 4096. */
void lce_b200_f32_conv_path_counts(uint64_t out[8]);
/* depth_multiplier 1; filter [1, fh, fw, C]; d->out_c == d->in_c */
int lce_b200_f32_depthwise_conv2d(const lce_f32_conv_desc* d, const float* in_dev,
                                  const float* filter_dev, const float* bias_dev,
                                  float* out_dev, void* stream);
int lce_b200_f32_pool_out_shape(const lce_f32_pool_desc* d, int* out_h, int* out_w);
int lce_b200_f32_max_pool(const lce_f32_pool_desc* d, const float* in_dev, float* out_dev,
                          void* stream);
int lce_b200_f32_avg_pool(const lce_f32_pool_desc* d, const float* in_dev, float* out_dev,
                          void* stream);
/* Fused MAX_POOL_2D(2x2, stride 1, VALID) -> DEPTHWISE_CONV_2D(3x3, depth_multiplier 1): the
 * anti-aliased down-sampling pair of QuickNet's transition blocks in one pass over the input
 * (the pooled tensor never reaches HBM). `pool` describes the max-pool on the input, `dw` the
 * depthwise conv on the POOLED tensor (dw->in_h / in_w = pooled size). channels % 4 == 0.
 * Bit-identical to running the two kernels one after the other. */
int lce_b200_f32_maxpool2x2_depthwise3x3(const lce_f32_pool_desc* pool, const lce_f32_conv_desc* dw,
                                         const float* in_dev, const float* filter_dev,
                                         const float* bias_dev, float* out_dev, void* stream);
/* Fused stem [DEQUANTIZE ->] CONV_2D(3x3, stride 2, 3 -> 16) -> DEPTHWISE_CONV_2D(3x3, stride 2)
 * (QuickNet's stem): one pass over the image; the dequantised image and the first conv's map stay
 * in shared memory. in_type LCE_T_FLOAT: `in_dev` is the float image (scale / zero point unused);
 * LCE_T_INT8 / LCE_T_BOOL (= uint8): the quantised image, dequantised as float(scale * (q - zp))
 * like lce_b200_dequantize_affine. `dw` describes the depthwise conv on the first conv's output.
 * The filters and biases are HOST pointers (w1 OHWI [16][3][3][3], w2 [1][3][3][16]; biases may be
 * NULL): 2.4 KB that travel by value in the kernel's parameter bank, where every FMA reads its
 * weight as a constant operand. Bit-identical to the separate kernels run one after the other. */
int lce_b200_f32_stem_conv_dw(const lce_f32_conv_desc* conv1, const lce_f32_conv_desc* dw, int in_type,
                              const void* in_dev, double in_scale, int32_t in_zero_point,
                              const float* w1_host, const float* b1_host, const float* w2_host,
                              const float* b2_host, float* out_dev, void* stream);
/* out[i] = act(a[i] (op) b[i % b_len]); b_len == n (same shape) or the last dim. */
int lce_b200_f32_add(const float* a_dev, const float* b_dev, float* out_dev, int64_t n,
                     int64_t b_len, int activation, void* stream);
int lce_b200_f32_mul(const float* a_dev, const float* b_dev, float* out_dev, int64_t n,
                     int64_t b_len, int activation, void* stream);
int lce_b200_f32_activation(const float* in_dev, float* out_dev, int64_t n, int activation,
                            void* stream);
/* mean over H and W: [B,H,W,C] -> [B,C] */
int lce_b200_f32_mean_hw(const float* in_dev, float* out_dev, int batch, int h, int w, int c,
                         void* stream);
/* the same with an activation applied to every element first: RELU -> MEAN of the model heads in one
 * pass (mean(act(x)), the same summation order as the two ops) */
int lce_b200_f32_mean_hw_act(const float* in_dev, float* out_dev, int batch, int h, int w, int c,
                             int pre_activation, void* stream);
/* softmax over the last dim: exp(beta*(x - max)) / sum */
int lce_b200_f32_softmax(const float* in_dev, float* out_dev, int64_t rows, int cols, float beta,
                         void* stream);

/* DEQUANTIZE of an int8 (LCE_T_INT8) or uint8 (LCE_T_BOOL's code) tensor:
 * out = float(scale * (q - zero_point)), TF/lite/kernels/internal/reference/dequantize.h:32-49.
 * The entry of a graph whose input was converted with inference_input_type int8 / uint8: a step
 * then ships a quarter of the bytes of float images over the host link. */
int lce_b200_dequantize_affine(int in_type, const void* in_dev, float* out_dev, int64_t n,
                               double scale, int32_t zero_point, void* stream);

/* PAD / PADV2 (TF/lite/kernels/internal/reference/pad.h) of a 4-D tensor of 32-bit elements
 * (float32 or bitpacked int32 words): out dims = in + before + after, border = fill_bits. */
int lce_b200_pad4d_32(const void* in_dev, void* out_dev, const int32_t* in_dims4,
                      const int32_t* pad_before4, const int32_t* pad_after4, uint32_t fill_bits,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif
