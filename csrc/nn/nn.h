// Launchers of the NN kernels (csrc/nn/*.cu). Raw-pointer C++ API; see nn_bindings.cpp.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace hefl {
namespace nn {

// Fused Adam with Keras' legacy time-based decay (FLPyfhelin.py:140):
//   lr_t = lr * lr_scale / (1 + decay * (t-1)),  t = *step (already incremented)
// Updates p, m, v in place, zeroes g, optionally writes a bf16 shadow of p.
void adam_step(float* p, float* g, float* m, float* v, void* shadow_bf16, int64_t n,
               const int64_t* step, const float* lr_scale, float lr, float decay, float beta1,
               float beta2, float eps, cudaStream_t st);

// ---- tcgen05 implicit-GEMM convolution (conv_tcgen05.cu) ----
void conv_fwd_pool(const void* X, const void* Wf, const float* bias, void* out, uint8_t* argmax, int B, int H,
                   int W, int CK, int CO, int spack, cudaStream_t st);
bool conv_fwd_pool_pair_supported(int H, int W, int CK, int CO);
void conv_fwd_pool_pair(const void* X, const void* Wf, const float* bias, void* out, uint8_t* argmax, int B, int H,
                        int W, int CK, int CO, int spack, cudaStream_t st);
void conv_set_debug(int mask);
void conv_dgrad(const void* dY, const void* Wd, void* dX, int B, int H, int W, int CK, int CO, const uint8_t* up_amax,
                int up_W, cudaStream_t st);
// dW32 += the weight gradient. part: workspace of conv_wgrad_part_floats(...) floats for the per-CTA partial sums,
// which are added in a fixed order, so the result does not change from run to run.
size_t conv_wgrad_part_floats(int B, int H, int W, int CK, int Co);
void conv_wgrad(const void* X, const void* DY, float* dW32, float* part, int B, int H, int W, int CK, int Co,
                cudaStream_t st);

// Dense head (Flatten -> Dense/ReLU -> Dense/ReLU -> Dense -> softmax-CE) forward + backward.
void head_forward_backward(const void* feat, const float* W1, const float* b1, const float* W2, const float* b2,
                           const float* W3, const float* b3, const int64_t* y, float* gW1, float* gb1, float* gW2,
                           float* gb2, float* gW3, float* gb3, void* dfeat, float* h1_buf, float* dh1_buf,
                           float* out, int64_t* step, int B, int F, int H1, int H2, int C, int train, cudaStream_t st);
void set_pdl(int on);
bool head_cluster_supported(int B, int F, int H1, int H2, int C);
void head_cluster(const void* feat, const float* W1, const float* b1, const float* W2, const float* b2,
                  const float* W3, const float* b3, const int64_t* y, float* gW1, float* gb1, float* gW2, float* gb2,
                  float* gW3, float* gb3, void* dfeat, float* out, int64_t* step, int B, int C, int train,
                  cudaStream_t st);
bool wgrad0_gather_supported(int W, int Wp, int CK, int Ci, int Co);
void wgrad0_gather(const void* X, const void* g, const uint8_t* amax, float* dW, int B, int H, int W, int Hp, int Wp,
                   cudaStream_t st);
// the same gradient as four masked GEMMs on the tensor cores (wgrad0_mma.cu); needs the s-packed layer-1 input
bool wgrad0_mma_supported(int W, int Wp, int CK, int Ci, int Co);
// (deterministic like conv_wgrad: part holds wgrad0_mma_part_floats(B, Hp) floats of per-CTA partial sums)
size_t wgrad0_mma_part_floats(int B, int Hp);
void wgrad0_mma(const void* X, const void* g, const uint8_t* amax, float* dW, float* part, int B, int H, int W, int Hp,
                int Wp, cudaStream_t st);
// ---- general tcgen05 GEMMs for the ResNet convolutions (gemm_tcgen05.cu) ----
// C[rows_out, N] (bf16) = sum_{t < taps} A[m + shifts[t], K] . B[t*N + n, K]^T. padded != 0: A rows index a zero-padded
// [Bn][H+2][W+2] grid and only interior pixels are written (to the dense [Bn*H*W, N] output). fp8: A and B hold e4m3
// bytes and the product of the two device scalars scale_a * scale_b multiplies the result.
void gemm_taps(const void* A, const void* Bm, void* C, int64_t a_rows, int N, int K, int taps, const int* shifts, int padded,
               int Bn, int H, int W, bool fp8, const float* scale_a, const float* scale_b, cudaStream_t st);
// dW[taps][Co][Ci] (fp32, zeroed by the caller) += dY[rows, Co]^T . X[rows + shift(tap), Ci]; taps = 1, or 9 on a padded
// grid whose rows are Wp pixels long.
void wgrad_taps(const void* DY, const void* X, float* dW, int64_t rows, int Co, int Ci, int taps, int Wp, cudaStream_t st);
void gemm_mxfp8(const void* A, const void* Bm, const void* sfa, const void* sfb, void* C, int64_t M, int N, int K,
                int idesc_variant, cudaStream_t st);
void pad_nhwc(const void* x, void* xp, int B, int H, int W, int C, cudaStream_t st);          // bf16, zero border of 1
void conv_weight_prep(const float* w, void* wt, void* wd, int Co, int Ci, int kk, cudaStream_t st);
void conv_wgrad_unpack(const float* dw, float* g, int Co, int Ci, int kk, cudaStream_t st);
// ---- ResNet building blocks (resnet_kernels.cu) ----
void bn_forward(const void* x, const void* res, const float* gamma, const float* beta, float* run_mean, float* run_var,
                float* mean, float* invstd, float* sums, void* y, int64_t P, int C, float momentum, float eps, int relu,
                cudaStream_t st);
void bn_backward(const void* dy, const void* x, const void* y, const float* mean, const float* invstd,
                 const float* gamma, float* sums, void* dx, void* dres, int64_t P, int C, int relu, cudaStream_t st);
void avgpool_forward(const void* x, float* out, int B, int HW, int C, cudaStream_t st);
void avgpool_backward(const float* dout, void* dx, int B, int HW, int C, cudaStream_t st);
void fp8_quantize(const void* x, uint8_t* q, const float* scale, float* amax, int64_t n, cudaStream_t st);
// bf16 [R,K] -> e4m3 [R,K] + UE8M0 scale tiles [ceil(R/128)][K/128][512] (rows beyond R must be pre-set by the caller)
void mxfp8_quantize(const void* x, uint8_t* q, uint8_t* sf, int64_t R, int K, cudaStream_t st);
void fp8_scale_update(float* amax, float* scale, float* inv, float target, cudaStream_t st);
void umma_shift_probe(const void* A, const void* Bm, float* out, int CK, int shift_rows, int mode, cudaStream_t st);

// ---- data-movement kernels around the convolutions (nn_kernels.cu) ----
constexpr int kMaxConvLayers = 8;
struct ConvLayerTable {
  int n;
  int Ci[kMaxConvLayers], CK[kMaxConvLayers], Co[kMaxConvLayers];
  int64_t w_off[kMaxConvLayers], b_off[kMaxConvLayers];       // offsets into the flat fp32 parameter buffer
  int64_t wf_off[kMaxConvLayers], wd_off[kMaxConvLayers];     // offsets (elements) into the bf16 Wf / Wd buffers
  int64_t dw_off[kMaxConvLayers];                             // offsets (elements) into the fp32 dW32 buffer
};
void preprocess_u8(const uint8_t* x, const float* theta, void* X, int B, int H, int W, uint64_t aug_seed,
                   const int64_t* step, int spack, cudaStream_t st);
void unpool_relu(const void* g, const uint8_t* amax, const void* ypool, void* dY, int B, int H, int W, int Hp,
                 int Wp, int Co, cudaStream_t st);
void conv_weight_relayout(const void* shadow, const ConvLayerTable& t, void* Wf, void* Wd, int l0, int l1,
                          int spack0, cudaStream_t st);
void conv_grad_finalize(float* dW32, const ConvLayerTable& t, float* grad, int l0, int l1, cudaStream_t st);
void fused_update(float* dW32, const ConvLayerTable& t, float* flat, float* grad, float* m, float* v, void* shadow,
                  void* Wf, void* Wd, const int64_t* step, const float* lr_scale, float lr, float decay, float beta1,
                  float beta2, float eps, int64_t dense_off, int64_t n_trainable, cudaStream_t st);

}  // namespace nn
}  // namespace hefl
