// torch.ops.hefl.* bindings for the NN kernels.
#include <ATen/cuda/CUDAContext.h>
#include <torch/library.h>
#include <torch/torch.h>

#include <cmath>

#include "nn.h"

namespace {

using at::Tensor;

void adam_step_(Tensor p, Tensor g, Tensor m, Tensor v, const c10::optional<Tensor>& shadow,
                const Tensor& step, const c10::optional<Tensor>& lr_scale, double lr, double decay,
                double beta1, double beta2, double eps) {
  TORCH_CHECK(p.scalar_type() == at::kFloat && p.is_contiguous(), "p must be contiguous float32");
  TORCH_CHECK(g.numel() == p.numel() && m.numel() == p.numel() && v.numel() == p.numel(), "size mismatch");
  TORCH_CHECK(step.scalar_type() == at::kLong && step.numel() == 1, "step must be a 1-element int64 tensor");
  const int64_t n = p.numel();
  if (p.is_cuda()) {
    void* sh = nullptr;
    if (shadow.has_value()) {
      TORCH_CHECK(shadow->scalar_type() == at::kBFloat16 && shadow->numel() >= n, "bad shadow");
      sh = shadow->data_ptr();
    }
    hefl::nn::adam_step(p.data_ptr<float>(), g.data_ptr<float>(), m.data_ptr<float>(), v.data_ptr<float>(),
                        sh, n, step.data_ptr<int64_t>(),
                        lr_scale.has_value() ? lr_scale->data_ptr<float>() : nullptr, (float)lr,
                        (float)decay, (float)beta1, (float)beta2, (float)eps,
                        at::cuda::getCurrentCUDAStream().stream());
    return;
  }
  const float t = (float)step.item<int64_t>();
  const float scale = lr_scale.has_value() ? lr_scale->item<float>() : 1.0f;
  const float lr_t = (float)lr * scale / (1.0f + (float)decay * (t - 1.0f));
  const float alpha = lr_t * std::sqrt(1.0f - std::pow((float)beta2, t)) / (1.0f - std::pow((float)beta1, t));
  float* pp = p.data_ptr<float>();
  float* gp = g.data_ptr<float>();
  float* mp = m.data_ptr<float>();
  float* vp = v.data_ptr<float>();
  for (int64_t i = 0; i < n; ++i) {
    const float gi = gp[i];
    mp[i] = (float)beta1 * mp[i] + (1.0f - (float)beta1) * gi;
    vp[i] = (float)beta2 * vp[i] + (1.0f - (float)beta2) * gi * gi;
    pp[i] -= alpha * mp[i] / (std::sqrt(vp[i]) + (float)eps);
    gp[i] = 0.0f;
  }
  if (shadow.has_value()) shadow->copy_(p);
}

// Native data-loader primitive: copy rows `indices` of a pinned host tensor straight into a
// device batch buffer with one cudaMemcpyAsync per row on the current stream (no CPU gather).
void gather_h2d_(Tensor dst, const Tensor& src, const Tensor& indices) {
  TORCH_CHECK(dst.is_cuda() && src.is_cpu() && indices.is_cpu(), "dst on GPU, src/indices on CPU");
  TORCH_CHECK(dst.is_contiguous() && src.is_contiguous(), "contiguous tensors required");
  TORCH_CHECK(indices.scalar_type() == at::kLong, "indices must be int64");
  TORCH_CHECK(dst.scalar_type() == src.scalar_type(), "dtype mismatch");
  const int64_t rows = indices.numel();
  TORCH_CHECK(dst.size(0) >= rows, "dst too small");
  const size_t row_bytes = (size_t)(src.numel() / src.size(0)) * src.element_size();
  TORCH_CHECK((size_t)(dst.numel() / dst.size(0)) * dst.element_size() == row_bytes, "row size mismatch");
  const char* sp = static_cast<const char*>(src.data_ptr());
  char* dp = static_cast<char*>(dst.data_ptr());
  const int64_t* ix = indices.data_ptr<int64_t>();
  cudaStream_t st = at::cuda::getCurrentCUDAStream().stream();
  for (int64_t r = 0; r < rows; ++r) {
    TORCH_CHECK(ix[r] >= 0 && ix[r] < src.size(0), "index out of range");
    cudaMemcpyAsync(dp + (size_t)r * row_bytes, sp + (size_t)ix[r] * row_bytes, row_bytes,
                    cudaMemcpyHostToDevice, st);
  }
}

inline cudaStream_t cur() { return at::cuda::getCurrentCUDAStream().stream(); }
inline void chk_bf16(const Tensor& t, const char* n) {
  TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kBFloat16 && t.is_contiguous(), n, " must be a contiguous CUDA bf16 tensor");
}

void conv_fwd_pool(const Tensor& X, const Tensor& Wf, const Tensor& bias, Tensor out,
                   const c10::optional<Tensor>& argmax, int64_t B, int64_t H, int64_t W, int64_t CK, int64_t CO,
                   bool spack) {
  chk_bf16(X, "X"); chk_bf16(Wf, "Wf"); chk_bf16(out, "out");
  TORCH_CHECK(X.numel() == B * H * W * CK, "X must be [B*H*W, CK]");
  TORCH_CHECK(Wf.numel() >= (spack ? 3 : 9) * CO * CK, "Wf must be [9, CO, CK] ([3, CO, CK] s-packed)");
  TORCH_CHECK(!spack || (CK == 16 && CO == 32), "s-packed input is the 3-channel first layer only");
  TORCH_CHECK(bias.is_cuda() && bias.scalar_type() == at::kFloat && bias.numel() == CO, "bias must be float32 [CO]");
  const int64_t Hp = (H - 2) / 2, Wp = (W - 2) / 2;
  TORCH_CHECK(out.numel() == B * Hp * Wp * CO, "out must be [B,Hp,Wp,CO]");
  uint8_t* am = nullptr;
  if (argmax.has_value()) {
    TORCH_CHECK(argmax->scalar_type() == at::kByte && argmax->numel() == out.numel(), "bad argmax");
    am = argmax->data_ptr<uint8_t>();
  }
  hefl::nn::conv_fwd_pool(X.data_ptr(), Wf.data_ptr(), bias.data_ptr<float>(), out.data_ptr(), am, (int)B, (int)H,
                          (int)W, (int)CK, (int)CO, spack ? 1 : 0, cur());
}

// up_amax given: the un-pooling of the previous layer is fused into the epilogue — dX is then that layer's
// conv-grid gradient [B*up_W*up_W, CO] (H = W = (up_W - 2) / 2 of this call), written at the arg-max positions.
// Pair-row forward kernel (conv_tcgen05.cu G1b): same contract as conv_fwd_pool with the plain [9, CO, CK] weights.
void conv_fwd_pool_pair(const Tensor& X, const Tensor& Wf, const Tensor& bias, Tensor out,
                        const c10::optional<Tensor>& argmax, int64_t B, int64_t H, int64_t W, int64_t CK, int64_t CO,
                        bool spack) {
  chk_bf16(X, "X"); chk_bf16(Wf, "Wf"); chk_bf16(out, "out");
  TORCH_CHECK(X.numel() >= B * H * W * CK && Wf.numel() >= (spack ? 3 : 9) * CO * CK, "shape mismatch");
  TORCH_CHECK(!spack || (CK == 16 && CO == 32), "s-packed input is the 3-channel first layer only");
  TORCH_CHECK(hefl::nn::conv_fwd_pool_pair_supported((int)H, (int)W, (int)CK, (int)CO), "conv_fwd_pool_pair: unsupported shape");
  const int64_t Hp = (H - 2) / 2, Wp = (W - 2) / 2;
  TORCH_CHECK(out.numel() == B * Hp * Wp * CO, "out must be [B,Hp,Wp,CO]");
  uint8_t* am = nullptr;
  if (argmax.has_value()) {
    TORCH_CHECK(argmax->scalar_type() == at::kByte && argmax->numel() == out.numel(), "bad argmax");
    am = argmax->data_ptr<uint8_t>();
  }
  hefl::nn::conv_fwd_pool_pair(X.data_ptr(), Wf.data_ptr(), bias.data_ptr<float>(), out.data_ptr(), am, (int)B, (int)H,
                               (int)W, (int)CK, (int)CO, spack ? 1 : 0, cur());
}

void conv_dgrad(const Tensor& dY, const Tensor& Wd, Tensor dX, int64_t B, int64_t H, int64_t W, int64_t CK,
                int64_t CO, const c10::optional<Tensor>& up_amax, int64_t up_W) {
  chk_bf16(dY, "dY"); chk_bf16(Wd, "Wd"); chk_bf16(dX, "dX");
  TORCH_CHECK(dY.numel() == B * H * W * CK && Wd.numel() == 9 * CO * CK, "shape mismatch");
  const uint8_t* up = nullptr;
  if (up_amax.has_value()) {
    TORCH_CHECK(up_amax->is_cuda() && up_amax->scalar_type() == at::kByte && up_amax->numel() == B * H * W * CO, "bad up_amax");
    TORCH_CHECK(H == W && (up_W - 2) / 2 == H && dX.numel() == B * up_W * up_W * CO, "fused un-pool: dX must be [B*up_W*up_W, CO]");
    up = up_amax->data_ptr<uint8_t>();
  } else {
    TORCH_CHECK(dX.numel() == B * H * W * CO, "dX must be [B*H*W, CO]");
  }
  hefl::nn::conv_dgrad(dY.data_ptr(), Wd.data_ptr(), dX.data_ptr(), (int)B, (int)H, (int)W, (int)CK, (int)CO, up, (int)up_W,
                       cur());
}

void conv_wgrad(const Tensor& X, const Tensor& DY, Tensor dW32, int64_t B, int64_t H, int64_t W, int64_t CK, int64_t Co) {
  chk_bf16(X, "X"); chk_bf16(DY, "DY");
  const int64_t P = B * H * W;
  TORCH_CHECK(X.numel() == P * CK && DY.numel() == P * Co, "X must be [B*H*W,CK] and DY [B*H*W,Co]");
  TORCH_CHECK(dW32.is_cuda() && dW32.scalar_type() == at::kFloat && dW32.numel() >= (9 * CK + 1) * Co, "dW32 too small");
  // per-CTA partial sums, summed in a fixed order by the launcher (from the caching allocator: graph-capture safe)
  Tensor part = at::empty({(int64_t)hefl::nn::conv_wgrad_part_floats((int)B, (int)H, (int)W, (int)CK, (int)Co)},
                          dW32.options());
  hefl::nn::conv_wgrad(X.data_ptr(), DY.data_ptr(), dW32.data_ptr<float>(), part.data_ptr<float>(), (int)B, (int)H, (int)W,
                       (int)CK, (int)Co, cur());
}

void preprocess_u8(const Tensor& x, const c10::optional<Tensor>& theta, Tensor X, int64_t aug_seed,
                   const c10::optional<Tensor>& step, bool spack) {
  TORCH_CHECK(x.is_cuda() && x.scalar_type() == at::kByte && x.is_contiguous() && x.dim() == 4 && x.size(3) == 3, "x must be uint8 [B,H,W,3]");
  chk_bf16(X, "X");
  const int64_t B = x.size(0), H = x.size(1), W = x.size(2);
  TORCH_CHECK(X.numel() == B * H * W * 16, "X must be [B*H*W, 16]");
  const float* th = nullptr;
  if (theta.has_value()) {
    TORCH_CHECK(theta->is_cuda() && theta->scalar_type() == at::kFloat && theta->numel() == B * 6 && theta->is_contiguous(), "theta must be float32 [B,2,3]");
    th = theta->data_ptr<float>();
  }
  const int64_t* sp = nullptr;
  if (step.has_value()) {
    TORCH_CHECK(step->is_cuda() && step->scalar_type() == at::kLong && step->numel() == 1, "step must be a CUDA int64 scalar tensor");
    sp = step->data_ptr<int64_t>();
  }
  hefl::nn::preprocess_u8(x.data_ptr<uint8_t>(), th, X.data_ptr(), (int)B, (int)H, (int)W, (uint64_t)aug_seed, sp, spack ? 1 : 0, cur());
}

void unpool_relu(const Tensor& g, const Tensor& amax, const Tensor& ypool, Tensor dY, int64_t B, int64_t H,
                 int64_t W, int64_t Co) {
  chk_bf16(g, "g"); chk_bf16(ypool, "ypool"); chk_bf16(dY, "dY");
  const int64_t Hp = (H - 2) / 2, Wp = (W - 2) / 2;
  TORCH_CHECK(g.numel() == B * Hp * Wp * Co && ypool.numel() == g.numel() && amax.numel() == g.numel(), "pooled shapes mismatch");
  TORCH_CHECK(amax.scalar_type() == at::kByte, "amax must be uint8");
  TORCH_CHECK(dY.numel() == B * H * W * Co, "dY must be [B*H*W, Co]");
  TORCH_CHECK(Co % 8 == 0, "Co must be a multiple of 8");
  hefl::nn::unpool_relu(g.data_ptr(), amax.data_ptr<uint8_t>(), ypool.data_ptr(), dY.data_ptr(), (int)B, (int)H,
                        (int)W, (int)Hp, (int)Wp, (int)Co, cur());
}

static int g_head_cluster = 1;

// flat / grad are the ParamPack buffers; offs = [W1, b1, W2, b2, W3, b3] element offsets.
void head_forward_backward(const Tensor& feat, const Tensor& flat, Tensor grad, at::IntArrayRef offs, const Tensor& y,
                           Tensor dfeat, Tensor h1_buf, Tensor dh1_buf, Tensor out, const c10::optional<Tensor>& step,
                           int64_t B, int64_t F, int64_t H1, int64_t H2, int64_t C, bool train) {
  chk_bf16(feat, "feat"); chk_bf16(dfeat, "dfeat");
  TORCH_CHECK(offs.size() == 6, "need six parameter offsets");
  TORCH_CHECK(B <= 32 && B >= 1, "the head kernels handle up to 32 samples per step");
  TORCH_CHECK(feat.numel() == B * F && dfeat.numel() == B * F, "feat/dfeat must be [B,F]");
  TORCH_CHECK(flat.is_cuda() && flat.scalar_type() == at::kFloat && grad.scalar_type() == at::kFloat, "float32 parameter buffers required");
  TORCH_CHECK(y.is_cuda() && y.scalar_type() == at::kLong && y.numel() == B, "labels must be int64 [B]");
  TORCH_CHECK(h1_buf.numel() >= B * H1 && dh1_buf.numel() >= B * (H1 + H2) && out.numel() >= 2, "scratch too small");
  const float* p = flat.data_ptr<float>();
  float* g = grad.data_ptr<float>();
  if (g_head_cluster && hefl::nn::head_cluster_supported((int)B, (int)F, (int)H1, (int)H2, (int)C)) {
    // one launch on a cluster of 8 CTAs (csrc/nn/head_cluster.cu)
    hefl::nn::head_cluster(feat.data_ptr(), p + offs[0], p + offs[1], p + offs[2], p + offs[3], p + offs[4], p + offs[5],
                           y.data_ptr<int64_t>(), g + offs[0], g + offs[1], g + offs[2], g + offs[3], g + offs[4],
                           g + offs[5], dfeat.data_ptr(), out.data_ptr<float>(),
                           step.has_value() ? step->data_ptr<int64_t>() : nullptr, (int)B, (int)C, train ? 1 : 0, cur());
    return;
  }
  TORCH_CHECK(B % 2 == 0 && H2 % 4 == 0 && H1 % 4 == 0 && F % 8 == 0, "head dims must be even / multiples of 4 / 8");
  hefl::nn::head_forward_backward(feat.data_ptr(), p + offs[0], p + offs[1], p + offs[2], p + offs[3], p + offs[4],
                                  p + offs[5], y.data_ptr<int64_t>(), g + offs[0], g + offs[1], g + offs[2],
                                  g + offs[3], g + offs[4], g + offs[5], dfeat.data_ptr(), h1_buf.data_ptr<float>(),
                                  dh1_buf.data_ptr<float>(), out.data_ptr<float>(),
                                  step.has_value() ? step->data_ptr<int64_t>() : nullptr, (int)B, (int)F, (int)H1, (int)H2,
                                  (int)C, train ? 1 : 0, cur());
}

void conv_set_debug(int64_t mask) { hefl::nn::conv_set_debug((int)mask); }

hefl::nn::ConvLayerTable table_from(const Tensor& t);

// x, res, y: NHWC bf16 viewed as [P, C]. Returns nothing; mean/invstd/sums are caller-provided fp32 scratch.
void bn_forward(const Tensor& x, const c10::optional<Tensor>& res, const Tensor& gamma, const Tensor& beta,
                const c10::optional<Tensor>& run_mean, const c10::optional<Tensor>& run_var, Tensor mean, Tensor invstd,
                Tensor sums, Tensor y, double momentum, double eps, bool relu) {
  chk_bf16(x, "x"); chk_bf16(y, "y");
  const int64_t C = gamma.numel();
  TORCH_CHECK(C % 8 == 0 && x.numel() % C == 0, "C must be a multiple of 8");
  const int64_t P = x.numel() / C;
  TORCH_CHECK(mean.numel() >= C && invstd.numel() >= C && sums.numel() >= 2 * C, "scratch too small");
  const void* rp = nullptr;
  if (res.has_value()) { chk_bf16(*res, "res"); TORCH_CHECK(res->numel() == x.numel(), "residual shape"); rp = res->data_ptr(); }
  hefl::nn::bn_forward(x.data_ptr(), rp, gamma.data_ptr<float>(), beta.data_ptr<float>(),
                       run_mean.has_value() ? run_mean->data_ptr<float>() : nullptr,
                       run_var.has_value() ? run_var->data_ptr<float>() : nullptr, mean.data_ptr<float>(),
                       invstd.data_ptr<float>(), sums.data_ptr<float>(), y.data_ptr(), P, (int)C, (float)momentum,
                       (float)eps, relu ? 1 : 0, cur());
}

void bn_backward(const Tensor& dy, const Tensor& x, const Tensor& y, const Tensor& mean, const Tensor& invstd,
                 const Tensor& gamma, Tensor sums, Tensor dx, const c10::optional<Tensor>& dres, bool relu) {
  chk_bf16(dy, "dy"); chk_bf16(x, "x"); chk_bf16(y, "y"); chk_bf16(dx, "dx");
  const int64_t C = gamma.numel();
  const int64_t P = x.numel() / C;
  void* dr = nullptr;
  if (dres.has_value()) { chk_bf16(*dres, "dres"); dr = dres->data_ptr(); }
  hefl::nn::bn_backward(dy.data_ptr(), x.data_ptr(), y.data_ptr(), mean.data_ptr<float>(), invstd.data_ptr<float>(),
                        gamma.data_ptr<float>(), sums.data_ptr<float>(), dx.data_ptr(), dr, P, (int)C, relu ? 1 : 0, cur());
}

// Layer-1 weight gradient from the pooled gradient (see wgrad_gather.cu). X: [B*H*W(+slack), 16] bf16,
// g: [B,Hp,Wp,32] bf16, amax: [B,Hp,Wp,32] u8 (bits 0-1 position, bit 2 active), dW32: [9*16+1, 32] fp32 (+=).
void wgrad0_gather(const Tensor& X, const Tensor& g, const Tensor& amax, Tensor dW32, int64_t B, int64_t H, int64_t W, bool spack) {
  chk_bf16(X, "X"); chk_bf16(g, "g");
  const int64_t Hp = (H - 2) / 2, Wp = (W - 2) / 2;
  TORCH_CHECK(hefl::nn::wgrad0_gather_supported((int)W, (int)Wp, 16, 3, 32), "wgrad0_gather: unsupported shape");
  TORCH_CHECK(X.numel() >= B * H * W * 16 && g.numel() == B * Hp * Wp * 32 && amax.numel() == g.numel(), "shape mismatch");
  TORCH_CHECK(amax.scalar_type() == at::kByte && dW32.scalar_type() == at::kFloat && dW32.numel() >= (9 * 16 + 1) * 32, "dtype / size");
  if (spack && hefl::nn::wgrad0_mma_supported((int)W, (int)Wp, 16, 3, 32)) {      // s-packed input: masked GEMMs on the tensor cores
    Tensor part = at::empty({(int64_t)hefl::nn::wgrad0_mma_part_floats((int)B, (int)Hp)}, dW32.options());
    hefl::nn::wgrad0_mma(X.data_ptr(), g.data_ptr(), amax.data_ptr<uint8_t>(), dW32.data_ptr<float>(), part.data_ptr<float>(),
                         (int)B, (int)H, (int)W, (int)Hp, (int)Wp, cur());
    return;
  }
  hefl::nn::wgrad0_gather(X.data_ptr(), g.data_ptr(), amax.data_ptr<uint8_t>(), dW32.data_ptr<float>(), (int)B, (int)H,
                          (int)W, (int)Hp, (int)Wp, cur());
}

void avgpool_forward(const Tensor& x, Tensor out, int64_t B, int64_t HW, int64_t C) {
  chk_bf16(x, "x");
  TORCH_CHECK(x.numel() == B * HW * C && out.numel() == B * C && out.scalar_type() == at::kFloat, "shape mismatch");
  hefl::nn::avgpool_forward(x.data_ptr(), out.data_ptr<float>(), (int)B, (int)HW, (int)C, cur());
}

void avgpool_backward(const Tensor& dout, Tensor dx, int64_t B, int64_t HW, int64_t C) {
  chk_bf16(dx, "dx");
  TORCH_CHECK(dx.numel() == B * HW * C && dout.numel() == B * C && dout.scalar_type() == at::kFloat, "shape mismatch");
  hefl::nn::avgpool_backward(dout.data_ptr<float>(), dx.data_ptr(), (int)B, (int)HW, (int)C, cur());
}

// q = e4m3(sat(x * scale)) (q: uint8 storage, viewed as float8_e4m3fn by the caller); amax = max(amax, |x|).
// out[rows_out, N] bf16 = sum_taps A[m + shift, K] . B[t*N + n, K]^T (tcgen05; csrc/nn/gemm_tcgen05.cu)
void gemm_taps(const Tensor& A, const Tensor& Bm, Tensor out, int64_t N, int64_t K, at::IntArrayRef shifts, int64_t padded,
               int64_t Bn, int64_t H, int64_t W, const c10::optional<Tensor>& scale_a, const c10::optional<Tensor>& scale_b) {
  TORCH_CHECK(A.is_cuda() && Bm.is_cuda() && out.is_cuda(), "gemm_taps is a CUDA (sm_100a) op");
  TORCH_CHECK(A.is_contiguous() && Bm.is_contiguous() && out.is_contiguous(), "contiguous operands expected");
  const bool fp8 = A.element_size() == 1;
  TORCH_CHECK(A.element_size() == Bm.element_size() && (fp8 || A.scalar_type() == at::kBFloat16), "bf16 or e4m3 operands");
  TORCH_CHECK(out.scalar_type() == at::kBFloat16, "bf16 output");
  const int taps = shifts.empty() ? 1 : (int)shifts.size();
  const int64_t a_rows = A.numel() / K;
  TORCH_CHECK(Bm.numel() == (int64_t)taps * N * K, "B must be [taps*N, K]");
  const int64_t rows_out = padded ? Bn * H * W : a_rows;
  TORCH_CHECK(out.numel() == rows_out * N, "output must be [rows_out, N]");
  if (padded) TORCH_CHECK(a_rows == Bn * (H + 2) * (W + 2), "A must cover the padded grid");
  std::vector<int> sh(shifts.begin(), shifts.end());
  hefl::nn::gemm_taps(A.data_ptr(), Bm.data_ptr(), out.data_ptr(), a_rows, (int)N, (int)K, taps, sh.empty() ? nullptr : sh.data(),
                      (int)padded, (int)Bn, (int)H, (int)W, fp8, scale_a.has_value() ? scale_a->data_ptr<float>() : nullptr,
                      scale_b.has_value() ? scale_b->data_ptr<float>() : nullptr, cur());
}

// dW [taps, Co, Ci] fp32 (zeroed here) = dY[rows, Co]^T . X[rows + shift(tap), Ci]
void wgrad_taps(const Tensor& DY, const Tensor& X, Tensor dW, int64_t taps, int64_t Wp) {
  TORCH_CHECK(DY.is_cuda() && X.is_cuda() && dW.is_cuda(), "wgrad_taps is a CUDA (sm_100a) op");
  TORCH_CHECK(DY.scalar_type() == at::kBFloat16 && X.scalar_type() == at::kBFloat16 && dW.scalar_type() == at::kFloat, "dtypes");
  TORCH_CHECK(DY.dim() == 2 && X.dim() == 2 && DY.size(0) == X.size(0) && DY.is_contiguous() && X.is_contiguous() && dW.is_contiguous(),
              "DY [rows, Co], X [rows, Ci]");
  const int64_t Co = DY.size(1), Ci = X.size(1);
  TORCH_CHECK(dW.numel() == taps * Co * Ci, "dW must be [taps, Co, Ci]");
  dW.zero_();
  hefl::nn::wgrad_taps(DY.data_ptr(), X.data_ptr(), dW.data_ptr<float>(), DY.size(0), (int)Co, (int)Ci, (int)taps, (int)Wp, cur());
}

// out [M,N] bf16 = block-scaled e4m3 GEMM (kind::mxf8f6f4.block_scale); sfa / sfb: uint8 tiles [rows/128][K/128][512]
void gemm_mxfp8(const Tensor& A, const Tensor& Bm, const Tensor& sfa, const Tensor& sfb, Tensor out, int64_t variant) {
  TORCH_CHECK(A.is_cuda() && A.element_size() == 1 && Bm.element_size() == 1 && A.dim() == 2 && Bm.dim() == 2 &&
              A.is_contiguous() && Bm.is_contiguous() && A.size(1) == Bm.size(1), "A [M,K], B [N,K] e4m3 bytes");
  const int64_t M = A.size(0), K = A.size(1), N = Bm.size(0);
  TORCH_CHECK(out.scalar_type() == at::kBFloat16 && out.numel() == M * N && out.is_contiguous(), "out [M,N] bf16");
  TORCH_CHECK(sfa.numel() == ((M + 127) / 128) * (K / 128) * 512 && sfb.numel() == (N / 128) * (K / 128) * 512 &&
              sfa.is_contiguous() && sfb.is_contiguous(), "scale-factor tiles have the wrong size");
  hefl::nn::gemm_mxfp8(A.data_ptr(), Bm.data_ptr(), sfa.data_ptr(), sfb.data_ptr(), out.data_ptr(), M, (int)N, (int)K, (int)variant, cur());
}

// x bf16 [R,K] (K % 128 == 0) -> (e4m3 bytes [R,K], UE8M0 scale tiles uint8 [ceil(R/128) * K/128 * 512])
std::tuple<Tensor, Tensor> mxfp8_quantize(const Tensor& x) {
  TORCH_CHECK(x.is_cuda() && x.scalar_type() == at::kBFloat16 && x.dim() == 2 && x.is_contiguous() && x.size(1) % 128 == 0,
              "bf16 [R,K] with K a multiple of 128");
  const int64_t R = x.size(0), K = x.size(1);
  Tensor q = at::empty({R, K}, x.options().dtype(at::kByte));
  Tensor sf = at::full({((R + 127) / 128) * (K / 128) * 512}, 127, x.options().dtype(at::kByte));
  hefl::nn::mxfp8_quantize(x.data_ptr(), q.data_ptr<uint8_t>(), sf.data_ptr<uint8_t>(), R, (int)K, cur());
  return {q, sf};
}

void fp8_scale_update(Tensor amax, Tensor scale, Tensor inv, double target) {
  TORCH_CHECK(amax.is_cuda() && amax.scalar_type() == at::kFloat && scale.scalar_type() == at::kFloat && inv.scalar_type() == at::kFloat,
              "fp32 CUDA scalars expected");
  hefl::nn::fp8_scale_update(amax.data_ptr<float>(), scale.data_ptr<float>(), inv.data_ptr<float>(), (float)target, cur());
}

// x: channels_last bf16 [B,C,H,W] (i.e. NHWC storage) -> zero-padded NHWC [B,H+2,W+2,C] in one pass
Tensor pad_nhwc(const Tensor& x) {
  TORCH_CHECK(x.is_cuda() && x.scalar_type() == at::kBFloat16 && x.dim() == 4 && x.is_contiguous(at::MemoryFormat::ChannelsLast),
              "pad_nhwc expects a channels_last bf16 CUDA tensor");
  const int64_t B = x.size(0), C = x.size(1), H = x.size(2), W = x.size(3);
  Tensor xp = at::empty({B, H + 2, W + 2, C}, x.options());
  hefl::nn::pad_nhwc(x.data_ptr(), xp.data_ptr(), (int)B, (int)H, (int)W, (int)C, cur());
  return xp;
}

// fp32 [Co,Ci,k,k] -> (bf16 [k*k*Co, Ci] forward taps, bf16 [k*k*Ci, Co] rotated / transposed taps for dgrad)
std::tuple<Tensor, Tensor> conv_weight_prep(const Tensor& w) {
  TORCH_CHECK(w.is_cuda() && w.scalar_type() == at::kFloat && w.dim() == 4 && w.is_contiguous(), "fp32 [Co,Ci,k,k] weights");
  const int64_t Co = w.size(0), Ci = w.size(1), kk = w.size(2) * w.size(3);
  Tensor wt = at::empty({kk * Co, Ci}, w.options().dtype(at::kBFloat16));
  Tensor wd = at::empty({kk * Ci, Co}, w.options().dtype(at::kBFloat16));
  hefl::nn::conv_weight_prep(w.data_ptr<float>(), wt.data_ptr(), wd.data_ptr(), (int)Co, (int)Ci, (int)kk, cur());
  return {wt, wd};
}

Tensor conv_wgrad_unpack(const Tensor& dw, int64_t Co, int64_t Ci, int64_t k) {
  TORCH_CHECK(dw.is_cuda() && dw.scalar_type() == at::kFloat && dw.is_contiguous() && dw.numel() == k * k * Co * Ci, "dW [k*k,Co,Ci]");
  Tensor g = at::empty({Co, Ci, k, k}, dw.options());
  hefl::nn::conv_wgrad_unpack(dw.data_ptr<float>(), g.data_ptr<float>(), (int)Co, (int)Ci, (int)(k * k), cur());
  return g;
}

void fp8_quantize(const Tensor& x, Tensor q, const Tensor& scale, Tensor amax) {
  chk_bf16(x, "x");
  TORCH_CHECK(q.is_cuda() && q.is_contiguous() && q.element_size() == 1 && q.numel() == x.numel(), "q must be a 1-byte tensor like x");
  TORCH_CHECK(x.numel() % 8 == 0, "numel must be a multiple of 8");
  TORCH_CHECK(scale.is_cuda() && scale.scalar_type() == at::kFloat && amax.is_cuda() && amax.scalar_type() == at::kFloat, "scale / amax must be float32 CUDA scalars");
  hefl::nn::fp8_quantize(x.data_ptr(), reinterpret_cast<uint8_t*>(q.data_ptr()), scale.data_ptr<float>(), amax.data_ptr<float>(),
                         x.numel(), cur());
}

void fused_update(Tensor dW32, const Tensor& table, Tensor flat, Tensor grad, Tensor m, Tensor v, Tensor shadow, Tensor Wf,
                  Tensor Wd, const Tensor& step, const c10::optional<Tensor>& lr_scale, double lr, double decay,
                  double beta1, double beta2, double eps, int64_t dense_off, int64_t n_trainable) {
  chk_bf16(shadow, "shadow"); chk_bf16(Wf, "Wf"); chk_bf16(Wd, "Wd");
  TORCH_CHECK(flat.scalar_type() == at::kFloat && grad.scalar_type() == at::kFloat && m.scalar_type() == at::kFloat &&
              v.scalar_type() == at::kFloat && dW32.scalar_type() == at::kFloat, "float32 buffers required");
  TORCH_CHECK(step.is_cuda() && step.scalar_type() == at::kLong, "step must be a CUDA int64 tensor");
  hefl::nn::fused_update(dW32.data_ptr<float>(), table_from(table), flat.data_ptr<float>(), grad.data_ptr<float>(),
                         m.data_ptr<float>(), v.data_ptr<float>(), shadow.data_ptr(), Wf.data_ptr(), Wd.data_ptr(),
                         step.data_ptr<int64_t>(), lr_scale.has_value() ? lr_scale->data_ptr<float>() : nullptr,
                         (float)lr, (float)decay, (float)beta1, (float)beta2, (float)eps, dense_off, n_trainable, cur());
}

Tensor umma_shift_probe(const Tensor& A, const Tensor& Bm, int64_t CK, int64_t shift_rows, int64_t mode) {
  chk_bf16(A, "A"); chk_bf16(Bm, "Bm");
  TORCH_CHECK(A.numel() == 144 * CK && Bm.numel() == 32 * CK, "A must be [144,CK], B [32,CK]");
  Tensor out = at::zeros({128, 32}, A.options().dtype(at::kFloat));
  hefl::nn::umma_shift_probe(A.data_ptr(), Bm.data_ptr(), out.data_ptr<float>(), (int)CK, (int)shift_rows, (int)mode, cur());
  return out;
}

hefl::nn::ConvLayerTable table_from(const Tensor& t) {
  TORCH_CHECK(t.is_cpu() && t.scalar_type() == at::kLong && t.dim() == 2 && t.size(1) == 8, "table must be CPU int64 [n,8]");
  hefl::nn::ConvLayerTable T;
  T.n = (int)t.size(0);
  TORCH_CHECK(T.n <= hefl::nn::kMaxConvLayers, "too many conv layers");
  const int64_t* p = t.data_ptr<int64_t>();
  for (int l = 0; l < T.n; ++l) {
    T.Ci[l] = (int)p[l * 8 + 0]; T.CK[l] = (int)p[l * 8 + 1]; T.Co[l] = (int)p[l * 8 + 2];
    T.w_off[l] = p[l * 8 + 3]; T.b_off[l] = p[l * 8 + 4]; T.wf_off[l] = p[l * 8 + 5];
    T.wd_off[l] = p[l * 8 + 6]; T.dw_off[l] = p[l * 8 + 7];
  }
  return T;
}

// l0/l1: layer range [l0, l1) (l1 = -1: all layers) so the update of the layers whose gradients are final can
// run on a side stream under the last weight-gradient kernel.
void conv_weight_relayout(const Tensor& shadow, const Tensor& table, Tensor Wf, Tensor Wd, int64_t l0, int64_t l1,
                          bool spack0) {
  chk_bf16(shadow, "shadow"); chk_bf16(Wf, "Wf"); chk_bf16(Wd, "Wd");
  const auto t = table_from(table);
  if (l1 < 0) l1 = t.n;
  TORCH_CHECK(0 <= l0 && l1 <= t.n, "layer range");
  hefl::nn::conv_weight_relayout(shadow.data_ptr(), t, Wf.data_ptr(), Wd.data_ptr(), (int)l0, (int)l1, spack0 ? 1 : 0, cur());
}

void conv_grad_finalize(Tensor dW32, const Tensor& table, Tensor grad, int64_t l0, int64_t l1) {
  TORCH_CHECK(dW32.is_cuda() && dW32.scalar_type() == at::kFloat && grad.is_cuda() && grad.scalar_type() == at::kFloat, "float32 CUDA tensors required");
  const auto t = table_from(table);
  if (l1 < 0) l1 = t.n;
  TORCH_CHECK(0 <= l0 && l1 <= t.n, "layer range");
  hefl::nn::conv_grad_finalize(dW32.data_ptr<float>(), t, grad.data_ptr<float>(), (int)l0, (int)l1, cur());
}

}  // namespace

TORCH_LIBRARY_FRAGMENT(hefl, m) {
  m.def("adam_step_(Tensor(a!) p, Tensor(b!) g, Tensor(c!) m, Tensor(d!) v, Tensor? shadow, Tensor step, Tensor? lr_scale, float lr, float decay, float beta1, float beta2, float eps) -> ()", &adam_step_);
  m.def("gather_h2d_(Tensor(a!) dst, Tensor src, Tensor indices) -> ()", &gather_h2d_);
  m.def("conv_fwd_pool(Tensor X, Tensor Wf, Tensor bias, Tensor(a!) out, Tensor(b!)? argmax, int B, int H, int W, int CK, int CO, bool spack=False) -> ()", &conv_fwd_pool);
  m.def("conv_fwd_pool_pair(Tensor X, Tensor Wf, Tensor bias, Tensor(a!) out, Tensor(b!)? argmax, int B, int H, int W, int CK, int CO, bool spack=False) -> ()", &conv_fwd_pool_pair);
  m.def("conv_dgrad(Tensor dY, Tensor Wd, Tensor(a!) dX, int B, int H, int W, int CK, int CO, Tensor? up_amax=None, int up_W=0) -> ()", &conv_dgrad);
  m.def("conv_wgrad(Tensor X, Tensor DY, Tensor(a!) dW32, int B, int H, int W, int CK, int Co) -> ()", &conv_wgrad);
  m.def("preprocess_u8(Tensor x, Tensor? theta, Tensor(a!) X, int aug_seed, Tensor? step, bool spack=False) -> ()", &preprocess_u8);
  m.def("unpool_relu(Tensor g, Tensor amax, Tensor ypool, Tensor(a!) dY, int B, int H, int W, int Co) -> ()", &unpool_relu);
  m.def("head_forward_backward(Tensor feat, Tensor flat, Tensor(a!) grad, int[] offs, Tensor y, Tensor(b!) dfeat, Tensor(c!) h1_buf, Tensor(d!) dh1_buf, Tensor(e!) out, Tensor(f!)? step, int B, int F, int H1, int H2, int C, bool train) -> ()", &head_forward_backward);
  m.def("fused_update(Tensor(a!) dW32, Tensor table, Tensor(b!) flat, Tensor(c!) grad, Tensor(d!) m, Tensor(e!) v, Tensor(f!) shadow, Tensor(g!) Wf, Tensor(h!) Wd, Tensor step, Tensor? lr_scale, float lr, float decay, float beta1, float beta2, float eps, int dense_off, int n_trainable) -> ()", &fused_update);
  m.def("conv_set_debug(int mask) -> ()", &conv_set_debug);
  m.def("set_head_cluster(int on) -> ()", [](int64_t on) { g_head_cluster = (int)on; });
  m.def("set_pdl(int on) -> ()", [](int64_t on) { hefl::nn::set_pdl((int)on); });
  m.def("wgrad0_gather(Tensor X, Tensor g, Tensor amax, Tensor(a!) dW32, int B, int H, int W, bool spack=False) -> ()", &wgrad0_gather);
  m.def("fp8_quantize(Tensor x, Tensor(a!) q, Tensor scale, Tensor(b!) amax) -> ()", &fp8_quantize);
  m.def("gemm_taps(Tensor A, Tensor B, Tensor(a!) out, int N, int K, int[] shifts, int padded, int Bn, int H, int W, Tensor? scale_a, Tensor? scale_b) -> ()", &gemm_taps);
  m.def("wgrad_taps(Tensor DY, Tensor X, Tensor(a!) dW, int taps, int Wp) -> ()", &wgrad_taps);
  m.def("pad_nhwc(Tensor x) -> Tensor", &pad_nhwc);
  m.def("mxfp8_quantize(Tensor x) -> (Tensor, Tensor)", &mxfp8_quantize);
  m.def("gemm_mxfp8(Tensor A, Tensor B, Tensor sfa, Tensor sfb, Tensor(a!) out, int variant) -> ()", &gemm_mxfp8);
  m.def("fp8_scale_update(Tensor(a!) amax, Tensor(b!) scale, Tensor(c!) inv, float target) -> ()", &fp8_scale_update);
  m.def("conv_weight_prep(Tensor w) -> (Tensor, Tensor)", &conv_weight_prep);
  m.def("conv_wgrad_unpack(Tensor dw, int Co, int Ci, int k) -> Tensor", &conv_wgrad_unpack);
  m.def("bn_forward(Tensor x, Tensor? res, Tensor gamma, Tensor beta, Tensor(a!)? run_mean, Tensor(b!)? run_var, Tensor(c!) mean, Tensor(d!) invstd, Tensor(e!) sums, Tensor(f!) y, float momentum, float eps, bool relu) -> ()", &bn_forward);
  m.def("bn_backward(Tensor dy, Tensor x, Tensor y, Tensor mean, Tensor invstd, Tensor gamma, Tensor(a!) sums, Tensor(b!) dx, Tensor(c!)? dres, bool relu) -> ()", &bn_backward);
  m.def("avgpool_forward(Tensor x, Tensor(a!) out, int B, int HW, int C) -> ()", &avgpool_forward);
  m.def("avgpool_backward(Tensor dout, Tensor(a!) dx, int B, int HW, int C) -> ()", &avgpool_backward);
  m.def("umma_shift_probe(Tensor A, Tensor Bm, int CK, int shift_rows, int mode) -> Tensor", &umma_shift_probe);
  m.def("conv_weight_relayout(Tensor shadow, Tensor table, Tensor(a!) Wf, Tensor(b!) Wd, int l0=0, int l1=-1, bool spack0=False) -> ()", &conv_weight_relayout);
  m.def("conv_grad_finalize(Tensor(a!) dW32, Tensor table, Tensor(b!) grad, int l0=0, int l1=-1) -> ()", &conv_grad_finalize);
}
