// Host-callable entry points of the single-GPU kernels (optimizer, losses, norms, linears).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "common.h"

namespace b200 {

// ---------------- multi-tensor optimizer (optim.cu) ------------------------------------------
constexpr int kMaxOptTensors = 120;
constexpr int kOptChunk = 8192;   // elements per block

struct OptSlot {
  void* p;              // model parameter (fp32 or bf16)
  const void* g;        // gradient (fp32 or bf16), may live anywhere (stolen autograd buffer or bucket view)
  unsigned long long flat_off;  // element offset into the flat fp32 master / momentum buffers
  uint32_t numel;
  uint32_t blk0;        // first block of this tensor inside the launch
};
struct OptTable {
  int count;
  int total_blocks;
  OptSlot t[kMaxOptTensors];
};
struct SgdHyper {
  const float* lr;          // device scalar: never baked into a CUDA graph
  const float* clip_coef;   // device scalar from clip_coef kernel (nullptr = 1)
  float* master;            // flat fp32 master weights (nullptr when params are fp32)
  float* momentum_buf;      // flat fp32 (nullptr when momentum == 0)
  const int* step_count;    // device scalar; 0 on the first step (momentum buffer init)
  float momentum, dampening, weight_decay, grad_scale;
  int nesterov;
  int zero_grad;            // write zeros back into g after use
};

void launch_multi_sqnorm(const OptTable& tab, DType g_dtype, float* partials /*[total_blocks]*/, cudaStream_t s);
void launch_clip_coef(const float* partials, int n, float max_norm, float grad_scale, float* coef_out,
                      float* norm_out, cudaStream_t s);
void launch_multi_sgd(const OptTable& tab, DType p_dtype, DType g_dtype, const SgdHyper& h, cudaStream_t s);
void launch_scale_inplace(float* x, size_t n, const float* scalar, cudaStream_t s);

// ---------------- losses (loss.cu) --------------------------------------------------------------
// MSE: loss = mean((o-t)^2) ; dO = 2 (o-t) / N * gscale      (reference criterion, ddp.py:164)
void launch_mse_fwd_bwd(const void* out, const void* target, DType dt, size_t n, float gscale,
                        float* loss /*1*/, void* dout, float* scratch /*[blocks+1]*/, int blocks, cudaStream_t s);
int mse_blocks(size_t n);
// Softmax cross-entropy over rows: loss = mean_i(lse_i - x[i, t_i]); dX = (softmax - onehot)/rows*gscale
void launch_xent_fwd_bwd(const void* logits, const long long* targets, DType dt, int rows, int cols,
                         long long ignore_index, float gscale, float* row_loss /*[rows+1]*/, float* loss /*1*/,
                         void* dlogits, cudaStream_t s);

// GELU (erf) forward: out = gelu(pre); backward: out = dy * gelu'(pre).  One vectorised pass each (loss.cu).
void launch_gelu(const void* pre, const void* dy, void* out, DType dt, size_t n, bool backward, cudaStream_t s);

// ---------------- layer norm (layernorm.cu) -----------------------------------------------------
void launch_layernorm_fwd(const void* x, const void* gamma, const void* beta, DType dt, int rows, int cols,
                          float eps, void* y, float* mean, float* rstd, cudaStream_t s);
void launch_layernorm_bwd(const void* dy, const void* x, const void* gamma, const float* mean, const float* rstd,
                          DType dt, int rows, int cols, void* dx, float* dgamma_partial, float* dbeta_partial,
                          int partial_rows, void* dgamma, void* dbeta, cudaStream_t s);
int layernorm_partial_rows(int rows);

// ---------------- small linears on CUDA cores (linear_small.cu) ------------------------------
// y[M,N] = act(x[M,K] w[N,K]^T + b[N]) ; fp32, dims far below one tensor-core tile (FooModel).
void launch_small_linear_fwd(const float* x, const float* w, const float* b, float* y, int M, int N, int K,
                             int relu, cudaStream_t s);
void launch_small_linear_bwd(const float* dy, const float* x, const float* w, const float* y, float* dx,
                             float* dw, float* db, int M, int N, int K, int relu, int accumulate, cudaStream_t s);

// ---------------- fused training BatchNorm (+residual) (+ReLU), channels_last (batchnorm.cu) --------------
// x viewed as row-major [R = N*H*W, C]; C % 8 == 0; gamma/beta/statistics fp32.
void bn_workspace_sizes(int R, int C, size_t* partial_floats, size_t* counters);
void launch_bn_forward(const void* x, const void* residual, void* y, unsigned char* relu_mask /*[R, C/8] or null*/, DType dt, int R, int C, const float* gamma, const float* beta,
                       float* running_mean, float* running_var, long long* num_batches, float* save_mean, float* save_rstd,
                       float* scale, float* shift, float* partial, unsigned int* counters, float eps, float momentum, bool relu,
                       cudaStream_t s);
// Same as launch_bn_forward, but the statistics come from `partial` = [2][groups][C] partial column sums / sums of squares
// (written by the GEMM epilogue that produced x): finish kernel + apply kernel, x is read once instead of twice.
void launch_bn_forward_from_partials(const void* x, const void* residual, void* y, unsigned char* relu_mask, DType dt, int R, int C,
                                     const float* gamma, const float* beta, float* running_mean, float* running_var,
                                     long long* num_batches, float* save_mean, float* save_rstd, const float* partial, int groups,
                                     float eps, float momentum, bool relu, cudaStream_t s);
// Backward with S1 / S2 partial sums ([2][groups][C]) from the data-gradient epilogue of the consuming convolution: one launch
// (reduce the partials per block, apply), no pass over dy and x for the reduction.
void launch_bn_backward_from_partials(const void* dy, const void* x, const void* relu_mask, void* dx, void* dres, DType dt, int R, int C, const float* gamma,
                                      const float* save_mean, const float* save_rstd, float* dgamma, float* dbeta, const float* partial, int groups,
                                      bool relu, cudaStream_t s);
void launch_bn_backward(const void* dy, const void* x, const void* relu_mask, void* dx, void* dres, DType dt, int R, int C, const float* gamma,
                        const float* save_mean, const float* save_rstd, float* dgamma, float* dbeta, float* coef, float* partial,
                        unsigned int* counters, bool relu, cudaStream_t s);

// ---------------- 3x3/s2/p1 max pooling, channels_last (pool.cu) ------------------------------------------
void launch_maxpool3x3s2_fwd(const void* x, void* y, unsigned char* idx, DType dt, int N, int H, int W, int C, cudaStream_t s);
void launch_maxpool3x3s2_bwd(const void* dy, const unsigned char* idx, void* dx, DType dt, int N, int H, int W, int C, cudaStream_t s);

// ---------------- input pipeline (input.cu) -----------------------------------------------------
// NCHW (u8 or fp32) -> NHWC-in-memory (channels_last) bf16/fp32 with per-channel (x*scale - mean)/std
void launch_normalize_to_channels_last(const void* src, DType src_dt, void* dst, DType dst_dt, int n, int c, int c_out,
                                       int h, int w, const float* mean, const float* inv_std, float in_scale,
                                       cudaStream_t s);

}  // namespace b200
