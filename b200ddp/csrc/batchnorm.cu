// Fused training BatchNorm (+ residual add) (+ ReLU) for channels_last activations.
//
// Why: in the ResNet-50 bf16 step the stock path (ATen batch_norm_collect_statistics / transform_input /
// backward_reduce / backward_elemt + separate ReLU, residual-add and threshold_backward kernels + per-layer
// num_batches_tracked / running-stat updates) is 58% of all kernel time (profiles/launches_graph.md) and runs
// ~16x below the HBM roofline at batch 32.  A [N,C,H,W] channels_last tensor is a row-major [R = N*H*W, C]
// matrix, so every per-channel quantity is a column reduction:
//
//   forward : bn_stats      column sum / sum-of-squares -> mean, rstd, scale = gamma*rstd, shift = beta - mean*scale,
//                           running statistics and num_batches_tracked updated by the last block (deterministic)
//             bn_apply      y = relu(x*scale + shift + residual)            one pass, 16-byte accesses
//   backward: bn_bwd_reduce sum(dy*), sum(dy* * xhat); the ReLU mask is a 1-bit/element bitmap written by bn_apply
//                           (1/16 of re-reading y in bf16, twice); dgamma/dbeta
//             bn_bwd_apply  dx = scale*(dy* - mean(dy*) - xhat*mean(dy* xhat)), and the residual branch's grad
//
// Threads own 8 consecutive channels (one 16-byte vector of bf16); rows are strided across the block and
// across gridDim.y "row splits"; partial sums land in a [splits, C] workspace and the last block of each
// channel tile finishes the reduction in a fixed order (no float atomics -> bitwise reproducible).
#include "ops.h"

namespace b200 {
namespace {

constexpr int kBnThreads = 256;
constexpr int kVec = 8;              // channels per thread

template <typename T> __device__ __forceinline__ void bn_load8(const T* p, float* f);
template <> __device__ __forceinline__ void bn_load8<__nv_bfloat16>(const __nv_bfloat16* p, float* f) {
  unpack8(*reinterpret_cast<const Bf16x8*>(p), f);
}
template <> __device__ __forceinline__ void bn_load8<float>(const float* p, float* f) {
  const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
template <typename T> __device__ __forceinline__ void bn_store8(T* p, const float* f);
template <> __device__ __forceinline__ void bn_store8<__nv_bfloat16>(__nv_bfloat16* p, const float* f) {
  *reinterpret_cast<Bf16x8*>(p) = pack8(f);
}
template <> __device__ __forceinline__ void bn_store8<float>(float* p, const float* f) {
  reinterpret_cast<float4*>(p)[0] = make_float4(f[0], f[1], f[2], f[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(f[4], f[5], f[6], f[7]);
}

struct Tile {
  int cvb;       // channel vectors handled by a block (threads along x)
  int ty;        // rows handled per block iteration
  int grid_x;    // channel tiles
  int grid_y;    // row splits
};

// Where a thread works in every kernel below: column tx of its block's cvb channel vectors (global channel vector cv, i.e.
// channels cv*8 .. cv*8+7) and row lane tyi of ty.
struct BnThread {
  int tx, tyi, cv;
};
__device__ __forceinline__ BnThread bn_thread(int cvb) {
  BnThread t;
  t.tx = threadIdx.x % cvb;
  t.tyi = threadIdx.x / cvb;
  t.cv = blockIdx.x * cvb + t.tx;
  return t;
}

// Rows [x, y) of R: this block's share of the gridDim.y row splits.
__device__ __forceinline__ int2 bn_row_split(int R) {
  const int S = gridDim.y;
  const int rows_per = (R + S - 1) / S;
  const int r0 = blockIdx.y * rows_per;
  return make_int2(r0, min(R, r0 + rows_per));
}

// Block-level reduction over the `ty` row-lanes of two 8-wide accumulators; result valid for threads with row-lane 0.
template <int NACC>
__device__ __forceinline__ void reduce_rows(float (*acc)[kVec], float* smem, int tx, int tyi, int cvb, int ty) {
  // smem layout: [NACC][ty][cvb*8]
  const int width = cvb * kVec;
#pragma unroll
  for (int a = 0; a < NACC; ++a)
#pragma unroll
    for (int i = 0; i < kVec; ++i) smem[(a * ty + tyi) * width + tx * kVec + i] = acc[a][i];
  __syncthreads();
  for (int idx = threadIdx.x; idx < NACC * width; idx += blockDim.x) {
    const int a = idx / width, c = idx % width;
    float s = 0.f;
    for (int r = 0; r < ty; ++r) s += smem[(a * ty + r) * width + c];
    smem[(a * ty) * width + c] = s;       // row-lane 0 slot now holds the block total
  }
  __syncthreads();
}

// Finishes a two-sum column reduction across the gridDim.y row splits of a channel tile, deterministically (no float atomics).
// Every block publishes its totals, left in smem by reduce_rows<2>, to partial = [2][S][C] and takes a ticket on its tile's
// counter.  The last block to arrive sums the S partials in a fixed order and calls epilogue(ch, s, q, 1/R) once per channel
// of the tile.  Returns true in that block only; after a __syncthreads it must reset counters[blockIdx.x] to 0 for the next
// launch (graph replay safe).
template <typename Epilogue>
__device__ __forceinline__ bool bn_finish_tile(float* __restrict__ partial, unsigned int* __restrict__ counters, float* smem, int R, int C,
                                               int cvb, int ty, Epilogue epilogue) {
  __shared__ bool is_last;
  const int S = gridDim.y;
  const int width = cvb * kVec;
  const int c0 = blockIdx.x * width;
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    if (c0 + c < C) {
      partial[(size_t)(0 * S + blockIdx.y) * C + c0 + c] = smem[c];
      partial[(size_t)(1 * S + blockIdx.y) * C + c0 + c] = smem[ty * width + c];
    }
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int ticket = atomicAdd(&counters[blockIdx.x], 1u);
    is_last = (ticket == (unsigned int)S - 1);
  }
  __syncthreads();
  if (!is_last) return false;
  __threadfence();
  const float inv_r = 1.f / (float)R;
  // `lanes` threads per channel each sum a strided subset of the S partials (independent loads in flight),
  // then a fixed-order combine through shared memory
  const int lanes = max(1, (int)blockDim.x / width);
  {
    const int c = threadIdx.x % width, l = threadIdx.x / width;
    float ps = 0.f, pq = 0.f;
    if (l < lanes && c0 + c < C) {
#pragma unroll 4
      for (int k = l; k < S; k += lanes) { ps += __ldcg(&partial[(size_t)(0 * S + k) * C + c0 + c]); pq += __ldcg(&partial[(size_t)(1 * S + k) * C + c0 + c]); }
    }
    __syncthreads();
    if (l < lanes) { smem[l * width + c] = ps; smem[(lanes + l) * width + c] = pq; }
    __syncthreads();
  }
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    const int ch = c0 + c;
    if (ch >= C) continue;
    float s = 0.f, q = 0.f;
    for (int l = 0; l < lanes; ++l) { s += smem[l * width + c]; q += smem[(lanes + l) * width + c]; }
    epilogue(ch, s, q, inv_r);
  }
  return true;
}

// Block totals of this thread's 8 channels over the G rows of partial = [2][G][C] (rows strided over the row lanes, then
// reduce_rows<2>): the first sums land at smem[tx*8 + i], the second at smem[ty*width + tx*8 + i].
__device__ __forceinline__ void bn_reduce_partials(const float* __restrict__ partial, int G, int C, bool live, int cv, int tx, int tyi, int cvb,
                                                   int ty, float* smem) {
  float acc[2][kVec];
#pragma unroll
  for (int i = 0; i < kVec; ++i) { acc[0][i] = 0.f; acc[1][i] = 0.f; }
  if (live) {
    for (int g = tyi; g < G; g += ty) {
      float a[kVec], b[kVec];
      bn_load8<float>(partial + (size_t)g * C + cv * kVec, a);
      bn_load8<float>(partial + ((size_t)G + g) * C + cv * kVec, b);
#pragma unroll
      for (int i = 0; i < kVec; ++i) { acc[0][i] += a[i]; acc[1][i] += b[i]; }
    }
  }
  reduce_rows<2>(acc, smem, tx, tyi, cvb, ty);
}

// ------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kBnThreads, 2) bn_stats_kernel(const T* __restrict__ x, int R, int C, int cvb, int ty,
                                                             float* __restrict__ partial /*[2][S][C]*/, unsigned int* __restrict__ counters,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             float* __restrict__ running_mean, float* __restrict__ running_var,
                                                             long long* __restrict__ num_batches, float* __restrict__ save_mean,
                                                             float* __restrict__ save_rstd, float* __restrict__ scale, float* __restrict__ shift,
                                                             float eps, float momentum) {
  extern __shared__ float smem[];
  const auto [tx, tyi, cv] = bn_thread(cvb);
  const auto [r0, r1] = bn_row_split(R);
  float acc[2][kVec];
#pragma unroll
  for (int i = 0; i < kVec; ++i) { acc[0][i] = 0.f; acc[1][i] = 0.f; }
  if (cv * kVec < C) {
    const T* base = x + (size_t)cv * kVec;
    int r = r0 + tyi;
    for (; r + 3 * ty < r1; r += 4 * ty) {              // 4 independent 16-byte loads in flight
      float f[4][kVec];
#pragma unroll
      for (int u = 0; u < 4; ++u) bn_load8<T>(base + (size_t)(r + u * ty) * C, f[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int i = 0; i < kVec; ++i) { acc[0][i] += f[u][i]; acc[1][i] = fmaf(f[u][i], f[u][i], acc[1][i]); }
    }
    for (; r < r1; r += ty) {
      float f[kVec];
      bn_load8<T>(base + (size_t)r * C, f);
#pragma unroll
      for (int i = 0; i < kVec; ++i) { acc[0][i] += f[i]; acc[1][i] = fmaf(f[i], f[i], acc[1][i]); }
    }
  }
  reduce_rows<2>(acc, smem, tx, tyi, cvb, ty);
  const auto epilogue = [&](int ch, float s, float q, float inv_r) {
    const float mean = s * inv_r;
    const float var = fmaxf(q * inv_r - mean * mean, 0.f);     // biased variance (normalisation)
    const float rstd = rsqrtf(var + eps);
    const float sc = gamma[ch] * rstd;
    save_mean[ch] = mean;
    save_rstd[ch] = rstd;
    scale[ch] = sc;
    shift[ch] = beta[ch] - mean * sc;
    if (running_mean != nullptr) {
      const float unbiased = R > 1 ? var * ((float)R / (float)(R - 1)) : var;
      running_mean[ch] = (1.f - momentum) * running_mean[ch] + momentum * mean;
      running_var[ch] = (1.f - momentum) * running_var[ch] + momentum * unbiased;
    }
  };
  if (!bn_finish_tile(partial, counters, smem, R, C, cvb, ty, epilogue)) return;
  __syncthreads();
  if (threadIdx.x == 0) {
    counters[blockIdx.x] = 0u;                                 // ready for the next launch (graph replay safe)
    if (blockIdx.x == 0 && num_batches != nullptr) *num_batches += 1;
  }
}

template <typename T>
__device__ __forceinline__ void bn_apply_rows(const T* __restrict__ x, const T* __restrict__ residual, T* __restrict__ y,
                                              unsigned char* __restrict__ mask, const float* __restrict__ scale,
                                              const float* __restrict__ shift, int C, int cv, int r0, int r1, int tyi, int ty, int relu) {
  float sc[kVec], sh[kVec];                       // per-channel constants stay in registers for the whole row loop
  bn_load8<float>(scale + cv * kVec, sc);
  bn_load8<float>(shift + cv * kVec, sh);
  const size_t col = (size_t)cv * kVec;
  int r = r0 + tyi;
  for (; r + 3 * ty < r1; r += 4 * ty) {
    float f[4][kVec], rs[4][kVec];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      bn_load8<T>(x + (size_t)(r + u * ty) * C + col, f[u]);
      if (residual != nullptr) bn_load8<T>(residual + (size_t)(r + u * ty) * C + col, rs[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      unsigned int bits = 0;
#pragma unroll
      for (int i = 0; i < kVec; ++i) {
        float v = fmaf(f[u][i], sc[i], sh[i]);
        if (residual != nullptr) v += rs[u][i];
        bits |= (v > 0.f ? 1u : 0u) << i;
        f[u][i] = relu ? fmaxf(v, 0.f) : v;
      }
      bn_store8<T>(y + (size_t)(r + u * ty) * C + col, f[u]);
      if (mask != nullptr) mask[(size_t)(r + u * ty) * (C / kVec) + cv] = (unsigned char)bits;
    }
  }
  for (; r < r1; r += ty) {
    float f[kVec], rs[kVec];
    bn_load8<T>(x + (size_t)r * C + col, f);
    if (residual != nullptr) bn_load8<T>(residual + (size_t)r * C + col, rs);
    unsigned int bits = 0;
#pragma unroll
    for (int i = 0; i < kVec; ++i) {
      float v = fmaf(f[i], sc[i], sh[i]);
      if (residual != nullptr) v += rs[i];
      bits |= (v > 0.f ? 1u : 0u) << i;
      f[i] = relu ? fmaxf(v, 0.f) : v;
    }
    bn_store8<T>(y + (size_t)r * C + col, f);
    if (mask != nullptr) mask[(size_t)r * (C / kVec) + cv] = (unsigned char)bits;
  }
}

template <typename T>
__global__ void __launch_bounds__(kBnThreads) bn_apply_kernel(const T* __restrict__ x, const T* __restrict__ residual, T* __restrict__ y,
                                                             unsigned char* __restrict__ mask, const float* __restrict__ scale,
                                                             const float* __restrict__ shift, int R, int C, int cvb, int ty, int relu) {
  const auto [tx, tyi, cv] = bn_thread(cvb);
  if (cv * kVec >= C) return;
  const auto [r0, r1] = bn_row_split(R);
  bn_apply_rows<T>(x, residual, y, mask, scale, shift, C, cv, r0, r1, tyi, ty, relu);
}

// ------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kBnThreads, 2) bn_bwd_reduce_kernel(const T* __restrict__ dy, const T* __restrict__ x, const unsigned char* __restrict__ y,
                                                                     int R, int C, int cvb, int ty, int relu, const float* __restrict__ save_mean,
                                                                     const float* __restrict__ save_rstd, float* __restrict__ partial,
                                                                     unsigned int* __restrict__ counters, float* __restrict__ dgamma,
                                                                     float* __restrict__ dbeta, float* __restrict__ coef /*[2][C]*/) {
  extern __shared__ float smem[];
  const auto [tx, tyi, cv] = bn_thread(cvb);
  const auto [r0, r1] = bn_row_split(R);
  float acc[2][kVec];
#pragma unroll
  for (int i = 0; i < kVec; ++i) { acc[0][i] = 0.f; acc[1][i] = 0.f; }
  if (cv * kVec < C) {
    float mean[kVec], rstd[kVec];
    bn_load8<float>(save_mean + cv * kVec, mean);
    bn_load8<float>(save_rstd + cv * kVec, rstd);
    const size_t col = (size_t)cv * kVec;
    int r = r0 + tyi;
    for (; r + ty < r1; r += 2 * ty) {                  // 2 rows x 3 streams = 6 independent 16-byte loads in flight
      float g[2][kVec], xv[2][kVec];
      unsigned int mk[2] = {0xffu, 0xffu};
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const size_t off = (size_t)(r + u * ty) * C + col;
        bn_load8<T>(dy + off, g[u]);
        bn_load8<T>(x + off, xv[u]);
        if (relu) mk[u] = y[(size_t)(r + u * ty) * (C / kVec) + cv];
      }
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int i = 0; i < kVec; ++i) {
          const float gm = ((mk[u] >> i) & 1u) ? g[u][i] : 0.f;
          acc[0][i] += gm;
          acc[1][i] = fmaf(gm, (xv[u][i] - mean[i]) * rstd[i], acc[1][i]);
        }
    }
    for (; r < r1; r += ty) {
      float g[kVec], xv[kVec];
      const size_t off = (size_t)r * C + col;
      bn_load8<T>(dy + off, g);
      bn_load8<T>(x + off, xv);
      const unsigned int mk = relu ? y[(size_t)r * (C / kVec) + cv] : 0xffu;
#pragma unroll
      for (int i = 0; i < kVec; ++i) {
        const float gm = ((mk >> i) & 1u) ? g[i] : 0.f;
        acc[0][i] += gm;
        acc[1][i] = fmaf(gm, (xv[i] - mean[i]) * rstd[i], acc[1][i]);
      }
    }
  }
  reduce_rows<2>(acc, smem, tx, tyi, cvb, ty);
  const auto epilogue = [&](int ch, float s, float q, float inv_r) {
    dbeta[ch] = s;
    dgamma[ch] = q;
    coef[ch] = s * inv_r;            // mean(dy*)
    coef[C + ch] = q * inv_r;        // mean(dy* xhat)
  };
  if (!bn_finish_tile(partial, counters, smem, R, C, cvb, ty, epilogue)) return;
  __syncthreads();
  if (threadIdx.x == 0) counters[blockIdx.x] = 0u;
}

// c1p / c2p point at THIS thread's 8 coefficients (global coef rows or a block's shared-memory copy)
template <typename T>
__device__ __forceinline__ void bn_bwd_apply_rows_coef(const T* __restrict__ dy, const T* __restrict__ x, const unsigned char* __restrict__ y,
                                                       T* __restrict__ dx, T* __restrict__ dres, const float* __restrict__ save_mean,
                                                       const float* __restrict__ save_rstd, const float* __restrict__ gamma,
                                                       const float* c1p, const float* c2p, int C, int cv, int r0, int r1, int tyi, int ty, int relu) {
  // dx = a*dy* + b*x + c  with per-channel a = gamma*rstd, b = -a*rstd*c2, c = -a*(c1 - mean*rstd*c2)
  float ka[kVec], kb[kVec], kc[kVec];
  {
    float mean[kVec], rstd[kVec], gam[kVec], c1[kVec], c2[kVec];
    bn_load8<float>(save_mean + cv * kVec, mean);
    bn_load8<float>(save_rstd + cv * kVec, rstd);
    bn_load8<float>(gamma + cv * kVec, gam);
    bn_load8<float>(c1p, c1);
    bn_load8<float>(c2p, c2);
#pragma unroll
    for (int i = 0; i < kVec; ++i) {
      ka[i] = gam[i] * rstd[i];
      kb[i] = -ka[i] * rstd[i] * c2[i];
      kc[i] = -ka[i] * (c1[i] - mean[i] * rstd[i] * c2[i]);
    }
  }
  const size_t col = (size_t)cv * kVec;
  int r = r0 + tyi;
  for (; r + ty < r1; r += 2 * ty) {                    // 2 rows x 3 streams in flight
    float g[2][kVec], xv[2][kVec];
    unsigned int mk[2] = {0xffu, 0xffu};
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const size_t off = (size_t)(r + u * ty) * C + col;
      bn_load8<T>(dy + off, g[u]);
      bn_load8<T>(x + off, xv[u]);
      if (relu) mk[u] = y[(size_t)(r + u * ty) * (C / kVec) + cv];
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const size_t off = (size_t)(r + u * ty) * C + col;
      float o[kVec];
#pragma unroll
      for (int i = 0; i < kVec; ++i) {
        if (!((mk[u] >> i) & 1u)) g[u][i] = 0.f;
        o[i] = fmaf(ka[i], g[u][i], fmaf(kb[i], xv[u][i], kc[i]));
      }
      if (dres != nullptr) bn_store8<T>(dres + off, g[u]);          // gradient of the residual branch = masked dy
      bn_store8<T>(dx + off, o);
    }
  }
  for (; r < r1; r += ty) {
    const size_t off = (size_t)r * C + col;
    float g[kVec], xv[kVec], o[kVec];
    bn_load8<T>(dy + off, g);
    bn_load8<T>(x + off, xv);
    const unsigned int mk = relu ? y[(size_t)r * (C / kVec) + cv] : 0xffu;
#pragma unroll
    for (int i = 0; i < kVec; ++i) {
      if (!((mk >> i) & 1u)) g[i] = 0.f;
      o[i] = fmaf(ka[i], g[i], fmaf(kb[i], xv[i], kc[i]));
    }
    if (dres != nullptr) bn_store8<T>(dres + off, g);
    bn_store8<T>(dx + off, o);
  }
}

template <typename T>
__global__ void __launch_bounds__(kBnThreads) bn_bwd_apply_kernel(const T* __restrict__ dy, const T* __restrict__ x, const unsigned char* __restrict__ y,
                                                                 T* __restrict__ dx, T* __restrict__ dres, const float* __restrict__ save_mean,
                                                                 const float* __restrict__ save_rstd, const float* __restrict__ gamma,
                                                                 const float* __restrict__ coef, int R, int C, int cvb, int ty, int relu) {
  const auto [tx, tyi, cv] = bn_thread(cvb);
  if (cv * kVec >= C) return;
  const auto [r0, r1] = bn_row_split(R);
  bn_bwd_apply_rows_coef<T>(dy, x, y, dx, dres, save_mean, save_rstd, gamma, coef + cv * kVec, coef + C + cv * kVec, C, cv, r0, r1, tyi, ty, relu);
}

Tile pick_tile(int R, int C) {
  Tile t;
  const int cv = C / kVec;
  t.cvb = cv < 8 ? cv : 8;                            // <= 64 channels per tile: 128-byte row segments, and the
  while (kBnThreads % t.cvb != 0) --t.cvb;            //    finishing block has >= 4 lanes per channel
  t.ty = kBnThreads / t.cvb;
  t.grid_x = (cv + t.cvb - 1) / t.cvb;
  // enough row splits to put ~4 blocks on every SM, but keep >= 4 row iterations per block
  int want = (4 * kNumSMs + t.grid_x - 1) / t.grid_x;
  int max_by_rows = R / (t.ty * 4);
  if (max_by_rows < 1) max_by_rows = 1;
  t.grid_y = want < max_by_rows ? want : max_by_rows;
  if (t.grid_y > 256) t.grid_y = 256;
  return t;
}

// apply kernels: same channel tiling, row splits sized so each thread sees >= 4 rows but the grid still fills the GPU
dim3 apply_grid(const Tile& t, int R) {
  int want = (8 * kNumSMs + t.grid_x - 1) / t.grid_x;
  int max_by_rows = R / (t.ty * 4);
  if (max_by_rows < 1) max_by_rows = 1;
  int gy = want < max_by_rows ? want : max_by_rows;
  return dim3(t.grid_x, gy);
}

// Calls launch(T()) with T the element type of `dt`: bf16, anything else fp32.
template <typename Launch>
void with_element_type(DType dt, Launch&& launch) {
  if (dt == DType::BF16) launch(__nv_bfloat16());
  else launch(float());
}

}  // namespace

// ------------------------------------------------------------------------------------------------------
// Statistics from the producing convolution's epilogue (csrc/conv_tcgen05.cu): partial = [2][G][C] per-CTA column sums and
// sums of squares, G <= 148.  NO separate finishing launch: every block of the normalisation kernel first reduces the G
// rows of ITS <= 64 channels (a few tens of KB out of L2, fixed order -> deterministic), then normalises its rows; the
// blocks of the first row split also publish mean / rstd (for the backward pass) and update the running statistics.
template <typename T>
__global__ void __launch_bounds__(kBnThreads) bn_apply_partials_kernel(const T* __restrict__ x, const T* __restrict__ residual, T* __restrict__ y,
                                                                      unsigned char* __restrict__ mask, const float* __restrict__ partial, int G,
                                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                      float* __restrict__ running_mean, float* __restrict__ running_var,
                                                                      long long* __restrict__ num_batches, float* __restrict__ save_mean,
                                                                      float* __restrict__ save_rstd, float eps, float momentum, int R, int C,
                                                                      int cvb, int ty, int relu) {
  extern __shared__ float bn_smem[];                 // [2][ty][cvb*8] reduction scratch, then [2][cvb*8] scale / shift
  const auto [tx, tyi, cv] = bn_thread(cvb);
  const bool live = cv * kVec < C;
  bn_reduce_partials(partial, G, C, live, cv, tx, tyi, cvb, ty, bn_smem);
  const int width = cvb * kVec;
  float* sc_s = bn_smem + 2 * ty * width;            // scale / shift of this block's channels
  float* sh_s = sc_s + width;
  if (tyi == 0 && live) {
    const float inv_r = 1.f / (float)R;
#pragma unroll
    for (int i = 0; i < kVec; ++i) {
      const int ch = cv * kVec + i;
      const float sum = bn_smem[tx * kVec + i], sq = bn_smem[ty * width + tx * kVec + i];
      const float mean = sum * inv_r;
      const float var = fmaxf(sq * inv_r - mean * mean, 0.f);
      const float rstd = rsqrtf(var + eps);
      const float sc = gamma[ch] * rstd;
      sc_s[tx * kVec + i] = sc;
      sh_s[tx * kVec + i] = beta[ch] - mean * sc;
      if (blockIdx.y == 0) {
        save_mean[ch] = mean;
        save_rstd[ch] = rstd;
        if (running_mean != nullptr) {
          const float unbiased = R > 1 ? var * ((float)R / (float)(R - 1)) : var;
          running_mean[ch] = (1.f - momentum) * running_mean[ch] + momentum * mean;
          running_var[ch] = (1.f - momentum) * running_var[ch] + momentum * unbiased;
        }
      }
    }
  }
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0 && num_batches != nullptr) *num_batches += 1;
  __syncthreads();
  if (!live) return;
  const auto [r0, r1] = bn_row_split(R);
  // bn_apply_rows indexes scale / shift by the global channel vector: hand it pointers rebased to this block's tile
  bn_apply_rows<T>(x, residual, y, mask, sc_s - (size_t)blockIdx.x * width, sh_s - (size_t)blockIdx.x * width, C, cv, r0, r1, tyi, ty, relu);
}

// Backward twin: partial = [2][G][C] with S1 = sum dy*m and S2 = sum dy*m*xhat from the data-gradient epilogue of the convolution
// that consumes this BatchNorm's output.  Every block reduces its channels' G rows, forms c1 = S1/R, c2 = S2/R, applies
// dx = gamma*rstd*(dy*m - c1 - xhat*c2); the first row split also writes dgamma = S2, dbeta = S1.
template <typename T>
__global__ void __launch_bounds__(kBnThreads) bn_bwd_apply_partials_kernel(const T* __restrict__ dy, const T* __restrict__ x, const unsigned char* __restrict__ y,
                                                                          T* __restrict__ dx, T* __restrict__ dres, const float* __restrict__ partial, int G,
                                                                          const float* __restrict__ save_mean, const float* __restrict__ save_rstd,
                                                                          const float* __restrict__ gamma, float* __restrict__ dgamma,
                                                                          float* __restrict__ dbeta, int R, int C, int cvb, int ty, int relu) {
  extern __shared__ float bn_smem[];                 // [2][ty][cvb*8] reduction scratch, then [2][cvb*8] coefficients
  const auto [tx, tyi, cv] = bn_thread(cvb);
  const bool live = cv * kVec < C;
  bn_reduce_partials(partial, G, C, live, cv, tx, tyi, cvb, ty, bn_smem);
  const int width = cvb * kVec;
  float* c1_s = bn_smem + 2 * ty * width;            // c1 / c2 of this block's channels
  float* c2_s = c1_s + width;
  if (tyi == 0 && live) {
    const float inv_r = 1.f / (float)R;
#pragma unroll
    for (int i = 0; i < kVec; ++i) {
      const int ch = cv * kVec + i;
      const float s1 = bn_smem[tx * kVec + i], s2 = bn_smem[ty * width + tx * kVec + i];
      c1_s[tx * kVec + i] = s1 * inv_r;
      c2_s[tx * kVec + i] = s2 * inv_r;
      if (blockIdx.y == 0) { dgamma[ch] = s2; dbeta[ch] = s1; }
    }
  }
  __syncthreads();
  if (!live) return;
  const auto [r0, r1] = bn_row_split(R);
  bn_bwd_apply_rows_coef<T>(dy, x, y, dx, dres, save_mean, save_rstd, gamma, c1_s + tx * kVec, c2_s + tx * kVec, C, cv, r0, r1, tyi, ty, relu);
}

void bn_workspace_sizes(int R, int C, size_t* partial_floats, size_t* counters) {
  const Tile t = pick_tile(R, C);
  *partial_floats = (size_t)2 * t.grid_y * C;
  *counters = (size_t)t.grid_x;              // one self-resetting ticket counter per channel tile
}

void launch_bn_forward(const void* x, const void* residual, void* y, unsigned char* mask, DType dt, int R, int C, const float* gamma, const float* beta,
                       float* running_mean, float* running_var, long long* num_batches, float* save_mean, float* save_rstd,
                       float* scale, float* shift, float* partial, unsigned int* counters, float eps, float momentum, bool relu,
                       cudaStream_t s) {
  if (C % kVec != 0) throw std::runtime_error("fused batch norm: channel count must be a multiple of 8");
  const Tile t = pick_tile(R, C);
  const size_t smem = (size_t)2 * t.ty * t.cvb * kVec * sizeof(float);
  const int r = relu ? 1 : 0;
  with_element_type(dt, [&](auto elem) {
    using T = decltype(elem);
    bn_stats_kernel<T><<<dim3(t.grid_x, t.grid_y), kBnThreads, smem, s>>>((const T*)x, R, C, t.cvb, t.ty, partial, counters, gamma, beta,
                                                                          running_mean, running_var, num_batches, save_mean, save_rstd,
                                                                          scale, shift, eps, momentum);
    B200_CUDA_CHECK(cudaGetLastError()); B200_COUNT_LAUNCH(1);
    bn_apply_kernel<T><<<apply_grid(t, R), kBnThreads, 0, s>>>((const T*)x, (const T*)residual, (T*)y, mask, scale, shift, R, C, t.cvb, t.ty, r);
    B200_CUDA_CHECK(cudaGetLastError()); B200_COUNT_LAUNCH(1);
  });
}

void launch_bn_forward_from_partials(const void* x, const void* residual, void* y, unsigned char* mask, DType dt, int R, int C,
                                     const float* gamma, const float* beta, float* running_mean, float* running_var,
                                     long long* num_batches, float* save_mean, float* save_rstd, const float* partial, int groups,
                                     float eps, float momentum, bool relu, cudaStream_t s) {
  if (C % kVec != 0) throw std::runtime_error("fused batch norm: channel count must be a multiple of 8");
  if (groups < 1) throw std::runtime_error("fused batch norm: empty partial statistics");
  const Tile t = pick_tile(R, C);
  const int r = relu ? 1 : 0;
  const size_t smem = (size_t)(2 * t.ty + 2) * t.cvb * kVec * sizeof(float);
  with_element_type(dt, [&](auto elem) {
    using T = decltype(elem);
    bn_apply_partials_kernel<T><<<apply_grid(t, R), kBnThreads, smem, s>>>((const T*)x, (const T*)residual, (T*)y, mask, partial, groups, gamma,
                                                                           beta, running_mean, running_var, num_batches, save_mean, save_rstd,
                                                                           eps, momentum, R, C, t.cvb, t.ty, r);
    B200_CUDA_CHECK(cudaGetLastError()); B200_COUNT_LAUNCH(1);
  });
}

void launch_bn_backward_from_partials(const void* dy, const void* x, const void* y, void* dx, void* dres, DType dt, int R, int C, const float* gamma,
                                      const float* save_mean, const float* save_rstd, float* dgamma, float* dbeta, const float* partial, int groups,
                                      bool relu, cudaStream_t s) {
  if (C % kVec != 0) throw std::runtime_error("fused batch norm: channel count must be a multiple of 8");
  if (groups < 1) throw std::runtime_error("fused batch norm: empty partial sums");
  const Tile t = pick_tile(R, C);
  const int r = relu ? 1 : 0;
  const size_t smem = (size_t)(2 * t.ty + 2) * t.cvb * kVec * sizeof(float);
  with_element_type(dt, [&](auto elem) {
    using T = decltype(elem);
    bn_bwd_apply_partials_kernel<T><<<apply_grid(t, R), kBnThreads, smem, s>>>((const T*)dy, (const T*)x, (const unsigned char*)y, (T*)dx, (T*)dres,
                                                                               partial, groups, save_mean, save_rstd, gamma, dgamma, dbeta, R, C,
                                                                               t.cvb, t.ty, r);
    B200_CUDA_CHECK(cudaGetLastError()); B200_COUNT_LAUNCH(1);
  });
}

void launch_bn_backward(const void* dy, const void* x, const void* y, void* dx, void* dres, DType dt, int R, int C, const float* gamma,
                        const float* save_mean, const float* save_rstd, float* dgamma, float* dbeta, float* coef, float* partial,
                        unsigned int* counters, bool relu, cudaStream_t s) {
  if (C % kVec != 0) throw std::runtime_error("fused batch norm: channel count must be a multiple of 8");
  const Tile t = pick_tile(R, C);
  const size_t smem = (size_t)2 * t.ty * t.cvb * kVec * sizeof(float);
  const int r = relu ? 1 : 0;
  with_element_type(dt, [&](auto elem) {
    using T = decltype(elem);
    bn_bwd_reduce_kernel<T><<<dim3(t.grid_x, t.grid_y), kBnThreads, smem, s>>>((const T*)dy, (const T*)x, (const unsigned char*)y, R, C, t.cvb, t.ty,
                                                                               r, save_mean, save_rstd, partial, counters, dgamma, dbeta, coef);
    B200_CUDA_CHECK(cudaGetLastError()); B200_COUNT_LAUNCH(1);
    bn_bwd_apply_kernel<T><<<apply_grid(t, R), kBnThreads, 0, s>>>((const T*)dy, (const T*)x, (const unsigned char*)y, (T*)dx, (T*)dres, save_mean,
                                                                   save_rstd, gamma, coef, R, C, t.cvb, t.ty, r);
    B200_CUDA_CHECK(cudaGetLastError()); B200_COUNT_LAUNCH(1);
  });
}

}  // namespace b200
