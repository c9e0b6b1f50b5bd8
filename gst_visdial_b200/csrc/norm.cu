// Fused normalisation / embedding / elementwise kernels (HBM-bound; one warp per row, 128-bit accesses, fp32 math).
//
//   add_layernorm   : y = LN(x + residual)            models/vilbert_dialog.py:283-296 used at :413,:455,:540,:582,:719,:726
//   embed_text      : y = LN(word[id]+pos[p]+type[s])  models/vilbert_dialog.py:324-352
//   image_embed_ln  : y = LN(x + loc*Wloc^T + bloc)    models/vilbert_dialog.py:1420-1427 (x = image_embeddings GEMM)
//   concat_fused    : cat(fc_v(v), fc_l(t)) + masks    models/visual_dialog_model.py:131-135
//   relu_mul        : relu(a) * relu(b)                models/vilbert_dialog.py:921-941,1030-1033
// LayerNorm is the TF-style one the reference uses: biased variance, eps = 1e-12 inside the sqrt, division (not rsqrt).
#include <stdexcept>

#include "common.cuh"
#include "kernels.h"

namespace gstvd {

namespace {

constexpr int kMaxChunks = 4;        // 4 chunks x 32 lanes x 8 elements = width <= 1024
constexpr float kLnEps = 1e-12f;
constexpr int kRowsPerBlock = 4;

// Normalises the per-lane register tile v (chunk c covers columns (lane + 32*c)*8 .. +8) and stores it.
template <typename T>
__device__ __forceinline__ void ln_finish(float (&v)[kMaxChunks][8], int width, int lane, const float* __restrict__ gamma,
                                          const float* __restrict__ beta, T* __restrict__ y) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c)
    if ((lane + 32 * c) * 8 < width)
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[c][j];
  const float mean = warp_sum(s) / (float)width;
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c)
    if ((lane + 32 * c) * 8 < width)
#pragma unroll
      for (int j = 0; j < 8; ++j) { float d = v[c][j] - mean; q += d * d; }
  const float var = warp_sum(q) / (float)width;
  const float denom = sqrtf(var + kLnEps);
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) {
      float g[8], b[8], o[8];
      Vec8<float>::load(gamma + col, g);
      Vec8<float>::load(beta + col, b);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = g[j] * ((v[c][j] - mean) / denom) + b[j];
      Vec8<T>::store(y + col, o);
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(kRowsPerBlock * 32)
add_layernorm_kernel(int rows, int width, const T* __restrict__ x, int64_t ldx, const T* __restrict__ res, int64_t ldr,
                     const float* __restrict__ gamma, const float* __restrict__ beta, T* __restrict__ y, int64_t ldy) {
  const int row = blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  // gamma / beta are weights: they do not depend on the previous kernel, so they are fetched before the PDL wait
  float g[kMaxChunks][8], b[kMaxChunks][8];
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) { Vec8<float>::load(gamma + col, g[c]); Vec8<float>::load(beta + col, b[c]); }
  }
  pdl_wait();
  pdl_launch_dependents();
  if (row >= rows) return;
  float v[kMaxChunks][8];
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) {
      Vec8<T>::load(x + (int64_t)row * ldx + col, v[c]);
      if (res != nullptr) {
        float r[8];
        Vec8<T>::load(res + (int64_t)row * ldr + col, r);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[c][j] += r[j];
      }
    }
  }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c)
    if ((lane + 32 * c) * 8 < width)
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[c][j];
  const float mean = warp_sum(s) / (float)width;
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c)
    if ((lane + 32 * c) * 8 < width)
#pragma unroll
      for (int j = 0; j < 8; ++j) { float d = v[c][j] - mean; q += d * d; }
  const float var = warp_sum(q) / (float)width;
  const float denom = sqrtf(var + kLnEps);
  T* yrow = y + (int64_t)row * ldy;
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = g[c][j] * ((v[c][j] - mean) / denom) + b[c][j];
      Vec8<T>::store(yrow + col, o);
    }
  }
}

// Large row counts (encoder: 16 384 x 768): warps loop over rows, gamma / beta come from L1 at normalise time instead of
// living in registers, so 32 warps per SM are resident and enough loads are in flight to approach the HBM rate.
constexpr int kStreamWarps = 8;
template <typename T>
__global__ void __launch_bounds__(kStreamWarps * 32, 4)
add_layernorm_stream_kernel(int rows, int width, const T* __restrict__ x, int64_t ldx, const T* __restrict__ res, int64_t ldr,
                            const float* __restrict__ gamma, const float* __restrict__ beta, T* __restrict__ y, int64_t ldy) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const int stride = gridDim.x * kStreamWarps;
  for (int row = blockIdx.x * kStreamWarps + (threadIdx.x >> 5); row < rows; row += stride) {
    float v[kMaxChunks][8];
#pragma unroll
    for (int c = 0; c < kMaxChunks; ++c) {
      const int col = (lane + 32 * c) * 8;
      if (col < width) {
        Vec8<T>::load(x + (int64_t)row * ldx + col, v[c]);
        if (res != nullptr) {
          float r[8];
          Vec8<T>::load(res + (int64_t)row * ldr + col, r);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[c][j] += r[j];
        }
      }
    }
    ln_finish<T>(v, width, lane, gamma, beta, y + (int64_t)row * ldy);
  }
}

template <typename T>
__global__ void __launch_bounds__(kRowsPerBlock * 32)
embed_text_kernel(int rows, int L, int width, const int64_t* __restrict__ ids, const int64_t* __restrict__ seg,
                  const int* __restrict__ d_pos_offset, int eos_to_pad, const float* __restrict__ word,
                  const float* __restrict__ pos, const float* __restrict__ type, const float* __restrict__ type_ext,
                  int type_vocab, const float* __restrict__ gamma, const float* __restrict__ beta, T* __restrict__ y) {
  const int row = blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  int64_t id = ids[row];
  if (eos_to_pad && (id == 102 || id < 0)) id = 0;   // negative: past the end of a shorter decoder prefix
  const int p = (row % L) + (d_pos_offset ? *d_pos_offset : 0);
  const int64_t s = seg ? seg[row] : 0;
  // segments >= type_vocab_size index the "extension" table (models/vilbert_dialog.py:335-346)
  const float* trow = (s < type_vocab) ? type + s * width : type_ext + (s - type_vocab) * width;
  float v[kMaxChunks][8];
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) {
      float a[8], b[8], t[8];
      Vec8<float>::load(word + id * width + col, a);
      Vec8<float>::load(pos + (int64_t)p * width + col, b);
      Vec8<float>::load(trow + col, t);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[c][j] = (a[j] + b[j]) + t[j];
    }
  }
  ln_finish<T>(v, width, lane, gamma, beta, y + (int64_t)row * width);
}

template <typename T>
__global__ void __launch_bounds__(kRowsPerBlock * 32)
embed_step_kernel(int rows, int width, const int32_t* __restrict__ tokens, int pos0, const int* __restrict__ p0s, int rows_per_image,
                  const int* __restrict__ d_step,
                  const float* __restrict__ word, const float* __restrict__ pos, const float* __restrict__ type,
                  const float* __restrict__ gamma, const float* __restrict__ beta, T* __restrict__ y) {
  pdl_wait();
  pdl_launch_dependents();
  const int row = blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  int id = tokens[row];
  if (id == 102) id = 0;      // the decoder never sees [SEP] as an input (models/visual_dialog_decoder.py:57)
  const int p = (p0s ? p0s[row / rows_per_image] : pos0) + *d_step;   // the image's decoder prefix length - 1, plus the step
  float v[kMaxChunks][8];
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) {
      float a[8], b[8], t[8];
      Vec8<float>::load(word + (int64_t)id * width + col, a);
      Vec8<float>::load(pos + (int64_t)p * width + col, b);
      Vec8<float>::load(type + col, t);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[c][j] = (a[j] + b[j]) + t[j];
    }
  }
  ln_finish<T>(v, width, lane, gamma, beta, y + (int64_t)row * width);
}

template <typename T>
__global__ void __launch_bounds__(kRowsPerBlock * 32)
image_embed_ln_kernel(int rows, int width, const T* __restrict__ x, const float* __restrict__ loc,
                      const float* __restrict__ wloc, const float* __restrict__ bloc, const float* __restrict__ gamma,
                      const float* __restrict__ beta, T* __restrict__ y) {
  const int row = blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float l[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) l[i] = loc[(int64_t)row * 5 + i];
  float v[kMaxChunks][8];
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) {
      Vec8<T>::load(x + (int64_t)row * width + col, v[c]);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float* w = wloc + (int64_t)(col + j) * 5;
        float a = bloc[col + j];
#pragma unroll
        for (int i = 0; i < 5; ++i) a = fmaf(l[i], w[i], a);
        v[c][j] += a;
      }
    }
  }
  ln_finish<T>(v, width, lane, gamma, beta, y + (int64_t)row * width);
}

// ---- deferred LayerNorm (decode step, GemmArgs::fold_stats / res_stats / stats_out) ---------------------------------------------
// Weight preparation, once per weight load: W'[n][k] = bf16(W[n][k] gamma[k]); c[n] = sum_k W'[n][k] (of the ROUNDED values: it
// cancels the mean term of what the tensor core actually multiplies); d[n] = sum_k beta[k] W[n][k] + bias[n].  One warp per row n.
__global__ void __launch_bounds__(kRowsPerBlock * 32)
fold_ln_weights_kernel(int N, int K, const float* __restrict__ W, const float* __restrict__ gamma, const float* __restrict__ beta,
                       const float* __restrict__ bias, bf16* __restrict__ Wf, float* __restrict__ c, float* __restrict__ d) {
  const int n = blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  float cs = 0.f, ds = 0.f;
  for (int k = lane * 8; k < K; k += 256) {
    float w[8], g[8], b[8], o[8];
    Vec8<float>::load(W + (int64_t)n * K + k, w);
    Vec8<float>::load(gamma + k, g);
    Vec8<float>::load(beta + k, b);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      o[j] = to_f32(__float2bfloat16_rn(w[j] * g[j]));
      cs += o[j];
      ds = fmaf(b[j], w[j], ds);
    }
    Vec8<bf16>::store(Wf + (int64_t)n * K + k, o);
  }
  cs = warp_sum(cs); ds = warp_sum(ds);
  if (lane == 0) { c[n] = cs; d[n] = ds + (bias ? bias[n] : 0.f); }
}

// y = LN(x) for a raw bf16 row whose statistics were stored by the producing GEMM as per-32-column partials (mean_i, M2_i):
// the one place of a decode step where the normalised tensor is materialised (input of the LM head).  One warp per row.
__global__ void __launch_bounds__(kRowsPerBlock * 32)
ln_apply_stats_kernel(int rows, int width, const bf16* __restrict__ x, const float2* __restrict__ stats, int64_t stats_ld, int parts,
                      const float* __restrict__ gamma, const float* __restrict__ beta, bf16* __restrict__ y) {
  const int row = blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  float g[kMaxChunks][8], b[kMaxChunks][8];
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) { Vec8<float>::load(gamma + col, g[c]); Vec8<float>::load(beta + col, b[c]); }
  }
  pdl_wait();
  pdl_launch_dependents();
  if (row >= rows) return;
  const float2 mine = lane < parts ? stats[(int64_t)lane * stats_ld + row] : make_float2(0.f, 0.f);
  const float mean = warp_sum(mine.x) / (float)parts;            // butterfly order: identical in every lane, deterministic
  const float dv = lane < parts ? mine.x - mean : 0.f;
  const float var = warp_sum(fmaf(32.f * dv, dv, mine.y)) / (32.f * (float)parts);
  const float rstd = 1.0f / sqrtf(var + kLnEpsDeferred);
#pragma unroll
  for (int c = 0; c < kMaxChunks; ++c) {
    const int col = (lane + 32 * c) * 8;
    if (col < width) {
      float v[8], o[8];
      Vec8<bf16>::load(x + (int64_t)row * width + col, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = fmaf((v[j] - mean) * rstd, g[c][j], b[c][j]);
      Vec8<bf16>::store(y + (int64_t)row * width + col, o);
    }
  }
}

template <typename T>
__global__ void cast_from_f32_kernel(const float* __restrict__ src, T* __restrict__ dst, int64_t n) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i + 8 <= n) {
    float v[8];
    Vec8<float>::load(src + i, v);
    Vec8<T>::store(dst + i, v);
  } else {
    for (; i < n; ++i) dst[i] = from_f32<T>(src[i]);
  }
}
template <typename T>
__global__ void cast_to_f32_kernel(const T* __restrict__ src, float* __restrict__ dst, int64_t n) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i + 8 <= n) {
    float v[8];
    Vec8<T>::load(src + i, v);
    Vec8<float>::store(dst + i, v);
  } else {
    for (; i < n; ++i) dst[i] = to_f32(src[i]);
  }
}

template <typename T>
__global__ void copy_rows_kernel(int rows, int width, const T* __restrict__ src, int64_t lds, T* __restrict__ dst, int64_t ldd) {
  const int chunks = width / 8;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)rows * chunks) return;
  const int r = (int)(i / chunks), c = (int)(i % chunks) * 8;
  float v[8];
  Vec8<T>::load(src + (int64_t)r * lds + c, v);
  Vec8<T>::store(dst + (int64_t)r * ldd + c, v);
}

template <typename T>
__global__ void concat_fused_kernel(int B, int Lv, int Lt, int width, const T* __restrict__ v, const T* __restrict__ t,
                                    T* __restrict__ fused, const float* __restrict__ imask, const float* __restrict__ tmask,
                                    float* __restrict__ fmask) {
  const int Le = Lv + Lt, chunks = width / 8;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * Le * chunks) return;
  const int c = (int)(i % chunks) * 8;
  const int64_t r = i / chunks;
  const int b = (int)(r / Le), pos = (int)(r % Le);
  const T* src = (pos < Lv) ? v + ((int64_t)b * Lv + pos) * width : t + ((int64_t)b * Lt + (pos - Lv)) * width;
  float x[8];
  Vec8<T>::load(src + c, x);
  Vec8<T>::store(fused + r * width + c, x);
  if (c == 0 && fmask != nullptr)
    fmask[r] = (pos < Lv) ? (imask ? imask[(int64_t)b * Lv + pos] : 1.f) : (tmask ? tmask[(int64_t)b * Lt + pos - Lv] : 1.f);
}

template <typename T>
__global__ void relu_mul_kernel(int64_t n, const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = from_f32<T>(fmaxf(to_f32(a[i]), 0.f) * fmaxf(to_f32(b[i]), 0.f));
}

template <typename T>
__global__ void gather_first_rows_kernel(int B, int L, int width, const T* __restrict__ src, T* __restrict__ dst) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)B * width) dst[i] = src[(i / width) * (int64_t)L * width + (i % width)];
}

void check_width(int width) {
  if (width % 8 != 0 || width > kMaxChunks * 256) throw std::runtime_error("row kernels need width % 8 == 0 and width <= 1024");
}
inline int grid_rows(int rows) { return (rows + kRowsPerBlock - 1) / kRowsPerBlock; }

}  // namespace

int launch_add_layernorm(int dtype, int rows, int width, const void* x, int64_t ldx, const void* residual, int64_t ldr,
                         const float* gamma, const float* beta, void* y, int64_t ldy, cudaStream_t stream) {
  if (rows <= 0) return 0;
  check_width(width);
  if (rows >= 4096) {
    static const int sms = [] { int d = 0, n = 148; cudaGetDevice(&d); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d); return n; }();
    const int want = (rows + kStreamWarps - 1) / kStreamWarps, cap = sms * 4 * 2;   // two rows per warp per wave at 4 CTAs / SM
    const int grid = want < cap ? want : cap;
    if (dtype == kF32)
      launch_k(add_layernorm_stream_kernel<float>, grid, kStreamWarps * 32, 0, stream, rows, width, (const float*)x, ldx, (const float*)residual, ldr, gamma, beta, (float*)y, ldy);
    else
      launch_k(add_layernorm_stream_kernel<bf16>, grid, kStreamWarps * 32, 0, stream, rows, width, (const bf16*)x, ldx, (const bf16*)residual, ldr, gamma, beta, (bf16*)y, ldy);
    return 1;
  }
  if (dtype == kF32)
    launch_k(add_layernorm_kernel<float>, grid_rows(rows), kRowsPerBlock * 32, 0, stream, rows, width, (const float*)x, ldx, (const float*)residual, ldr, gamma, beta, (float*)y, ldy);
  else
    launch_k(add_layernorm_kernel<bf16>, grid_rows(rows), kRowsPerBlock * 32, 0, stream, rows, width, (const bf16*)x, ldx, (const bf16*)residual, ldr, gamma, beta, (bf16*)y, ldy);
  return 1;
}

int launch_fold_ln_weights(int N, int K, const float* W, const float* gamma, const float* beta, const float* bias, void* Wf, float* c,
                           float* d, cudaStream_t stream) {
  if (K % 8 != 0) throw std::runtime_error("fold_ln_weights: K % 8 != 0");
  fold_ln_weights_kernel<<<grid_rows(N), kRowsPerBlock * 32, 0, stream>>>(N, K, W, gamma, beta, bias, (bf16*)Wf, c, d);
  return 1;
}

int launch_ln_apply_stats(int rows, int width, const void* x, const float2* stats, int64_t stats_ld, int parts, const float* gamma,
                          const float* beta, void* y, cudaStream_t stream) {
  if (rows <= 0) return 0;
  check_width(width);
  if (parts < 1 || parts > 32 || parts * 32 != width) throw std::runtime_error("ln_apply_stats: width must be 32 * parts <= 1024");
  launch_k(ln_apply_stats_kernel, grid_rows(rows), kRowsPerBlock * 32, 0, stream, rows, width, (const bf16*)x, stats, stats_ld, parts, gamma, beta, (bf16*)y);
  return 1;
}

int launch_embed_text(int dtype, int rows, int L, int width, const int64_t* ids, const int64_t* seg, const int* d_pos_offset,
                      int eos_to_pad, const float* word, const float* pos, const float* type, const float* type_ext,
                      int type_vocab, const float* gamma, const float* beta, void* y, cudaStream_t stream) {
  if (rows <= 0) return 0;
  check_width(width);
  if (dtype == kF32)
    embed_text_kernel<float><<<grid_rows(rows), kRowsPerBlock * 32, 0, stream>>>(rows, L, width, ids, seg, d_pos_offset, eos_to_pad, word, pos, type, type_ext, type_vocab, gamma, beta, (float*)y);
  else
    embed_text_kernel<bf16><<<grid_rows(rows), kRowsPerBlock * 32, 0, stream>>>(rows, L, width, ids, seg, d_pos_offset, eos_to_pad, word, pos, type, type_ext, type_vocab, gamma, beta, (bf16*)y);
  return 1;
}

int launch_embed_step(int dtype, int rows, int width, const int32_t* tokens, int pos0, const int* p0s, int rows_per_image, const int* d_step,
                      const float* word, const float* pos, const float* type, const float* gamma, const float* beta, void* y,
                      cudaStream_t stream) {
  if (rows <= 0) return 0;
  check_width(width);
  if (p0s && rows_per_image < 1) throw std::runtime_error("embed_step: rows_per_image must be >= 1");
  if (dtype == kF32)
    launch_k(embed_step_kernel<float>, grid_rows(rows), kRowsPerBlock * 32, 0, stream, rows, width, tokens, pos0, p0s, rows_per_image, d_step, word,
             pos, type, gamma, beta, (float*)y);
  else
    launch_k(embed_step_kernel<bf16>, grid_rows(rows), kRowsPerBlock * 32, 0, stream, rows, width, tokens, pos0, p0s, rows_per_image, d_step, word,
             pos, type, gamma, beta, (bf16*)y);
  return 1;
}

int launch_image_embed_ln(int dtype, int rows, int width, const void* x, const float* loc, const float* wloc,
                          const float* bloc, const float* gamma, const float* beta, void* y, cudaStream_t stream) {
  if (rows <= 0) return 0;
  check_width(width);
  if (dtype == kF32)
    image_embed_ln_kernel<float><<<grid_rows(rows), kRowsPerBlock * 32, 0, stream>>>(rows, width, (const float*)x, loc, wloc, bloc, gamma, beta, (float*)y);
  else
    image_embed_ln_kernel<bf16><<<grid_rows(rows), kRowsPerBlock * 32, 0, stream>>>(rows, width, (const bf16*)x, loc, wloc, bloc, gamma, beta, (bf16*)y);
  return 1;
}

int launch_cast_f32_to(int dtype, const float* src, void* dst, int64_t n, cudaStream_t stream) {
  if (n <= 0) return 0;
  const int64_t threads = (n + 7) / 8;
  const int grid = (int)((threads + 255) / 256);
  if (dtype == kF32) cast_from_f32_kernel<float><<<grid, 256, 0, stream>>>(src, (float*)dst, n);
  else cast_from_f32_kernel<bf16><<<grid, 256, 0, stream>>>(src, (bf16*)dst, n);
  return 1;
}
int launch_cast_to_f32(int dtype, const void* src, float* dst, int64_t n, cudaStream_t stream) {
  if (n <= 0) return 0;
  const int64_t threads = (n + 7) / 8;
  const int grid = (int)((threads + 255) / 256);
  if (dtype == kF32) cast_to_f32_kernel<float><<<grid, 256, 0, stream>>>((const float*)src, dst, n);
  else cast_to_f32_kernel<bf16><<<grid, 256, 0, stream>>>((const bf16*)src, dst, n);
  return 1;
}

int launch_copy_rows(int dtype, int rows, int width, const void* src, int64_t lds, void* dst, int64_t ldd, cudaStream_t stream) {
  if (rows <= 0) return 0;
  if (width % 8) throw std::runtime_error("copy_rows: width % 8 != 0");
  const int64_t n = (int64_t)rows * (width / 8);
  const int grid = (int)((n + 255) / 256);
  if (dtype == kF32) copy_rows_kernel<float><<<grid, 256, 0, stream>>>(rows, width, (const float*)src, lds, (float*)dst, ldd);
  else copy_rows_kernel<bf16><<<grid, 256, 0, stream>>>(rows, width, (const bf16*)src, lds, (bf16*)dst, ldd);
  return 1;
}

int launch_concat_fused(int dtype, int B, int Lv, int Lt, int width, const void* v, const void* t, void* fused,
                        const float* imask, const float* tmask, float* fmask, cudaStream_t stream) {
  if (B <= 0) return 0;
  if (width % 8) throw std::runtime_error("concat_fused: width % 8 != 0");
  const int64_t n = (int64_t)B * (Lv + Lt) * (width / 8);
  const int grid = (int)((n + 255) / 256);
  if (dtype == kF32) concat_fused_kernel<float><<<grid, 256, 0, stream>>>(B, Lv, Lt, width, (const float*)v, (const float*)t, (float*)fused, imask, tmask, fmask);
  else concat_fused_kernel<bf16><<<grid, 256, 0, stream>>>(B, Lv, Lt, width, (const bf16*)v, (const bf16*)t, (bf16*)fused, imask, tmask, fmask);
  return 1;
}

int launch_relu_mul(int dtype, int64_t n, const void* a, const void* b, void* out, cudaStream_t stream) {
  if (n <= 0) return 0;
  const int grid = (int)((n + 255) / 256);
  if (dtype == kF32) relu_mul_kernel<float><<<grid, 256, 0, stream>>>(n, (const float*)a, (const float*)b, (float*)out);
  else relu_mul_kernel<bf16><<<grid, 256, 0, stream>>>(n, (const bf16*)a, (const bf16*)b, (bf16*)out);
  return 1;
}

int launch_gather_first_rows(int dtype, int B, int L, int width, const void* src, void* dst, cudaStream_t stream) {
  if (B <= 0) return 0;
  const int64_t n = (int64_t)B * width;
  const int grid = (int)((n + 255) / 256);
  if (dtype == kF32) gather_first_rows_kernel<float><<<grid, 256, 0, stream>>>(B, L, width, (const float*)src, (float*)dst);
  else gather_first_rows_kernel<bf16><<<grid, 256, 0, stream>>>(B, L, width, (const bf16*)src, (bf16*)dst);
  return 1;
}

}  // namespace gstvd
