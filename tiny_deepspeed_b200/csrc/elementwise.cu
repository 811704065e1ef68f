// Memory-bound ops of the GPT-2 step for sm_100a: LayerNorm fwd/bwd, embedding gather/scatter, causal
// softmax fwd/bwd, cross-entropy fwd/bwd, GELU, column-sum.  All are single-pass over HBM with 16-byte
// accesses and fp32 math; the reductions are warp/CTA-local (no global locks, no atomics except the
// embedding scatter).  Replaces the reference's three Triton LayerNorm kernels
// (tiny_deepspeed/core/module/ops/layernorm.py:158-298) and the ATen ops of SURVEY §2.3(b).
#include "common.cuh"
#include "kernels.h"

namespace tds {

// 8-element vector access for both dtypes -----------------------------------------------------------
template <typename T> struct V8;
template <> struct V8<__nv_bfloat16> {
  static TDS_DEVICE void ld(const __nv_bfloat16* p, float* f) { unpack8(ld8(p), f); }
  static TDS_DEVICE void st(__nv_bfloat16* p, const float* f) { st8(p, pack8(f)); }
};
template <> struct V8<float> {
  static TDS_DEVICE void ld(const float* p, float* f) {
    float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  }
  static TDS_DEVICE void st(float* p, const float* f) {
    reinterpret_cast<float4*>(p)[0] = make_float4(f[0], f[1], f[2], f[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(f[4], f[5], f[6], f[7]);
  }
};

#define TDS_DISPATCH(dtype, ...)                                   \
  do {                                                             \
    if ((dtype) == kBF16) { using T = __nv_bfloat16; __VA_ARGS__; } \
    else { using T = float; __VA_ARGS__; }                          \
  } while (0)

// =====================================================================================================
// LayerNorm.  One warp per row; the row is swept from L1/L2 (it is 1.5-3 KB), statistics in fp32.
// =====================================================================================================
constexpr int kLnWarps = 4;

// VEC: the 16-byte path is legal for this launch (rows_vec16); otherwise the scalar tail loops cover the whole row.
template <typename T, bool VEC>
__global__ void __launch_bounds__(kLnWarps * 32) ln_fwd_kernel(const T* __restrict__ x, const T* __restrict__ w,
                                                              const T* __restrict__ b, T* __restrict__ y,
                                                              float* __restrict__ mean, float* __restrict__ rstd,
                                                              int M, int N, float eps) {
  pdl_launch(); pdl_wait();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * kLnWarps + (threadIdx.x >> 5);
  if (row >= M) return;
  const T* xr = x + (size_t)row * N;
  T* yr = y + (size_t)row * N;
  const int nvec = VEC ? N >> 3 : 0;
  float s = 0.f;
  for (int i = lane; i < nvec; i += 32) {
    float f[8];
    V8<T>::ld(xr + i * 8, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) s += f[j];
  }
  for (int i = (nvec << 3) + lane; i < N; i += 32) s += ldf(xr + i);
  const float mu = warp_sum(s) / N;
  float q = 0.f;
  for (int i = lane; i < nvec; i += 32) {
    float f[8];
    V8<T>::ld(xr + i * 8, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { float d = f[j] - mu; q += d * d; }
  }
  for (int i = (nvec << 3) + lane; i < N; i += 32) { float d = ldf(xr + i) - mu; q += d * d; }
  const float rs = rsqrtf(warp_sum(q) / N + eps);
  if (lane == 0) { mean[row] = mu; rstd[row] = rs; }
  for (int i = lane; i < nvec; i += 32) {
    float f[8], wv[8], bv[8];
    V8<T>::ld(xr + i * 8, f);
    V8<T>::ld(w + i * 8, wv);
    V8<T>::ld(b + i * 8, bv);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = (f[j] - mu) * rs * wv[j] + bv[j];
    V8<T>::st(yr + i * 8, f);
  }
  for (int i = (nvec << 3) + lane; i < N; i += 32) stf(yr + i, (ldf(xr + i) - mu) * rs * ldf(w + i) + ldf(b + i));
}

void layernorm_fwd(const void* x, const void* w, const void* b, void* y, float* mean, float* rstd, int M, int N,
                   float eps, int dtype, cudaStream_t s) {
  dim3 grid((M + kLnWarps - 1) / kLnWarps), block(kLnWarps * 32);
  const bool vec = rows_vec16((int64_t)N * (dtype == kBF16 ? 2 : 4), {x, w, b, y});
  TDS_DISPATCH(dtype, (launch_k(vec ? ln_fwd_kernel<T, true> : ln_fwd_kernel<T, false>, dim3(grid), dim3(block), 0, s, (const T*)x,
                                (const T*)w, (const T*)b, (T*)y, mean, rstd, M, N, eps)));
}

// Backward: grid of kLnBwdCtas persistent CTAs; every warp walks rows (stride = total warps), producing dx
// and accumulating its dw/db partial column sums in SHARED memory (lane-private columns → no conflicts on
// ownership); partials go to scratch[warp][2][N]; a second kernel reduces the scratch columns.
constexpr int kLnBwdCtas = 148;
int layernorm_bwd_scratch_rows() { return kLnBwdCtas; }  // >= rows used by either backward variant

template <typename T, bool VEC>
__global__ void __launch_bounds__(kLnWarps * 32) ln_bwd_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                                              const T* __restrict__ w, const float* __restrict__ mean,
                                                              const float* __restrict__ rstd, const T* __restrict__ add,
                                                              T* __restrict__ dx, float* __restrict__ scratch, int M,
                                                              int N) {
  pdl_launch(); pdl_wait();
  extern __shared__ float sm[];  // [kLnWarps][2][N]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* sdw = sm + (size_t)wid * 2 * N;
  float* sdb = sdw + N;
  for (int i = lane; i < N; i += 32) { sdw[i] = 0.f; sdb[i] = 0.f; }
  __syncwarp();
  const int nvec = VEC ? N >> 3 : 0;
  const int gw = blockIdx.x * kLnWarps + wid, nw = gridDim.x * kLnWarps;
  for (int row = gw; row < M; row += nw) {
    const T* xr = x + (size_t)row * N;
    const T* dyr = dy + (size_t)row * N;
    T* dxr = dx + (size_t)row * N;
    const float mu = mean[row], rs = rstd[row];
    float c1 = 0.f, c2 = 0.f;
    for (int i = lane; i < nvec; i += 32) {
      float xv[8], dv[8], wv[8];
      V8<T>::ld(xr + i * 8, xv); V8<T>::ld(dyr + i * 8, dv); V8<T>::ld(w + i * 8, wv);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float xh = (xv[j] - mu) * rs, wdy = wv[j] * dv[j];
        c1 += xh * wdy; c2 += wdy;
      }
    }
    for (int i = (nvec << 3) + lane; i < N; i += 32) {
      float xh = (ldf(xr + i) - mu) * rs, wdy = ldf(w + i) * ldf(dyr + i);
      c1 += xh * wdy; c2 += wdy;
    }
    c1 = warp_sum(c1) / N;
    c2 = warp_sum(c2) / N;
    for (int i = lane; i < nvec; i += 32) {
      float xv[8], dv[8], wv[8], o[8];
      V8<T>::ld(xr + i * 8, xv); V8<T>::ld(dyr + i * 8, dv); V8<T>::ld(w + i * 8, wv);
      if (add) V8<T>::ld(add + (size_t)row * N + i * 8, o);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float xh = (xv[j] - mu) * rs, wdy = wv[j] * dv[j];
        float d = (wdy - (xh * c1 + c2)) * rs;
        o[j] = add ? o[j] + d : d;
        sdw[i * 8 + j] += dv[j] * xh;
        sdb[i * 8 + j] += dv[j];
      }
      V8<T>::st(dxr + i * 8, o);
    }
    for (int i = (nvec << 3) + lane; i < N; i += 32) {
      float xh = (ldf(xr + i) - mu) * rs, dv = ldf(dyr + i), wdy = ldf(w + i) * dv;
      float d = (wdy - (xh * c1 + c2)) * rs;
      if (add) d += ldf(add + (size_t)row * N + i);
      stf(dxr + i, d);
      sdw[i] += dv * xh;
      sdb[i] += dv;
    }
  }
  __syncthreads();
  // fold the CTA's warps and publish one partial row per CTA
  float* out = scratch + (size_t)blockIdx.x * 2 * N;
  for (int i = threadIdx.x; i < 2 * N; i += blockDim.x) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < kLnWarps; ++k) a += sm[(size_t)k * 2 * N + i];
    out[i] = a;
  }
}

template <typename T>
__global__ void ln_bwd_reduce_kernel(const float* __restrict__ scratch, T* __restrict__ dw, T* __restrict__ db, int P,
                                     int N, int accumulate) {
  pdl_launch(); pdl_wait();
  // one warp per 32 columns x {dw,db}; lanes own a column, loop over the P partial rows (coalesced)
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= 2 * N) return;
  float a = 0.f;
  for (int r = 0; r < P; ++r) a += scratch[(size_t)r * 2 * N + col];
  T* dst = col < N ? dw + col : db + (col - N);
  if (accumulate) a += ldf(dst);
  stf(dst, a);
}

void layernorm_bwd_generic(const void* dy, const void* x, const void* w, const float* mean, const float* rstd, const void* add,
                   void* dx, float* scratch, void* dw, void* db, bool accumulate, int M, int N, int dtype,
                   cudaStream_t s) {
  const int ctas = kLnBwdCtas;
  const size_t smem = (size_t)kLnWarps * 2 * N * sizeof(float);
  const bool vec = rows_vec16((int64_t)N * (dtype == kBF16 ? 2 : 4), {dy, x, w, add, dx});
  TDS_DISPATCH(dtype, {
    auto kern = vec ? ln_bwd_kernel<T, true> : ln_bwd_kernel<T, false>;
    if (smem > 48 * 1024)
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    launch_k(kern, dim3(ctas), dim3(kLnWarps * 32), smem, s, (const T*)dy, (const T*)x, (const T*)w, mean, rstd,
                                                        (const T*)add, (T*)dx, scratch, M, N);
    launch_k(ln_bwd_reduce_kernel<T>, dim3((2 * N + 127) / 128), dim3(128), 0, s, scratch, (T*)dw, (T*)db, ctas, N, accumulate ? 1 : 0);
  });
}

// =====================================================================================================
// Embedding
// =====================================================================================================
template <typename T, bool VEC>
__global__ void emb_fwd_kernel(const int64_t* __restrict__ idx, const T* __restrict__ weight, const T* __restrict__ add,
                               int add_rows, T* __restrict__ out, int ntok, int dim, int64_t vocab) {
  pdl_launch(); pdl_wait();
  const int lane = threadIdx.x & 31;
  const int tok = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (tok >= ntok) return;
  int64_t id = idx[tok];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  const T* src = weight + (size_t)id * dim;
  const T* ar = add ? add + (size_t)(tok % add_rows) * dim : nullptr;
  T* dst = out + (size_t)tok * dim;
  const int nvec = VEC ? dim >> 3 : 0;
  for (int i = lane; i < nvec; i += 32) {
    float f[8];
    V8<T>::ld(src + i * 8, f);
    if (ar) {
      float g[8];
      V8<T>::ld(ar + i * 8, g);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] += g[j];
    }
    V8<T>::st(dst + i * 8, f);
  }
  for (int i = (nvec << 3) + lane; i < dim; i += 32) stf(dst + i, ldf(src + i) + (ar ? ldf(ar + i) : 0.f));
}

void embedding_fwd(const int64_t* idx, const void* weight, const void* add, int add_rows, void* out, int ntok, int dim,
                   int64_t vocab, int dtype, cudaStream_t s) {
  const int warps = 4;
  const bool vec = rows_vec16((int64_t)dim * (dtype == kBF16 ? 2 : 4), {weight, add, out});
  TDS_DISPATCH(dtype, (launch_k(vec ? emb_fwd_kernel<T, true> : emb_fwd_kernel<T, false>, dim3((ntok + warps - 1) / warps),
                                dim3(warps * 32), 0, s, idx, (const T*)weight, (const T*)add, add_rows > 0 ? add_rows : 1, (T*)out,
                                ntok, dim, vocab)));
}

TDS_DEVICE void atomic_add2(__nv_bfloat16* p, float a, float b) {
  atomicAdd(reinterpret_cast<__nv_bfloat162*>(p), __floats2bfloat162_rn(a, b));
}
TDS_DEVICE void atomic_add2(float* p, float a, float b) {
  atomicAdd(p, a);
  atomicAdd(p + 1, b);
}
TDS_DEVICE void atomic_add1(__nv_bfloat16* p, float a) { atomicAdd(p, __float2bfloat16_rn(a)); }   // native on sm_90+
TDS_DEVICE void atomic_add1(float* p, float a) { atomicAdd(p, a); }

// PAIR: element pairs (i, i + 1) of every gradient row are one 4-byte __nv_bfloat162 atomic (host: even dim and a 4-byte
// aligned dw, always for fp32, whose pair is two scalar atomics); otherwise one scalar atomic per element.
template <typename T, bool PAIR>
__global__ void emb_bwd_kernel(const int64_t* __restrict__ idx, const T* __restrict__ dy, T* __restrict__ dw, int ntok,
                               int dim, int64_t vocab, int64_t padding_idx) {
  pdl_launch(); pdl_wait();
  const int lane = threadIdx.x & 31;
  const int tok = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (tok >= ntok) return;
  const int64_t id = idx[tok];
  if (id < 0 || id >= vocab || id == padding_idx) return;
  const T* src = dy + (size_t)tok * dim;
  T* dst = dw + (size_t)id * dim;
  if (PAIR) {
    for (int i = lane * 2; i + 1 < dim; i += 64) atomic_add2(dst + i, ldf(src + i), ldf(src + i + 1));
    // odd tail: fp32 only, the host runs bf16 pairs for even dims only (odd bf16 dims take the scalar loop below)
    if (sizeof(T) == 4 && (dim & 1) && lane == 0) atomic_add1(dst + dim - 1, ldf(src + dim - 1));
  } else {
    for (int i = lane; i < dim; i += 32) atomic_add1(dst + i, ldf(src + i));
  }
}

void embedding_bwd(const int64_t* idx, const void* dy, void* dw, bool accumulate, int64_t padding_idx, int ntok, int dim,
                   int64_t vocab, int dtype, cudaStream_t s) {
  const size_t esz = dtype == kBF16 ? 2 : 4;
  if (!accumulate) cudaMemsetAsync(dw, 0, (size_t)vocab * dim * esz, s);
  const int warps = 4;
  const bool pair = dtype != kBF16 || (dim % 2 == 0 && (reinterpret_cast<uintptr_t>(dw) & 3) == 0);
  TDS_DISPATCH(dtype, (launch_k(pair ? emb_bwd_kernel<T, true> : emb_bwd_kernel<T, false>, dim3((ntok + warps - 1) / warps),
                                dim3(warps * 32), 0, s, idx, (const T*)dy, (T*)dw, ntok, dim, vocab, padding_idx)));
}

// =====================================================================================================
// Causal softmax over materialised scores S[nmat][T][T] (bf16, in place).  One warp per row; only the
// valid prefix [0, r] is read; the masked suffix is written as zeros so the P·V / P^T·dY GEMMs can consume
// whole tiles.
// =====================================================================================================
__global__ void __launch_bounds__(128) softmax_causal_fwd_kernel(__nv_bfloat16* __restrict__ S, int nrows, int T,
                                                                 float scale_log2e) {
  pdl_launch(); pdl_wait();
  const int lane = threadIdx.x & 31;
  const int gr = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (gr >= nrows) return;
  const int r = gr % T;
  __nv_bfloat16* row = S + (size_t)gr * T;
  const int valid = r + 1;
  const int nv = (valid + 7) >> 3;  // vectors touching valid columns
  float mx = -INFINITY;
  for (int i = lane; i < nv; i += 32) {
    float f[8];
    unpack8(ld8(row + i * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) if (i * 8 + j < valid) mx = fmaxf(mx, f[j]);
  }
  mx = warp_max(mx) * scale_log2e;
  float sum = 0.f;
  for (int i = lane; i < nv; i += 32) {
    float f[8];
    unpack8(ld8(row + i * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) if (i * 8 + j < valid) sum += exp2f(f[j] * scale_log2e - mx);
  }
  const float inv = 1.f / warp_sum(sum);
  const int tv = T >> 3;
  for (int i = lane; i < tv; i += 32) {
    float f[8];
    if (i < nv) {
      unpack8(ld8(row + i * 8), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = (i * 8 + j < valid) ? exp2f(f[j] * scale_log2e - mx) * inv : 0.f;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = 0.f;
    }
    st8(row + i * 8, pack8(f));
  }
}

void softmax_causal_fwd_generic(void* s_inout, int nmat, int T, float scale, cudaStream_t s) {
  const int nrows = nmat * T;
  launch_k(softmax_causal_fwd_kernel, dim3((nrows + 3) / 4), dim3(128), 0, s, (__nv_bfloat16*)s_inout, nrows, T,
                                                            scale * 1.4426950408889634f);
}

// dS = P * (dP - sum_j dP_j P_j) * scale, written over dP (masked suffix -> 0)
__global__ void __launch_bounds__(128) softmax_causal_bwd_kernel(const __nv_bfloat16* __restrict__ P,
                                                                 __nv_bfloat16* __restrict__ dP, int nrows, int T,
                                                                 float scale) {
  pdl_launch(); pdl_wait();
  const int lane = threadIdx.x & 31;
  const int gr = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (gr >= nrows) return;
  const int r = gr % T;
  const __nv_bfloat16* p = P + (size_t)gr * T;
  __nv_bfloat16* d = dP + (size_t)gr * T;
  const int valid = r + 1, nv = (valid + 7) >> 3;
  float dot = 0.f;
  for (int i = lane; i < nv; i += 32) {
    float a[8], b[8];
    unpack8(ld8(p + i * 8), a);
    unpack8(ld8(d + i * 8), b);
#pragma unroll
    for (int j = 0; j < 8; ++j) if (i * 8 + j < valid) dot += a[j] * b[j];
  }
  dot = warp_sum(dot);
  const int tv = T >> 3;
  for (int i = lane; i < tv; i += 32) {
    float a[8], b[8];
    if (i < nv) {
      unpack8(ld8(p + i * 8), a);
      unpack8(ld8(d + i * 8), b);
#pragma unroll
      for (int j = 0; j < 8; ++j) b[j] = (i * 8 + j < valid) ? a[j] * (b[j] - dot) * scale : 0.f;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) b[j] = 0.f;
    }
    st8(d + i * 8, pack8(b));
  }
}

void softmax_causal_bwd_generic(const void* p, void* dp_inout, int nmat, int T, float scale, cudaStream_t s) {
  const int nrows = nmat * T;
  launch_k(softmax_causal_bwd_kernel, dim3((nrows + 3) / 4), dim3(128), 0, s, (const __nv_bfloat16*)p, (__nv_bfloat16*)dp_inout, nrows,
                                                            T, scale);
}

// =====================================================================================================
// Cross-entropy.  One CTA per row of logits [M, V]; online max/sum in one sweep.
// =====================================================================================================
constexpr int kXentThreads = 512;

template <typename T, bool VEC>
__global__ void __launch_bounds__(kXentThreads) xent_fwd_kernel(const T* __restrict__ logits,
                                                                const int64_t* __restrict__ tgt,
                                                                float* __restrict__ row_loss, float* __restrict__ lse,
                                                                int V) {
  pdl_launch(); pdl_wait();
  __shared__ float red[32];
  const int row = blockIdx.x;
  const T* l = logits + (size_t)row * V;
  const int nvec = VEC ? V >> 3 : 0;
  float mx = -INFINITY, sum = 0.f;
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
    float f[8];
    V8<T>::ld(l + i * 8, f);
    float m8 = f[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) m8 = fmaxf(m8, f[j]);
    if (m8 > mx) { sum *= __expf(mx - m8); mx = m8; }
#pragma unroll
    for (int j = 0; j < 8; ++j) sum += __expf(f[j] - mx);
  }
  for (int i = (nvec << 3) + threadIdx.x; i < V; i += blockDim.x) {
    float v = ldf(l + i);
    if (v > mx) { sum *= __expf(mx - v); mx = v; }
    sum += __expf(v - mx);
  }
  const float gmx = block_max(mx, red);
  sum *= (mx == -INFINITY) ? 0.f : __expf(mx - gmx);
  const float gsum = block_sum(sum, red);
  if (threadIdx.x == 0) {
    const float z = gmx + __logf(gsum);
    lse[row] = z;
    int64_t t = tgt[row];
    row_loss[row] = (t >= 0 && t < V) ? z - ldf(l + t) : 0.f;
  }
}

__global__ void mean_kernel(const float* __restrict__ v, float* __restrict__ out, int n) {
  pdl_launch(); pdl_wait();
  __shared__ float red[32];
  float a = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) a += v[i];
  a = block_sum(a, red);
  if (threadIdx.x == 0) out[0] = a / n;
}

void xent_fwd(const void* logits, const int64_t* tgt, float* row_loss, float* lse, float* loss, int M, int V, int dtype,
              cudaStream_t s) {
  const bool vec = rows_vec16((int64_t)V * (dtype == kBF16 ? 2 : 4), {logits});
  TDS_DISPATCH(dtype, (launch_k(vec ? xent_fwd_kernel<T, true> : xent_fwd_kernel<T, false>, dim3(M), dim3(kXentThreads), 0, s,
                                (const T*)logits, tgt, row_loss, lse, V)));
  launch_k(mean_kernel, dim3(1), dim3(1024), 0, s, row_loss, loss, M);
}

template <typename T, bool VEC>
__global__ void __launch_bounds__(kXentThreads) xent_bwd_kernel(const T* __restrict__ logits,
                                                                const int64_t* __restrict__ tgt,
                                                                const float* __restrict__ lse,
                                                                const float* __restrict__ gloss, T* __restrict__ dl,
                                                                int M, int V) {
  pdl_launch(); pdl_wait();
  const int row = blockIdx.x;
  const T* l = logits + (size_t)row * V;
  T* d = dl + (size_t)row * V;
  const float z = lse[row], g = gloss[0] / M;
  const int64_t t = tgt[row];
  const int nvec = VEC ? V >> 3 : 0;
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
    float f[8];
    V8<T>::ld(l + i * 8, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = (__expf(f[j] - z) - ((int64_t)(i * 8 + j) == t ? 1.f : 0.f)) * g;
    V8<T>::st(d + i * 8, f);
  }
  for (int i = (nvec << 3) + threadIdx.x; i < V; i += blockDim.x)
    stf(d + i, (__expf(ldf(l + i) - z) - ((int64_t)i == t ? 1.f : 0.f)) * g);
}

void xent_bwd(const void* logits, const int64_t* tgt, const float* lse, const float* gloss, void* dlogits, int M, int V,
              int dtype, cudaStream_t s) {
  const bool vec = rows_vec16((int64_t)V * (dtype == kBF16 ? 2 : 4), {logits, dlogits});
  TDS_DISPATCH(dtype, (launch_k(vec ? xent_bwd_kernel<T, true> : xent_bwd_kernel<T, false>, dim3(M), dim3(kXentThreads), 0, s,
                                (const T*)logits, tgt, lse, gloss, (T*)dlogits, M, V)));
}

// =====================================================================================================
// GELU (stand-alone) and column sum (bias gradient)
// =====================================================================================================
template <typename T, bool BWD>
__global__ void gelu_kernel(const T* __restrict__ a, const T* __restrict__ x, T* __restrict__ out, int64_t n) {
  pdl_launch(); pdl_wait();
  const int64_t nvec = n >> 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    float xv[8], av[8];
    V8<T>::ld(x + i * 8, xv);
    if (BWD) V8<T>::ld(a + i * 8, av);
#pragma unroll
    for (int j = 0; j < 8; ++j) xv[j] = BWD ? av[j] * gelu_tanh_grad(xv[j]) : gelu_tanh(xv[j]);
    V8<T>::st(out + i * 8, xv);
  }
  if (blockIdx.x == 0)
    for (int64_t i = (nvec << 3) + threadIdx.x; i < n; i += blockDim.x)
      stf(out + i, BWD ? ldf(a + i) * gelu_tanh_grad(ldf(x + i)) : gelu_tanh(ldf(x + i)));
}

static int ew_grid(int64_t n) {
  int64_t b = (n / 8 + 255) / 256;
  return (int)(b < 1 ? 1 : (b > 148 * 8 ? 148 * 8 : b));
}
void gelu_fwd(const void* x, void* y, int64_t n, int dtype, cudaStream_t s) {
  TDS_DISPATCH(dtype, (launch_k(gelu_kernel<T, false>, dim3(ew_grid(n)), dim3(256), 0, s, nullptr, (const T*)x, (T*)y, n)));
}
void gelu_bwd(const void* dy, const void* x, void* dx, int64_t n, int dtype, cudaStream_t s) {
  TDS_DISPATCH(dtype, (launch_k(gelu_kernel<T, true>, dim3(ew_grid(n)), dim3(256), 0, s, (const T*)dy, (const T*)x, (T*)dx, n)));
}

// dtype conversion bf16 <-> fp32 (fp32 models run their attention core on the bf16 flash kernels)
template <typename TI, typename TO>
__global__ void cast_kernel(const TI* __restrict__ x, TO* __restrict__ out, int64_t n) {
  pdl_launch(); pdl_wait();
  const int64_t nvec = n >> 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    float v[8];
    V8<TI>::ld(x + i * 8, v);
    V8<TO>::st(out + i * 8, v);
  }
  if (blockIdx.x == 0)
    for (int64_t i = (nvec << 3) + threadIdx.x; i < n; i += blockDim.x) stf(out + i, ldf(x + i));
}
void cast(const void* x, int in_dtype, void* out, int64_t n, cudaStream_t s) {
  if (in_dtype == kBF16)
    launch_k(cast_kernel<__nv_bfloat16, float>, dim3(ew_grid(n)), dim3(256), 0, s, (const __nv_bfloat16*)x, (float*)out, n);
  else
    launch_k(cast_kernel<float, __nv_bfloat16>, dim3(ew_grid(n)), dim3(256), 0, s, (const float*)x, (__nv_bfloat16*)out, n);
}

// out[n] (+)= sum_m x[m][n]; CTA = 32 columns x 8 row-lanes, rows strided, then smem fold
template <typename T>
__global__ void colsum_kernel(const T* __restrict__ x, T* __restrict__ out, int M, int N, int accumulate) {
  pdl_launch(); pdl_wait();
  __shared__ float sm[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  float a = 0.f;
  if (col < N)
    for (int r = ty; r < M; r += 8) a += ldf(x + (size_t)r * N + col);
  sm[ty][tx] = a;
  __syncthreads();
  if (ty == 0 && col < N) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sm[k][tx];
    if (accumulate) t += ldf(out + col);
    stf(out + col, t);
  }
}
void colsum(const void* x, void* out, bool accumulate, int M, int N, int dtype, cudaStream_t s) {
  TDS_DISPATCH(dtype, (launch_k(colsum_kernel<T>, dim3((N + 31) / 32), dim3(256), 0, s, (const T*)x, (T*)out, M, N, accumulate ? 1 : 0)));
}

}  // namespace tds
