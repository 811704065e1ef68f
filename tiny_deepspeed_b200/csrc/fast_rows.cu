// Register-resident row kernels for the common GPT-2 sizes (sm_100a): LayerNorm backward and causal softmax
// forward/backward with ONE global read and ONE global write per element (rows cached in registers as packed
// bf16), falling back to the generic multi-pass kernels in elementwise.cu for other shapes / fp32.
#include "common.cuh"
#include "kernels.h"

namespace tds {

void layernorm_bwd_generic(const void* dy, const void* x, const void* w, const float* mean, const float* rstd,
                           const void* add, void* dx, float* scratch, void* dw, void* db, bool accumulate, int M, int N,
                           int dtype, cudaStream_t s);
void softmax_causal_fwd_generic(void* s_inout, int nmat, int T, float scale, cudaStream_t s);
void softmax_causal_bwd_generic(const void* p, void* dp_inout, int nmat, int T, float scale, cudaStream_t s);

// =====================================================================================================
// LayerNorm backward, bf16, N % 8 == 0, N <= 256 * MAXV.   CTA = 8 warps, one row per warp per iteration.
//   kernel 1: dx (+ residual-branch gradient) and per-CTA partial dw/db  -> scratch[cta][2N]
//   kernel 2: column-parallel fold of the partials (32 columns x 8 row-lanes per CTA)
// =====================================================================================================
constexpr int kRowWarps = 8;
constexpr int kAccCopies = 8;   // single-launch variant: accumulator copies (scratch holds kAccCopies x 2N floats)

template <int MAXV>
__global__ void __launch_bounds__(kRowWarps * 32) ln_bwd_fast_kernel(
    const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w,
    const float* __restrict__ mean, const float* __restrict__ rstd, const __nv_bfloat16* __restrict__ add,
    __nv_bfloat16* __restrict__ dx, float* __restrict__ scratch, int M, int N, int* __restrict__ counter,
    __nv_bfloat16* __restrict__ dw, __nv_bfloat16* __restrict__ db, int accumulate) {
  pdl_launch(); pdl_wait();
  extern __shared__ float sm[];   // [kRowWarps][2N]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* sdw = sm + (size_t)wid * 2 * N;
  float* sdb = sdw + N;
  const int nvec = N >> 3;
  // weight vector of this lane's columns, cached once
  bf16x8 wv[MAXV];
#pragma unroll
  for (int k = 0; k < MAXV; ++k) { const int i = lane + 32 * k; if (i < nvec) wv[k] = ld8(w + i * 8); }
  bool first = true;
  const int gw = blockIdx.x * kRowWarps + wid, nw = gridDim.x * kRowWarps;
  for (int row = gw; row < M; row += nw) {
    const __nv_bfloat16* xr = x + (size_t)row * N;
    const __nv_bfloat16* dyr = dy + (size_t)row * N;
    bf16x8 xv[MAXV], dv[MAXV], av[MAXV];
#pragma unroll
    for (int k = 0; k < MAXV; ++k) {
      const int i = lane + 32 * k;
      if (i < nvec) { xv[k] = ld8(xr + i * 8); dv[k] = ld8(dyr + i * 8); if (add) av[k] = ld8(add + (size_t)row * N + i * 8); }
    }
    const float mu = mean[row], rs = rstd[row];
    float c1 = 0.f, c2 = 0.f;
#pragma unroll
    for (int k = 0; k < MAXV; ++k) {
      if (lane + 32 * k < nvec) {
        float xf[8], df[8], wf[8];
        unpack8(xv[k], xf); unpack8(dv[k], df); unpack8(wv[k], wf);
#pragma unroll
        for (int j = 0; j < 8; ++j) { const float xh = (xf[j] - mu) * rs, wdy = wf[j] * df[j]; c1 += xh * wdy; c2 += wdy; }
      }
    }
    c1 = warp_sum(c1) / N;
    c2 = warp_sum(c2) / N;
#pragma unroll
    for (int k = 0; k < MAXV; ++k) {
      const int i = lane + 32 * k;
      if (i < nvec) {
        float xf[8], df[8], wf[8], o[8], af[8];
        unpack8(xv[k], xf); unpack8(dv[k], df); unpack8(wv[k], wf);
        if (add) unpack8(av[k], af);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (xf[j] - mu) * rs, wdy = wf[j] * df[j];
          const float d = (wdy - (xh * c1 + c2)) * rs;
          o[j] = add ? af[j] + d : d;
          const float pw = df[j] * xh;
          if (first) { sdw[i * 8 + j] = pw; sdb[i * 8 + j] = df[j]; }
          else { sdw[i * 8 + j] += pw; sdb[i * 8 + j] += df[j]; }
        }
        st8(dx + (size_t)row * N + i * 8, pack8(o));
      }
    }
    first = false;
  }
  if (first) for (int i = lane; i < 2 * N; i += 32) sdw[i] = 0.f;   // warp had no row
  __syncthreads();
  if (counter == nullptr) {
    // two-kernel variant (deterministic summation order): per-CTA partials, ln_fold_kernel finishes the job
    float* out = scratch + (size_t)blockIdx.x * 2 * N;
    for (int i = threadIdx.x; i < 2 * N; i += blockDim.x) {
      float a = 0.f;
#pragma unroll
      for (int k = 0; k < kRowWarps; ++k) a += sm[(size_t)k * 2 * N + i];
      out[i] = a;
    }
    return;
  }
  // single-launch variant: every CTA adds its column sums into ONE persistent fp32 accumulator (`scratch`, 2N floats,
  // zero on entry) with fire-and-forget L2 reductions — 128 CTAs x 2N adds overlap the other CTAs' row work — and the last
  // CTA to arrive converts the totals to bf16 and leaves accumulator + ticket counter zeroed for the next launch.
  // (The first attempt let the last CTA fold 128 x 2N partials by itself: +0.36 ms/step, profiles/r1_overlap_pdl.md; this
  // form is within 0.07 ms/step of the two-kernel default and stays opt-in: TDS_LN_SINGLE=1.)
  for (int i = threadIdx.x; i < 2 * N; i += blockDim.x) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < kRowWarps; ++k) a += sm[(size_t)k * 2 * N + i];
    // kAccCopies interleaved accumulators: 128 CTAs adding into ONE address each serialise in the L2 atomic unit
    atomicAdd(scratch + (size_t)(blockIdx.x % kAccCopies) * 2 * N + i, a);
  }
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(counter, 1) == (int)gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int col = threadIdx.x; col < 2 * N; col += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < kAccCopies; ++k) { t += __ldcg(scratch + (size_t)k * 2 * N + col); __stcg(scratch + (size_t)k * 2 * N + col, 0.f); }
    __nv_bfloat16* dst = col < N ? dw + col : db + (col - N);
    if (accumulate) t += __bfloat162float(*dst);
    *dst = __float2bfloat16_rn(t);
  }
  if (threadIdx.x == 0) *counter = 0;        // ready for the next launch
}

__global__ void __launch_bounds__(256) ln_fold_kernel(const float* __restrict__ scratch, __nv_bfloat16* __restrict__ dw,
                                                     __nv_bfloat16* __restrict__ db, int P, int N, int accumulate) {
  pdl_launch(); pdl_wait();
  __shared__ float sm[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  float a = 0.f;
  if (col < 2 * N)
    for (int r = ty; r < P; r += 8) a += scratch[(size_t)r * 2 * N + col];
  sm[ty][tx] = a;
  __syncthreads();
  if (ty == 0 && col < 2 * N) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sm[k][tx];
    __nv_bfloat16* dst = col < N ? dw + col : db + (col - N);
    if (accumulate) t += __bfloat162float(*dst);
    *dst = __float2bfloat16_rn(t);
  }
}

template <int MAXV>
static void launch_ln_bwd(const void* dy, const void* x, const void* w, const float* mean, const float* rstd,
                          const void* add, void* dx, float* scratch, void* dw, void* db, bool accumulate, int M, int N,
                          int* counter, cudaStream_t s) {
  int ctas = (M + kRowWarps - 1) / kRowWarps;
  const int cap = layernorm_bwd_scratch_rows();
  if (ctas > cap) ctas = cap;
  const size_t smem = (size_t)kRowWarps * 2 * N * sizeof(float);
  static bool attr = false;
  if (!attr) { cudaFuncSetAttribute(ln_bwd_fast_kernel<MAXV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; }
  launch_k(ln_bwd_fast_kernel<MAXV>, dim3(ctas), dim3(kRowWarps * 32), smem, s, 
      (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (const __nv_bfloat16*)w, mean, rstd, (const __nv_bfloat16*)add,
      (__nv_bfloat16*)dx, scratch, M, N, counter, (__nv_bfloat16*)dw, (__nv_bfloat16*)db, accumulate ? 1 : 0);
  if (counter == nullptr)
    launch_k(ln_fold_kernel, dim3((2 * N + 31) / 32), dim3(256), 0, s, scratch, (__nv_bfloat16*)dw, (__nv_bfloat16*)db, ctas, N, accumulate ? 1 : 0);
}

bool layernorm_bwd_fast_ok(const void* dy, const void* x, const void* w, const void* add, const void* dx, int N, int dtype) {
  return dtype == kBF16 && N % 8 == 0 && N <= 2048 && rows_vec16((int64_t)N * 2, {dy, x, w, add, dx});
}

void layernorm_bwd(const void* dy, const void* x, const void* w, const float* mean, const float* rstd, const void* add,
                   void* dx, float* scratch, void* dw, void* db, bool accumulate, int M, int N, int dtype,
                   cudaStream_t s, int* counter) {
  if (layernorm_bwd_fast_ok(dy, x, w, add, dx, N, dtype)) {
    if (N <= 1024) launch_ln_bwd<4>(dy, x, w, mean, rstd, add, dx, scratch, dw, db, accumulate, M, N, counter, s);
    else launch_ln_bwd<8>(dy, x, w, mean, rstd, add, dx, scratch, dw, db, accumulate, M, N, counter, s);
    return;
  }
  layernorm_bwd_generic(dy, x, w, mean, rstd, add, dx, scratch, dw, db, accumulate, M, N, dtype, s);
}

// =====================================================================================================
// Causal softmax, T % 8 == 0, T <= 256 * MAXV.  One warp per row, valid prefix held in registers.
// =====================================================================================================
template <int MAXV>
__global__ void __launch_bounds__(256) softmax_fwd_fast_kernel(__nv_bfloat16* __restrict__ S, int nrows, int T,
                                                              float scale_log2e) {
  pdl_launch(); pdl_wait();
  const int lane = threadIdx.x & 31;
  const int gr = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (gr >= nrows) return;
  const int r = gr % T, valid = r + 1, nv = (valid + 7) >> 3, tv = T >> 3;
  __nv_bfloat16* row = S + (size_t)gr * T;
  float f[MAXV][8];
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int i = lane + 32 * k;
    if (i < nv) {
      unpack8(ld8(row + i * 8), f[k]);
#pragma unroll
      for (int j = 0; j < 8; ++j) { if (i * 8 + j >= valid) f[k][j] = -INFINITY; mx = fmaxf(mx, f[k][j]); }
    }
  }
  mx = warp_max(mx) * scale_log2e;
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    if (lane + 32 * k < nv) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { f[k][j] = exp2f(f[k][j] * scale_log2e - mx); sum += f[k][j]; }
    }
  }
  const float inv = 1.f / warp_sum(sum);
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int i = lane + 32 * k;
    if (i < tv) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (i < nv) ? f[k][j] * inv : 0.f;
      st8(row + i * 8, pack8(o));
    }
  }
}

template <int MAXV>
__global__ void __launch_bounds__(256) softmax_bwd_fast_kernel(const __nv_bfloat16* __restrict__ P,
                                                              __nv_bfloat16* __restrict__ dP, int nrows, int T, float scale) {
  pdl_launch(); pdl_wait();
  const int lane = threadIdx.x & 31;
  const int gr = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (gr >= nrows) return;
  const int r = gr % T, valid = r + 1, nv = (valid + 7) >> 3, tv = T >> 3;
  const __nv_bfloat16* p = P + (size_t)gr * T;
  __nv_bfloat16* d = dP + (size_t)gr * T;
  float a[MAXV][8], b[MAXV][8];
  float dot = 0.f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int i = lane + 32 * k;
    if (i < nv) {
      unpack8(ld8(p + i * 8), a[k]);
      unpack8(ld8(d + i * 8), b[k]);
#pragma unroll
      for (int j = 0; j < 8; ++j) { if (i * 8 + j >= valid) { a[k][j] = 0.f; b[k][j] = 0.f; } dot += a[k][j] * b[k][j]; }
    }
  }
  dot = warp_sum(dot);
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int i = lane + 32 * k;
    if (i < tv) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (i < nv) ? a[k][j] * (b[k][j] - dot) * scale : 0.f;
      st8(d + i * 8, pack8(o));
    }
  }
}

void softmax_causal_fwd(void* s_inout, int nmat, int T, float scale, cudaStream_t s) {
  const int nrows = nmat * T;
  const float sl = scale * 1.4426950408889634f;
  if (T % 8 == 0 && T <= 1024) launch_k(softmax_fwd_fast_kernel<4>, dim3((nrows + 7) / 8), dim3(256), 0, s, (__nv_bfloat16*)s_inout, nrows, T, sl);
  else if (T % 8 == 0 && T <= 2048) launch_k(softmax_fwd_fast_kernel<8>, dim3((nrows + 7) / 8), dim3(256), 0, s, (__nv_bfloat16*)s_inout, nrows, T, sl);
  else softmax_causal_fwd_generic(s_inout, nmat, T, scale, s);
}

void softmax_causal_bwd(const void* p, void* dp_inout, int nmat, int T, float scale, cudaStream_t s) {
  const int nrows = nmat * T;
  if (T % 8 == 0 && T <= 1024)
    launch_k(softmax_bwd_fast_kernel<4>, dim3((nrows + 7) / 8), dim3(256), 0, s, (const __nv_bfloat16*)p, (__nv_bfloat16*)dp_inout, nrows, T, scale);
  else if (T % 8 == 0 && T <= 2048)
    launch_k(softmax_bwd_fast_kernel<8>, dim3((nrows + 7) / 8), dim3(256), 0, s, (const __nv_bfloat16*)p, (__nv_bfloat16*)dp_inout, nrows, T, scale);
  else softmax_causal_bwd_generic(p, dp_inout, nmat, T, scale, s);
}

// =====================================================================================================
// out[i] = sum_s ws[s][i]   (split-K reduction, fp32 slices -> bf16)
// =====================================================================================================
__global__ void sum_slices_kernel(const float* __restrict__ ws, __nv_bfloat16* __restrict__ out, int64_t n, int S) {
  pdl_launch(); pdl_wait();
  const int64_t nvec = n >> 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int sIdx = 0; sIdx < S; ++sIdx) {
      const float4 a = reinterpret_cast<const float4*>(ws + (size_t)sIdx * n + i * 8)[0];
      const float4 b = reinterpret_cast<const float4*>(ws + (size_t)sIdx * n + i * 8)[1];
      acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w; acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
    }
    st8(out + i * 8, pack8(acc));
  }
  if (blockIdx.x == 0)
    for (int64_t i = (nvec << 3) + threadIdx.x; i < n; i += blockDim.x) {
      float a = 0.f;
      for (int sIdx = 0; sIdx < S; ++sIdx) a += ws[(size_t)sIdx * n + i];
      out[i] = __float2bfloat16_rn(a);
    }
}

void sum_slices(const float* ws, void* out, int64_t n, int S, cudaStream_t s) {
  int64_t blocks = (n / 8 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(sum_slices_kernel, dim3((int)blocks), dim3(256), 0, s, ws, (__nv_bfloat16*)out, n, S);
}

}  // namespace tds
