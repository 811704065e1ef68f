// Host-side launch API of the sm_100a kernels (raw pointers + stream; no torch types here).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <initializer_list>

namespace tds {

enum DType : int { kBF16 = 0, kF32 = 1 };

// The row kernels read and write 16 bytes at a time at `base + row * pitch + 16 * i`.  That is legal only when every row
// starts on a 16-byte boundary: the row pitch is a multiple of 16 bytes and every base pointer (nullptr = operand absent)
// is 16-byte aligned.  Otherwise (bf16 rows of N % 8 != 0 elements, fp32 rows of N % 4 != 0, offset views) the kernels
// run their scalar loop over the whole row.  Decided once per launch, never per row.
inline bool rows_vec16(int64_t row_bytes, std::initializer_list<const void*> ptrs) {
  if (row_bytes % 16 != 0) return false;
  for (const void* p : ptrs)
    if (reinterpret_cast<uintptr_t>(p) & 15) return false;
  return true;
}

// ---- GEMM (gemm_sm100.cu) ---------------------------------------------------------------------
// D[b][m][n] = alpha * sum_k A(b,m,k) * B(b,n,k)  (+ epilogue).  bf16 (or fp32-as-TF32) operands, fp32 accumulate in TMEM.
struct GemmOperand {
  const void* ptr;      // bf16
  int64_t ld;           // elements between consecutive rows of the stored 2-D matrix
  int64_t batch_stride; // elements between batches (outer batch dim)
  int64_t batch_stride2; // elements between inner batch index (batch = outer * nbatch2 + inner)
  bool mn_major;        // false: stored [rows = M|N][K]; true: stored [K][rows = M|N]
};
struct GemmParams {
  GemmOperand a, b;
  void* d;  int d_dtype;  int64_t ldd, d_batch_stride, d_batch_stride2;
  int in_dtype;           // kBF16: bf16 operands (kind::f16); kF32: fp32 operands consumed as TF32 (kind::tf32)
  int io_dtype;           // dtype of bias / aux (kBF16 or kF32)
  const void* bias;       // [N] or nullptr
  void* aux;  int64_t ld_aux;   // [M,N] (no batch) or nullptr
  int epi;                // EPI_* (see ops/__init__.py)
  bool accumulate;        // D += result
  bool reduce_out;        // EXPERIMENTAL: D (fp32, may be peer memory) += result via TMA reduce-add (fused reduce-scatter epilogue)
  float alpha;
  int M, N, K, batch, nbatch2;
  int config;             // tile configuration index, -1 = heuristic
  int cluster_m;          // requested cluster size along M for B-tile multicast (0 = default, 1 = off)
  int tri;                // causal structure: 0 none, 1 skip tiles above the diagonal (S, dP),
                          // 2 K-range ends at the tile's last row (P.V, dS.K), 3 K-range starts at the tile's first row (P^T.dY, dS^T.Q)
  // L2 prefetch hint: `prefetch_bytes` bytes at `prefetch` (the weight / saved activation the NEXT kernel will stream) are
  // requested into L2 by this kernel's otherwise idle epilogue warps while its own main loop runs.  nullptr = none.
  const void* prefetch = nullptr;  int64_t prefetch_bytes = 0;
};
void gemm_bf16(const GemmParams& p, cudaStream_t stream);
void set_pdl_enabled(bool on);   // programmatic-dependent-launch edges between our kernels (common.cuh); optim.cu
// EXPERIMENTAL CTA-pair (cta_group::2) variant, gemm2_sm100.cu: returns false without launching when the problem is outside
// its coverage (then call gemm_bf16).  Opt-in through TDS_GEMM_2CTA=1 in the binding.
bool gemm2_bf16(const GemmParams& p, cudaStream_t stream);
int gemm_num_configs();
void gemm_set_prof(long long* buf);   // tools/gemm_timeline.py: per-CTA phase timestamps (nullptr = off)

// ---- elementwise / reductions (elementwise.cu) ----------------------------------------------------
void layernorm_fwd(const void* x, const void* w, const void* b, void* y, float* mean, float* rstd,
                   int M, int N, float eps, int dtype, cudaStream_t s);
int layernorm_bwd_scratch_rows();
void layernorm_bwd(const void* dy, const void* x, const void* w, const float* mean, const float* rstd,
                   const void* add, void* dx, float* scratch, void* dw, void* db, bool accumulate,
                   int M, int N, int dtype, cudaStream_t s, int* counter = nullptr);   // counter: zeroed int -> single launch
// true when layernorm_bwd takes the register-resident bf16 kernels (fast_rows.cu), the only ones that honour `counter`
bool layernorm_bwd_fast_ok(const void* dy, const void* x, const void* w, const void* add, const void* dx, int N, int dtype);
void embedding_fwd(const int64_t* idx, const void* weight, const void* add, int add_rows, void* out,
                   int ntok, int dim, int64_t vocab, int dtype, cudaStream_t s);
void embedding_bwd(const int64_t* idx, const void* dy, void* dw, bool accumulate, int64_t padding_idx,
                   int ntok, int dim, int64_t vocab, int dtype, cudaStream_t s);
void softmax_causal_fwd(void* s_inout, int nmat, int T, float scale, cudaStream_t s);
void softmax_causal_bwd(const void* p, void* dp_inout, int nmat, int T, float scale, cudaStream_t s);
void xent_fwd(const void* logits, const int64_t* tgt, float* row_loss, float* lse, float* loss, int M, int V,
              int dtype, cudaStream_t s);
void xent_bwd(const void* logits, const int64_t* tgt, const float* lse, const float* gloss, void* dlogits,
              int M, int V, int dtype, cudaStream_t s);
void gelu_fwd(const void* x, void* y, int64_t n, int dtype, cudaStream_t s);
void gelu_bwd(const void* dy, const void* x, void* dx, int64_t n, int dtype, cudaStream_t s);
void cast(const void* x, int in_dtype, void* out, int64_t n, cudaStream_t s);   // bf16 <-> fp32 (out is the other dtype)
void colsum(const void* x, void* out, bool accumulate, int M, int N, int dtype, cudaStream_t s);
void sum_slices(const float* ws, void* out_bf16, int64_t n, int S, cudaStream_t s);   // split-K fold (fast_rows.cu)

// ---- fused causal attention (flash_sm100.cu): head size 64, T % 128 == 0 -------------------------------------------
bool flash_supported(int T, int hs);
void flash_fwd(const void* qkv, void* y, float* lse_log2, int B, int T, int nh, float scale, cudaStream_t s);
void flash_bwd(const void* qkv, const void* y, const void* dy, const float* lse_log2, float* dsum_scratch, float* dq_ws,
               void* dqkv, int B, int T, int nh, float scale, cudaStream_t s);

// ---- optimizers (optim.cu) ---------------------------------------------------------------------------
constexpr int kMaxTensorsPerLaunch = 320;
struct TensorList {
  void* p[kMaxTensorsPerLaunch];        // parameter (bf16 or fp32)
  const void* g[kMaxTensorsPerLaunch];  // gradient (same dtype as p)
  float* m[kMaxTensorsPerLaunch];       // exp_avg / momentum buffer (may be null for SGD w/o momentum)
  float* v[kMaxTensorsPerLaunch];       // exp_avg_sq
  float* master[kMaxTensorsPerLaunch];  // fp32 master weights or null
  float* vmax[kMaxTensorsPerLaunch];    // amsgrad running max or null
  int blk_start[kMaxTensorsPerLaunch + 1];
  int64_t numel[kMaxTensorsPerLaunch];
  int count;
};
struct AdamHyper {
  float lr, beta1, beta2, eps, weight_decay, grad_scale;
  int decoupled, maximize;
  const int* step_ptr;  // device step counter (already incremented for this step)
};
struct SgdHyper {
  float lr, momentum, dampening, weight_decay, grad_scale;
  int nesterov, maximize;
  const int* step_ptr;  // momentum buffer is initialised with g when *step_ptr == 1
};
void step_increment(int* step_ptr, cudaStream_t s);
void adamw_multi(const TensorList& tl, const AdamHyper& h, int dtype, cudaStream_t s, int background_ctas = 0);   // > 0: fixed small grid (optimizer-in-backward)
void sgd_multi(const TensorList& tl, const SgdHyper& h, int dtype, cudaStream_t s);
constexpr int kOptChunk = 256 * 8 * 4;   // elements per CTA in the multi-tensor kernels

}  // namespace tds
