// torch <-> kernel glue for tiny_deepspeed_b200._C.  The only translation unit that sees torch headers.
#include <cstdlib>
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>

#include <vector>

#include "kernels.h"
#include "comm.h"

using torch::Tensor;
using namespace tds;

namespace {

cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

int dtype_of(const Tensor& t) {
  if (t.scalar_type() == at::kBFloat16) return kBF16;
  if (t.scalar_type() == at::kFloat) return kF32;
  TORCH_CHECK(false, "tiny_deepspeed_b200: unsupported dtype ", t.scalar_type(), " (bf16 / fp32 only)");
}

void check_cuda(const Tensor& t, const char* name) { TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor"); }

void check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  TORCH_CHECK(e == cudaSuccess, "tiny_deepspeed_b200 kernel launch failed in ", what, ": ", cudaGetErrorString(e));
}

// ---------------------------------------------------------------------------------------------------
// GEMM
// ---------------------------------------------------------------------------------------------------
GemmOperand operand(const Tensor& t, bool mn, int64_t& rows_out, int64_t& k_out, int64_t& nb1, int64_t& nb2) {
  TORCH_CHECK(t.scalar_type() == at::kBFloat16 || t.scalar_type() == at::kFloat, "gemm operands must be bf16 or fp32 (TF32 MMA)");
  TORCH_CHECK(t.dim() >= 2 && t.dim() <= 4, "gemm operand rank must be 2..4");
  TORCH_CHECK(t.stride(-1) == 1, "gemm operand inner stride must be 1");
  GemmOperand op{};
  op.ptr = t.data_ptr();
  op.ld = t.stride(-2);
  op.mn_major = mn;
  const int64_t r = t.size(-2), c = t.size(-1);
  rows_out = mn ? c : r;
  k_out = mn ? r : c;
  nb1 = 1; nb2 = 1;
  op.batch_stride = 0; op.batch_stride2 = 0;
  if (t.dim() == 3) { nb1 = t.size(0); op.batch_stride = t.stride(0); }
  if (t.dim() == 4) { nb1 = t.size(0); nb2 = t.size(1); op.batch_stride = t.stride(0); op.batch_stride2 = t.stride(1); }
  const int64_t al = t.scalar_type() == at::kFloat ? 4 : 8;   // elements per 16 bytes
  TORCH_CHECK(op.ld % al == 0 && (reinterpret_cast<uintptr_t>(op.ptr) % 16) == 0 && op.batch_stride % al == 0 &&
                  op.batch_stride2 % al == 0,
              "gemm operand must be 16-byte aligned with row/batch strides multiple of 16 bytes (TMA)");
  return op;
}

static int g_use_pair = -1;   // CTA-pair (cta_group::2) kernel: -1 = read TDS_GEMM_2CTA on first use
void set_gemm_pair(int64_t on) { g_use_pair = (int)on; }
void gemm_set_prof_t(const c10::optional<Tensor>& buf) {
  if (buf) TORCH_CHECK(buf->is_cuda() && buf->scalar_type() == at::kLong && buf->is_contiguous(), "prof buffer: int64 CUDA tensor");
  gemm_set_prof(buf ? reinterpret_cast<long long*>(buf->data_ptr()) : nullptr);
}

// L2 prefetch hint consumed by the next gemm() call (ops.prefetch_next): pointer + bytes of a resident tensor
static const void* g_prefetch_ptr = nullptr;
static int64_t g_prefetch_bytes = 0;
void gemm_set_prefetch(const Tensor& t) {
  if (!t.defined() || !t.is_cuda() || t.numel() == 0 || !t.is_contiguous()) { g_prefetch_ptr = nullptr; g_prefetch_bytes = 0; return; }
  g_prefetch_ptr = t.data_ptr();
  g_prefetch_bytes = (int64_t)t.numel() * (int64_t)t.element_size();
}

void gemm(const Tensor& a, const Tensor& b, Tensor& d, bool a_mn, bool b_mn, const c10::optional<Tensor>& bias,
          const c10::optional<Tensor>& aux, int64_t epi, bool accumulate, double alpha, int64_t config, int64_t tri,
          int64_t cluster, bool reduce_out) {
  check_cuda(a, "a"); check_cuda(b, "b"); check_cuda(d, "d");
  c10::cuda::CUDAGuard guard(a.device());
  GemmParams p{};
  int64_t M, K, N, K2, a1, a2, b1, b2;
  p.a = operand(a, a_mn, M, K, a1, a2);
  p.b = operand(b, b_mn, N, K2, b1, b2);
  TORCH_CHECK(a.scalar_type() == b.scalar_type(), "gemm: operand dtypes differ");
  p.in_dtype = dtype_of(a);
  p.io_dtype = kBF16;
  TORCH_CHECK(K == K2, "gemm: reduction dims differ: ", K, " vs ", K2);
  TORCH_CHECK(a1 == b1 && a2 == b2, "gemm: batch dims differ");
  TORCH_CHECK(K > 0, "gemm: empty reduction dim");
  TORCH_CHECK(d.stride(-1) == 1 && d.size(-2) == M && d.size(-1) == N, "gemm: bad output shape/stride");
  p.d = d.data_ptr(); p.d_dtype = dtype_of(d); p.ldd = d.stride(-2);
  p.d_batch_stride = 0; p.d_batch_stride2 = 0;
  if (d.dim() == 3) { TORCH_CHECK(d.size(0) == a1); p.d_batch_stride = d.stride(0); }
  if (d.dim() == 4) { TORCH_CHECK(d.size(0) == a1 && d.size(1) == a2); p.d_batch_stride = d.stride(0); p.d_batch_stride2 = d.stride(1); }
  p.bias = nullptr;
  if (bias.has_value() && bias->defined()) {
    TORCH_CHECK(bias->numel() == N && bias->is_contiguous(), "gemm: bias must be a contiguous [N]");
    p.io_dtype = dtype_of(*bias);
    p.bias = bias->data_ptr();
  }
  p.aux = nullptr; p.ld_aux = 0;
  if (aux.has_value() && aux->defined()) {
    TORCH_CHECK(aux->dim() == 2 && aux->size(0) == M && aux->size(1) == N && aux->stride(1) == 1, "gemm: aux must be [M,N]");
    TORCH_CHECK(!p.bias || dtype_of(*aux) == p.io_dtype, "gemm: bias and aux dtypes differ");
    p.io_dtype = dtype_of(*aux);
    TORCH_CHECK(a1 * a2 == 1, "gemm: aux epilogues are not batched");
    p.aux = aux->data_ptr(); p.ld_aux = aux->stride(0);
  }
  p.epi = (int)epi; p.accumulate = accumulate; p.alpha = (float)alpha;
  p.M = (int)M; p.N = (int)N; p.K = (int)K; p.batch = (int)(a1 * a2); p.nbatch2 = (int)a2;
  p.config = (int)config; p.tri = (int)tri; p.cluster_m = (int)cluster;
  p.reduce_out = reduce_out;
  if (reduce_out)
    TORCH_CHECK(d.scalar_type() == at::kFloat && d.dim() == 2 && a.scalar_type() == at::kBFloat16 && !p.bias && !p.aux,
                "gemm(reduce_out): bf16 operands, fp32 2-D destination, no epilogue functor");
  if (g_use_pair < 0) g_use_pair = getenv("TDS_GEMM_2CTA") ? atoi(getenv("TDS_GEMM_2CTA")) : 0;
  if (g_use_pair && gemm2_bf16(p, cur_stream())) {
    check_launch("gemm2");
    return;
  }
  if (g_prefetch_ptr) {   // one-shot L2 hint set by gemm_set_prefetch(): the operand the NEXT kernel will stream
    p.prefetch = g_prefetch_ptr; p.prefetch_bytes = g_prefetch_bytes;
    g_prefetch_ptr = nullptr; g_prefetch_bytes = 0;
  }
  gemm_bf16(p, cur_stream());
  check_launch("gemm");
}

// ---------------------------------------------------------------------------------------------------
// elementwise
// ---------------------------------------------------------------------------------------------------
std::vector<Tensor> layernorm_fwd_(const Tensor& x, const Tensor& w, const Tensor& b, double eps) {
  check_cuda(x, "x");
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(x.dim() == 2 && x.is_contiguous() && w.is_contiguous() && b.is_contiguous());
  const int M = x.size(0), N = x.size(1);
  TORCH_CHECK(w.numel() == N && b.numel() == N && w.scalar_type() == x.scalar_type() && b.scalar_type() == x.scalar_type(),
              "layernorm_fwd: weight and bias must be [N] of the input's dtype");
  Tensor y = torch::empty_like(x);
  auto fopt = x.options().dtype(at::kFloat);
  Tensor mean = torch::empty({M}, fopt), rstd = torch::empty({M}, fopt);
  layernorm_fwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), mean.data_ptr<float>(), rstd.data_ptr<float>(),
                M, N, (float)eps, dtype_of(x), cur_stream());
  check_launch("layernorm_fwd");
  return {y, mean, rstd};
}

// variant: -1 = TDS_LN_SINGLE decides, 0 = two kernels (partials + fold), 1 = single launch (candidates of the RuntimeAutoTuner)
Tensor layernorm_bwd_(const Tensor& dy, const Tensor& x, const Tensor& w, const Tensor& mean, const Tensor& rstd,
                      Tensor& dw, Tensor& db, bool accumulate, const c10::optional<Tensor>& add, int64_t variant) {
  check_cuda(x, "x");
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(dy.is_contiguous() && x.is_contiguous() && w.is_contiguous() && dw.is_contiguous() && db.is_contiguous());
  TORCH_CHECK(dw.scalar_type() == x.scalar_type() && db.scalar_type() == x.scalar_type());
  const int M = x.size(0), N = x.size(1);
  Tensor dx = torch::empty_like(x);
  const void* addp = nullptr;
  if (add.has_value() && add->defined()) { TORCH_CHECK(add->is_contiguous() && add->scalar_type() == x.scalar_type()); addp = add->data_ptr(); }
  // TDS_LN_SINGLE=1: single launch — all CTAs reduce their column sums into 8 interleaved persistent, self-cleaning fp32
  // accumulators (L2 reductions) and the last CTA converts; no fold kernel (25 launches / step less).  Measured on B200
  // (GPT-2 small step, profiles/r2_step_sweeps.md): 3.46 ms vs 3.40 ms for the default two-kernel form (per-CTA partials +
  // ln_fold_kernel, deterministic summation order) — 128 CTAs finishing together serialise in the L2 atomic units.
  static const bool deterministic = !(getenv("TDS_LN_SINGLE") && atoi(getenv("TDS_LN_SINGLE")) != 0);
  const bool want_single = variant < 0 ? !deterministic : variant == 1;
  const bool single = want_single && layernorm_bwd_fast_ok(dy.data_ptr(), x.data_ptr(), w.data_ptr(), addp, dx.data_ptr(), N,
                                                           dtype_of(x));
  static std::vector<Tensor> counters(64), accs(64);
  const int dev = x.get_device();
  Tensor scratch;
  int* counter = nullptr;
  if (single) {
    if (!counters[dev].defined()) {
      counters[dev] = torch::zeros({1}, x.options().dtype(at::kInt));
      accs[dev] = torch::zeros({8 * 2 * 2048}, x.options().dtype(at::kFloat));   // kAccCopies x 2N
    }
    scratch = accs[dev];
    counter = counters[dev].data_ptr<int>();
  } else {
    scratch = torch::empty({layernorm_bwd_scratch_rows(), 2 * N}, x.options().dtype(at::kFloat));
  }
  layernorm_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), mean.data_ptr<float>(), rstd.data_ptr<float>(), addp,
                dx.data_ptr(), scratch.data_ptr<float>(), dw.data_ptr(), db.data_ptr(), accumulate, M, N, dtype_of(x),
                cur_stream(), counter);
  check_launch("layernorm_bwd");
  return dx;
}

Tensor embedding_fwd_(const Tensor& idx, const Tensor& weight, const c10::optional<Tensor>& add, int64_t add_rows) {
  check_cuda(weight, "weight");
  c10::cuda::CUDAGuard guard(weight.device());
  TORCH_CHECK(idx.scalar_type() == at::kLong && idx.is_contiguous() && weight.is_contiguous());
  const int ntok = idx.numel(), dim = weight.size(1);
  Tensor out = torch::empty({ntok, dim}, weight.options());
  const void* addp = nullptr;
  if (add.has_value() && add->defined()) { TORCH_CHECK(add->is_contiguous() && add->scalar_type() == weight.scalar_type() && add->size(-1) == dim); addp = add->data_ptr(); }
  embedding_fwd(idx.data_ptr<int64_t>(), weight.data_ptr(), addp, (int)add_rows, out.data_ptr(), ntok, dim,
                weight.size(0), dtype_of(weight), cur_stream());
  check_launch("embedding_fwd");
  return out;
}

void embedding_bwd_(const Tensor& idx, const Tensor& dy, Tensor& dw, bool accumulate, int64_t padding_idx) {
  check_cuda(dy, "dy");
  c10::cuda::CUDAGuard guard(dy.device());
  TORCH_CHECK(idx.scalar_type() == at::kLong && idx.is_contiguous() && dy.is_contiguous() && dw.is_contiguous());
  TORCH_CHECK(dy.scalar_type() == dw.scalar_type());
  embedding_bwd(idx.data_ptr<int64_t>(), dy.data_ptr(), dw.data_ptr(), accumulate, padding_idx, (int)idx.numel(),
                (int)dw.size(1), dw.size(0), dtype_of(dw), cur_stream());
  check_launch("embedding_bwd");
}

void softmax_causal_fwd_(Tensor& s, double scale) {
  check_cuda(s, "s");
  c10::cuda::CUDAGuard guard(s.device());
  TORCH_CHECK(s.dim() == 3 && s.is_contiguous() && s.scalar_type() == at::kBFloat16 && s.size(1) == s.size(2) && s.size(2) % 8 == 0);
  softmax_causal_fwd(s.data_ptr(), (int)s.size(0), (int)s.size(1), (float)scale, cur_stream());
  check_launch("softmax_causal_fwd");
}

void softmax_causal_bwd_(const Tensor& p, Tensor& dp, double scale) {
  check_cuda(p, "p");
  c10::cuda::CUDAGuard guard(p.device());
  TORCH_CHECK(p.dim() == 3 && p.is_contiguous() && dp.is_contiguous() && p.scalar_type() == at::kBFloat16 &&
              dp.scalar_type() == at::kBFloat16 && p.sizes() == dp.sizes() && p.size(2) % 8 == 0);
  softmax_causal_bwd(p.data_ptr(), dp.data_ptr(), (int)p.size(0), (int)p.size(1), (float)scale, cur_stream());
  check_launch("softmax_causal_bwd");
}

std::vector<Tensor> cross_entropy_fwd_(const Tensor& logits, const Tensor& tgt) {
  check_cuda(logits, "logits");
  c10::cuda::CUDAGuard guard(logits.device());
  TORCH_CHECK(logits.dim() == 2 && logits.is_contiguous() && tgt.scalar_type() == at::kLong && tgt.is_contiguous());
  const int M = logits.size(0), V = logits.size(1);
  auto fopt = logits.options().dtype(at::kFloat);
  Tensor row_loss = torch::empty({M}, fopt), lse = torch::empty({M}, fopt), loss = torch::empty({}, fopt);
  xent_fwd(logits.data_ptr(), tgt.data_ptr<int64_t>(), row_loss.data_ptr<float>(), lse.data_ptr<float>(),
           loss.data_ptr<float>(), M, V, dtype_of(logits), cur_stream());
  check_launch("cross_entropy_fwd");
  return {loss, lse};
}

void cross_entropy_bwd_(const Tensor& logits, const Tensor& tgt, const Tensor& lse, const Tensor& gloss, Tensor& dl) {
  check_cuda(logits, "logits");
  c10::cuda::CUDAGuard guard(logits.device());
  TORCH_CHECK(logits.is_contiguous() && dl.is_contiguous() && gloss.scalar_type() == at::kFloat && dl.scalar_type() == logits.scalar_type());
  xent_bwd(logits.data_ptr(), tgt.data_ptr<int64_t>(), lse.data_ptr<float>(), gloss.data_ptr<float>(), dl.data_ptr(),
           (int)logits.size(0), (int)logits.size(1), dtype_of(logits), cur_stream());
  check_launch("cross_entropy_bwd");
}

Tensor gelu_fwd_(const Tensor& x) {
  check_cuda(x, "x");
  c10::cuda::CUDAGuard guard(x.device());
  Tensor y = torch::empty_like(x);
  gelu_fwd(x.data_ptr(), y.data_ptr(), x.numel(), dtype_of(x), cur_stream());
  check_launch("gelu_fwd");
  return y;
}
Tensor gelu_bwd_(const Tensor& dy, const Tensor& x) {
  check_cuda(x, "x");
  c10::cuda::CUDAGuard guard(x.device());
  Tensor dx = torch::empty_like(x);
  gelu_bwd(dy.data_ptr(), x.data_ptr(), dx.data_ptr(), x.numel(), dtype_of(x), cur_stream());
  check_launch("gelu_bwd");
  return dx;
}
Tensor cast_(const Tensor& x) {
  check_cuda(x, "x");
  TORCH_CHECK(x.is_contiguous(), "cast: input must be contiguous");
  c10::cuda::CUDAGuard guard(x.device());
  const int dt = dtype_of(x);
  Tensor y = torch::empty(x.sizes(), x.options().dtype(dt == kBF16 ? at::kFloat : at::kBFloat16));
  cast(x.data_ptr(), dt, y.data_ptr(), x.numel(), cur_stream());
  check_launch("cast");
  return y;
}
void colsum_(const Tensor& x, Tensor& out, bool accumulate) {
  check_cuda(x, "x");
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(x.dim() == 2 && x.is_contiguous() && out.is_contiguous() && out.scalar_type() == x.scalar_type());
  colsum(x.data_ptr(), out.data_ptr(), accumulate, (int)x.size(0), (int)x.size(1), dtype_of(x), cur_stream());
  check_launch("colsum");
}

std::vector<Tensor> flash_fwd_(const Tensor& qkv, int64_t n_head) {
  check_cuda(qkv, "qkv");
  c10::cuda::CUDAGuard guard(qkv.device());
  TORCH_CHECK(qkv.dim() == 3 && qkv.is_contiguous() && qkv.scalar_type() == at::kBFloat16);
  const int B = qkv.size(0), T = qkv.size(1), C = qkv.size(2) / 3, hs = C / (int)n_head;
  TORCH_CHECK(flash_supported(T, hs), "flash attention needs head size 64 and T % 128 == 0");
  Tensor y = torch::empty({B, T, C}, qkv.options());
  Tensor lse = torch::empty({B, n_head, T}, qkv.options().dtype(at::kFloat));
  flash_fwd(qkv.data_ptr(), y.data_ptr(), lse.data_ptr<float>(), B, T, (int)n_head, 1.0f / sqrtf((float)hs), cur_stream());
  check_launch("flash_fwd");
  return {y, lse};
}

Tensor flash_bwd_(const Tensor& dy, const Tensor& qkv, const Tensor& y, const Tensor& lse, int64_t n_head) {
  check_cuda(qkv, "qkv");
  c10::cuda::CUDAGuard guard(qkv.device());
  TORCH_CHECK(qkv.is_contiguous() && y.is_contiguous() && dy.is_contiguous() && lse.is_contiguous());
  TORCH_CHECK(qkv.scalar_type() == at::kBFloat16 && y.scalar_type() == at::kBFloat16 && dy.scalar_type() == at::kBFloat16 &&
              lse.scalar_type() == at::kFloat);
  const int B = qkv.size(0), T = qkv.size(1), C = qkv.size(2) / 3, hs = C / (int)n_head;
  TORCH_CHECK(flash_supported(T, hs));
  Tensor dqkv = torch::empty_like(qkv);
  auto fopt = qkv.options().dtype(at::kFloat);
  Tensor dsum = torch::empty({B, n_head, T}, fopt);
  Tensor dq_ws = torch::empty({3, B, n_head, T, hs}, fopt);      // dQ, dK, dV fp32 workspaces (flash_sm100.cu)
  flash_bwd(qkv.data_ptr(), y.data_ptr(), dy.data_ptr(), lse.data_ptr<float>(), dsum.data_ptr<float>(),
            dq_ws.data_ptr<float>(), dqkv.data_ptr(), B, T, (int)n_head, 1.0f / sqrtf((float)hs), cur_stream());
  check_launch("flash_bwd");
  return dqkv;
}

void sum_slices_(const Tensor& ws, Tensor& out) {
  check_cuda(ws, "ws");
  c10::cuda::CUDAGuard guard(ws.device());
  TORCH_CHECK(ws.scalar_type() == at::kFloat && ws.is_contiguous() && out.scalar_type() == at::kBFloat16 && out.is_contiguous());
  TORCH_CHECK(ws.numel() % out.numel() == 0);
  sum_slices(ws.data_ptr<float>(), out.data_ptr(), out.numel(), (int)(ws.numel() / out.numel()), cur_stream());
  check_launch("sum_slices");
}

// ---------------------------------------------------------------------------------------------------
// optimizers
// ---------------------------------------------------------------------------------------------------
template <typename Fn>
void for_each_chunk(const std::vector<Tensor>& ps, const std::vector<Tensor>& gs, const std::vector<Tensor>& ms,
                    const std::vector<Tensor>& vs, const std::vector<Tensor>& masters, const std::vector<Tensor>& vmax,
                    Fn&& fn) {
  const size_t n = ps.size();
  TORCH_CHECK(gs.size() == n, "params/grads length mismatch");
  size_t i = 0;
  while (i < n) {
    TensorList tl{};
    int cnt = 0, blk = 0;
    while (i < n && cnt < kMaxTensorsPerLaunch) {
      const Tensor& p = ps[i];
      TORCH_CHECK(p.is_contiguous() && gs[i].is_contiguous() && gs[i].scalar_type() == p.scalar_type() &&
                      gs[i].numel() == p.numel(), "optimizer: param/grad must be contiguous and of equal dtype/size");
      tl.p[cnt] = p.data_ptr();
      tl.g[cnt] = gs[i].data_ptr();
      tl.m[cnt] = ms.empty() ? nullptr : ms[i].data_ptr<float>();
      tl.v[cnt] = vs.empty() ? nullptr : vs[i].data_ptr<float>();
      tl.master[cnt] = masters.empty() ? nullptr : masters[i].data_ptr<float>();
      tl.vmax[cnt] = vmax.empty() ? nullptr : vmax[i].data_ptr<float>();
      tl.numel[cnt] = p.numel();
      tl.blk_start[cnt] = blk;
      blk += (int)((p.numel() + kOptChunk - 1) / kOptChunk);
      ++cnt; ++i;
    }
    tl.blk_start[cnt] = blk;
    tl.count = cnt;
    fn(tl);
  }
}

void step_increment_(Tensor& step) {
  c10::cuda::CUDAGuard guard(step.device());
  TORCH_CHECK(step.scalar_type() == at::kInt && step.numel() == 1);
  step_increment(step.data_ptr<int>(), cur_stream());
  check_launch("step_increment");
}

int64_t adamw_multi_(std::vector<Tensor> ps, std::vector<Tensor> gs, std::vector<Tensor> ms, std::vector<Tensor> vs,
                     std::vector<Tensor> masters, std::vector<Tensor> vmax, double lr, double b1, double b2, double eps,
                     double wd, const Tensor& step, bool decoupled, bool maximize, double grad_scale, int64_t background_ctas) {
  if (ps.empty()) return 0;
  c10::cuda::CUDAGuard guard(ps[0].device());
  AdamHyper h{(float)lr, (float)b1, (float)b2, (float)eps, (float)wd, (float)grad_scale, decoupled ? 1 : 0,
              maximize ? 1 : 0, step.data_ptr<int>()};
  const int dt = dtype_of(ps[0]);
  int64_t launches = 0;
  for_each_chunk(ps, gs, ms, vs, masters, vmax, [&](const TensorList& tl) { adamw_multi(tl, h, dt, cur_stream(), (int)background_ctas); ++launches; });
  check_launch("adamw_multi");
  return launches;
}

int64_t sgd_multi_(std::vector<Tensor> ps, std::vector<Tensor> gs, std::vector<Tensor> bufs, std::vector<Tensor> masters,
                   double lr, double momentum, double dampening, double wd, bool nesterov, bool maximize,
                   const Tensor& step, double grad_scale) {
  if (ps.empty()) return 0;
  c10::cuda::CUDAGuard guard(ps[0].device());
  SgdHyper h{(float)lr, (float)momentum, (float)dampening, (float)wd, (float)grad_scale, nesterov ? 1 : 0,
             maximize ? 1 : 0, step.data_ptr<int>()};
  const int dt = dtype_of(ps[0]);
  int64_t launches = 0;
  std::vector<Tensor> none;
  for_each_chunk(ps, gs, bufs, none, masters, none, [&](const TensorList& tl) { sgd_multi(tl, h, dt, cur_stream()); ++launches; });
  check_launch("sgd_multi");
  return launches;
}

}  // namespace

void bind_comm(pybind11::module_& m);  // comm_bindings.cpp

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "tiny_deepspeed_b200 sm_100a kernels";
  m.def("gemm", &gemm, "persistent tcgen05 GEMM");
  m.def("gemm_set_prefetch", &gemm_set_prefetch, "one-shot L2 prefetch hint for the next gemm launch");
  m.def("set_pdl", [](bool on) { set_pdl_enabled(on); }, "programmatic-dependent-launch edges between our kernels on / off");
  m.def("gemm_num_configs", &gemm_num_configs);
  m.def("set_gemm_pair", &set_gemm_pair, "route eligible GEMMs through the cta_group::2 kernel (0/1)");
  m.def("gemm_set_prof", &gemm_set_prof_t, "install / clear the per-CTA phase timestamp buffer (tools/gemm_timeline.py)");
  m.def("layernorm_fwd", &layernorm_fwd_);
  m.def("layernorm_bwd", &layernorm_bwd_, pybind11::arg("dy"), pybind11::arg("x"), pybind11::arg("w"), pybind11::arg("mean"),
        pybind11::arg("rstd"), pybind11::arg("dw"), pybind11::arg("db"), pybind11::arg("accumulate"), pybind11::arg("add"),
        pybind11::arg("variant") = -1);
  m.def("embedding_fwd", &embedding_fwd_);
  m.def("embedding_bwd", &embedding_bwd_);
  m.def("softmax_causal_fwd", &softmax_causal_fwd_);
  m.def("softmax_causal_bwd", &softmax_causal_bwd_);
  m.def("cross_entropy_fwd", &cross_entropy_fwd_);
  m.def("cross_entropy_bwd", &cross_entropy_bwd_);
  m.def("gelu_fwd", &gelu_fwd_);
  m.def("gelu_bwd", &gelu_bwd_);
  m.def("cast", &cast_);
  m.def("colsum", &colsum_);
  m.def("sum_slices", &sum_slices_);
  m.def("flash_fwd", &flash_fwd_);
  m.def("flash_bwd", &flash_bwd_);
  m.def("flash_supported", &flash_supported);
  m.def("step_increment", &step_increment_);
  m.def("adamw_multi", &adamw_multi_);
  m.def("sgd_multi", &sgd_multi_);
  bind_comm(m);
}
