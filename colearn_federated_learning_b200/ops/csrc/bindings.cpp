// Torch bindings for the colearn sm_100a kernels.  Only this translation unit sees torch headers.
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <cuda_runtime.h>

#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "colearn_kernels.h"

namespace py = pybind11;
using namespace colearn;

namespace {

inline cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

inline void check(cudaError_t e, const char* what) {
  TORCH_CHECK(e == cudaSuccess, what, ": ", cudaGetErrorString(e));
}
template <class T>
inline T* ptr_of(int64_t p) { return reinterpret_cast<T*>(static_cast<uintptr_t>(p)); }

#define CHECK_CUDA_F32(t) TORCH_CHECK((t).is_cuda() && (t).scalar_type() == at::kFloat && (t).is_contiguous(), #t " must be a contiguous CUDA float32 tensor")

// ---- persistent MLP -----------------------------------------------------------------------------
#include "client_desc.inc"
int64_t client_desc_size() { return (int64_t)sizeof(ClientDesc); }

// p[0:n] *= scale for a raw device pointer (the symmetric work arena)
void scale_inplace(int64_t ptr, int64_t n, double scale) {
  check(launch_scale_inplace(ptr_of<float>(ptr), (float)scale, n, cur_stream()), "scale_inplace");
}

// limit of every bounded cross-GPU flag wait on the CURRENT device (colearn_kernels.h: spin_wait_ge); 0 = wait forever
void set_spin_limit(double seconds) {
  const unsigned long long ns = seconds <= 0 ? 0ull : (unsigned long long)(seconds * 1e9);
  check(set_spin_limit_comm(ns), "set_spin_limit (comm)");
  check(set_spin_limit_mlp(ns), "set_spin_limit (mlp)");
  check(set_spin_limit_gemm(ns), "set_spin_limit (gemm)");
  check(preload_comm_kernels(), "preload_comm_kernels");     // same call site: once per device, before any round
}

void mlp_local_sgd(int64_t net_kind, torch::Tensor descs, int64_t desc_offset, int64_t n_clients,
                   int64_t batch_size, int64_t epochs, int64_t max_steps, int64_t loss, double lr, int64_t variant) {
  TORCH_CHECK(descs.is_cuda() && descs.scalar_type() == at::kByte && descs.is_contiguous(), "descs must be CUDA uint8");
  TORCH_CHECK((desc_offset + n_clients) * (int64_t)sizeof(ClientDesc) <= descs.numel(), "descs too small");
  c10::cuda::CUDAGuard guard(descs.device());
  SgdHyper hp;
  hp.batch_size = (int)batch_size; hp.epochs = (int)epochs; hp.max_steps = (int)max_steps;
  hp.loss = (int)loss; hp.lr = (float)lr; hp.variant = (int)variant;
  const ClientDesc* d = reinterpret_cast<const ClientDesc*>(descs.data_ptr<uint8_t>()) + desc_offset;
  check(launch_mlp_local_sgd((int)net_kind, d, (int)n_clients, hp, cur_stream()), "mlp_local_sgd launch");
}
int64_t mlp_net_params(int64_t net_kind) { return mlp_net_num_params((int)net_kind); }
int64_t mlp_smem_bytes(int64_t net_kind, int64_t batch) { return mlp_local_sgd_smem_bytes((int)net_kind, (int)batch); }

// any small MLP (mlp_generic.cu): one client = one cluster of `cluster` CTAs (0 = the smallest that fits)
void mlp_local_sgd_generic(std::vector<int64_t> dims, bool sigmoid, torch::Tensor descs, int64_t desc_offset, int64_t n_clients,
                           int64_t batch_size, int64_t epochs, int64_t max_steps, int64_t loss, double lr, int64_t cluster) {
  TORCH_CHECK(descs.is_cuda() && descs.scalar_type() == at::kByte && descs.is_contiguous(), "descs must be CUDA uint8");
  TORCH_CHECK((desc_offset + n_clients) * (int64_t)sizeof(ClientDesc) <= descs.numel(), "descs too small");
  TORCH_CHECK(dims.size() >= 2 && dims.size() <= 9, "dims: 2..9 widths");
  std::vector<int> d(dims.begin(), dims.end());
  c10::cuda::CUDAGuard guard(descs.device());
  SgdHyper hp;
  hp.batch_size = (int)batch_size; hp.epochs = (int)epochs; hp.max_steps = (int)max_steps;
  hp.loss = (int)loss; hp.lr = (float)lr; hp.variant = 0;
  const ClientDesc* p = reinterpret_cast<const ClientDesc*>(descs.data_ptr<uint8_t>()) + desc_offset;
  check(launch_mlp_local_sgd_generic(d.data(), (int)d.size() - 1, sigmoid ? 1 : 0, p, (int)n_clients, hp, (int)cluster, cur_stream()),
        "mlp_local_sgd_generic launch");
}
int64_t generic_plan(std::vector<int64_t> dims, int64_t batch_size, int64_t cluster) {
  if (dims.size() < 2 || dims.size() > 9) return -1;
  std::vector<int> d(dims.begin(), dims.end());
  return mlp_generic_plan(d.data(), (int)d.size() - 1, (int)batch_size, (int)cluster, nullptr);
}

torch::Tensor mlp_forward(int64_t net_kind, torch::Tensor theta, torch::Tensor x, int64_t d_out) {
  CHECK_CUDA_F32(theta); CHECK_CUDA_F32(x);
  c10::cuda::CUDAGuard guard(x.device());
  auto out = torch::empty({x.size(0), d_out}, x.options());
  check(launch_mlp_forward((int)net_kind, theta.data_ptr<float>(), x.data_ptr<float>(), out.data_ptr<float>(),
                           (int)x.size(0), cur_stream()), "mlp_forward launch");
  return out;
}

// ---- elementwise -----------------------------------------------------------------------------------
void sgd_step(torch::Tensor p, torch::Tensor g, double lr) {
  CHECK_CUDA_F32(p);
  TORCH_CHECK(g.is_cuda() && g.is_contiguous() && g.numel() == p.numel(), "grad shape");
  c10::cuda::CUDAGuard guard(p.device());
  if (g.scalar_type() == at::kFloat)
    check(launch_sgd_step(p.data_ptr<float>(), g.data_ptr<float>(), (float)lr, p.numel(), cur_stream()), "sgd_step");
  else if (g.scalar_type() == at::kBFloat16)
    check(launch_sgd_step_bf16grad(p.data_ptr<float>(), g.data_ptr(), (float)lr, p.numel(), cur_stream()), "sgd_step_bf16");
  else
    TORCH_CHECK(false, "grad dtype must be float32 or bfloat16");
}

void fedavg_apply(torch::Tensor theta, torch::Tensor slots, torch::Tensor weights, double server_lr) {
  CHECK_CUDA_F32(theta); CHECK_CUDA_F32(slots); CHECK_CUDA_F32(weights);
  TORCH_CHECK(slots.dim() == 2 && slots.size(1) >= theta.numel() && weights.numel() == slots.size(0), "shapes");
  c10::cuda::CUDAGuard guard(theta.device());
  check(launch_fedavg_apply(theta.data_ptr<float>(), slots.data_ptr<float>(), slots.stride(0), weights.data_ptr<float>(),
                            (int)slots.size(0), (float)server_lr, theta.numel(), cur_stream()), "fedavg_apply");
}
torch::Tensor fedavg_flat(torch::Tensor slots, torch::Tensor weights) {
  CHECK_CUDA_F32(slots); CHECK_CUDA_F32(weights);
  TORCH_CHECK(slots.dim() == 2 && weights.numel() == slots.size(0), "shapes");
  c10::cuda::CUDAGuard guard(slots.device());
  auto out = torch::empty({slots.size(1)}, slots.options());
  check(launch_fedavg_flat(out.data_ptr<float>(), slots.data_ptr<float>(), slots.stride(0), weights.data_ptr<float>(),
                           (int)slots.size(0), slots.size(1), cur_stream()), "fedavg_flat");
  return out;
}

std::vector<torch::Tensor> sigmoid_bce(torch::Tensor z, torch::Tensor y) {
  CHECK_CUDA_F32(z); CHECK_CUDA_F32(y);
  TORCH_CHECK(z.numel() == y.numel(), "shape");
  c10::cuda::CUDAGuard guard(z.device());
  auto dz = torch::empty_like(z);
  auto loss = torch::empty({}, z.options());
  check(launch_sigmoid_bce(z.data_ptr<float>(), y.data_ptr<float>(), dz.data_ptr<float>(), loss.data_ptr<float>(), z.numel(), cur_stream()), "sigmoid_bce");
  return {loss, dz};
}
std::vector<torch::Tensor> sse_loss(torch::Tensor out, torch::Tensor y, double scale) {
  CHECK_CUDA_F32(out); CHECK_CUDA_F32(y);
  TORCH_CHECK(out.numel() == y.numel(), "shape");
  c10::cuda::CUDAGuard guard(out.device());
  auto dz = torch::empty_like(out);
  auto loss = torch::empty({}, out.options());
  check(launch_sse(out.data_ptr<float>(), y.data_ptr<float>(), dz.data_ptr<float>(), loss.data_ptr<float>(), out.numel(), (float)scale, cur_stream()), "sse");
  return {loss, dz};
}
std::vector<torch::Tensor> softmax_xent(torch::Tensor logits, torch::Tensor labels, bool want_bf16_grad) {
  TORCH_CHECK(logits.is_cuda() && logits.is_contiguous() && logits.dim() == 2, "logits");
  TORCH_CHECK(labels.is_cuda() && labels.scalar_type() == at::kLong && labels.is_contiguous() && labels.numel() == logits.size(0), "labels");
  const bool bf16 = logits.scalar_type() == at::kBFloat16;
  TORCH_CHECK(bf16 || logits.scalar_type() == at::kFloat, "logits dtype");
  c10::cuda::CUDAGuard guard(logits.device());
  auto loss = torch::empty({}, logits.options().dtype(at::kFloat));
  torch::Tensor dl, dlb;
  if (want_bf16_grad) dlb = torch::empty(logits.sizes(), logits.options().dtype(at::kBFloat16));
  else dl = torch::empty(logits.sizes(), logits.options().dtype(at::kFloat));
  check(launch_softmax_xent(logits.data_ptr(), bf16 ? 1 : 0, labels.data_ptr<int64_t>(),
                            want_bf16_grad ? nullptr : dl.data_ptr<float>(), want_bf16_grad ? dlb.data_ptr() : nullptr,
                            loss.data_ptr<float>(), (int)logits.size(0), (int)logits.size(1), cur_stream()), "softmax_xent");
  return {loss, want_bf16_grad ? dlb : dl};
}
// Fused loss head on padded operands (see softmax_xent_head_kernel): returns the mean loss; writes dl_bf16[:rows, :cols] and db[:cols].
torch::Tensor softmax_xent_head(torch::Tensor logits, torch::Tensor labels, int64_t rows, int64_t cols, c10::optional<torch::Tensor> dl_f32,
                                c10::optional<torch::Tensor> dl_bf16, c10::optional<torch::Tensor> db) {
  TORCH_CHECK(logits.is_cuda() && logits.dim() == 2 && logits.stride(1) == 1 && rows >= 1 && rows <= logits.size(0) && cols >= 1 &&
              cols <= logits.size(1), "logits [>= rows, >= cols], unit column stride");
  const bool bf16 = logits.scalar_type() == at::kBFloat16;
  TORCH_CHECK(bf16 || logits.scalar_type() == at::kFloat, "logits dtype");
  TORCH_CHECK(labels.is_cuda() && labels.scalar_type() == at::kLong && labels.is_contiguous() && labels.numel() >= rows, "labels int64 [rows]");
  float* dlp = nullptr; int ld_dl = 0; void* dbp16 = nullptr; int ld16 = 0; float* dbp = nullptr;
  if (dl_f32.has_value()) {
    TORCH_CHECK(dl_f32->is_cuda() && dl_f32->scalar_type() == at::kFloat && dl_f32->dim() == 2 && dl_f32->stride(1) == 1 &&
                dl_f32->size(0) >= rows && dl_f32->size(1) >= cols, "dl_f32");
    dlp = dl_f32->data_ptr<float>(); ld_dl = (int)dl_f32->stride(0);
  }
  if (dl_bf16.has_value()) {
    TORCH_CHECK(dl_bf16->is_cuda() && dl_bf16->scalar_type() == at::kBFloat16 && dl_bf16->dim() == 2 && dl_bf16->stride(1) == 1 &&
                dl_bf16->size(0) >= rows && dl_bf16->size(1) >= cols, "dl_bf16");
    dbp16 = dl_bf16->data_ptr(); ld16 = (int)dl_bf16->stride(0);
  }
  if (db.has_value()) {
    TORCH_CHECK(db->is_cuda() && db->scalar_type() == at::kFloat && db->is_contiguous() && db->numel() >= cols, "db fp32 [>= cols]");
    dbp = db->data_ptr<float>();
  }
  c10::cuda::CUDAGuard guard(logits.device());
  auto loss = torch::empty({}, logits.options().dtype(at::kFloat));
  check(launch_softmax_xent_head(logits.data_ptr(), bf16 ? 1 : 0, (int)logits.stride(0), labels.data_ptr<int64_t>(), dlp, ld_dl, dbp16, ld16, dbp,
                                 loss.data_ptr<float>(), (int)rows, (int)cols, cur_stream()), "softmax_xent_head");
  return loss;
}
std::vector<torch::Tensor> eval_binary(torch::Tensor p, torch::Tensor y) {
  CHECK_CUDA_F32(p); CHECK_CUDA_F32(y);
  c10::cuda::CUDAGuard guard(p.device());
  auto loss = torch::empty({}, p.options());
  auto correct = torch::empty({}, p.options().dtype(at::kInt));
  check(launch_eval_binary(p.data_ptr<float>(), y.data_ptr<float>(), loss.data_ptr<float>(), correct.data_ptr<int>(), p.numel(), cur_stream()), "eval_binary");
  return {loss, correct};
}
torch::Tensor argmax_rows(torch::Tensor x) {
  CHECK_CUDA_F32(x);
  TORCH_CHECK(x.dim() == 2, "2-D");
  c10::cuda::CUDAGuard guard(x.device());
  auto out = torch::empty({x.size(0), 1}, x.options().dtype(at::kLong));
  check(launch_argmax_rows(x.data_ptr<float>(), out.data_ptr<int64_t>(), (int)x.size(0), (int)x.size(1), cur_stream()), "argmax");
  return out;
}
torch::Tensor minmax_scale(torch::Tensor x) {
  CHECK_CUDA_F32(x);
  TORCH_CHECK(x.dim() == 2, "2-D");
  c10::cuda::CUDAGuard guard(x.device());
  auto out = torch::empty_like(x);
  check(launch_minmax_scale(x.data_ptr<float>(), out.data_ptr<float>(), (int)x.size(0), (int)x.size(1), cur_stream()), "minmax");
  return out;
}
torch::Tensor feistel_permutation(int64_t n, int64_t rows, int64_t seed, torch::Device device) {
  if (device.is_cpu()) {   // the same bijection on the host (tests; CPU-side users of a kernel-generated order)
    auto out = torch::empty({rows, n}, torch::TensorOptions().dtype(at::kInt));
    const FeistelDomain dom = feistel_domain((uint32_t)n);
    int* p = out.data_ptr<int>();
    for (int64_t r = 0; r < rows; ++r)
      for (int64_t i = 0; i < n; ++i) p[r * n + i] = (int)feistel_index((uint32_t)i, (uint32_t)n, dom, (uint64_t)seed, (int)r);
    return out;
  }
  c10::cuda::CUDAGuard guard(device);
  auto out = torch::empty({rows, n}, torch::TensorOptions().dtype(at::kInt).device(device));
  check(launch_feistel_permutation(out.data_ptr<int>(), (int)n, (int)rows, (uint64_t)seed, cur_stream()), "feistel");
  return out;
}
torch::Tensor fp32_to_bf16(torch::Tensor x) {
  CHECK_CUDA_F32(x);
  c10::cuda::CUDAGuard guard(x.device());
  auto out = torch::empty(x.sizes(), x.options().dtype(at::kBFloat16));
  check(launch_fp32_to_bf16(x.data_ptr<float>(), out.data_ptr(), x.numel(), cur_stream()), "fp32_to_bf16");
  return out;
}
void fp32_to_bf16_into(int64_t src, int64_t dst, int64_t n) {
  check(launch_fp32_to_bf16(ptr_of<const float>(src), ptr_of<void>(dst), n, cur_stream()), "fp32_to_bf16");
}
torch::Tensor transpose_bf16(torch::Tensor x, c10::optional<torch::Tensor> out) {
  TORCH_CHECK(x.is_cuda() && x.scalar_type() == at::kBFloat16 && x.dim() == 2 && x.is_contiguous(), "x must be contiguous CUDA bf16 [R,C]");
  c10::cuda::CUDAGuard guard(x.device());
  torch::Tensor o = out.has_value() ? *out : torch::empty({x.size(1), x.size(0)}, x.options());
  TORCH_CHECK(o.is_contiguous() && o.numel() == x.numel() && o.scalar_type() == at::kBFloat16, "out");
  check(launch_transpose_bf16(x.data_ptr(), o.data_ptr(), (int)x.size(0), (int)x.size(1), cur_stream()), "transpose_bf16");
  return o;
}
torch::Tensor fix_precision(torch::Tensor x, double base) {
  CHECK_CUDA_F32(x);
  c10::cuda::CUDAGuard guard(x.device());
  auto out = torch::empty(x.sizes(), x.options().dtype(at::kLong));
  check(launch_fix_precision(x.data_ptr<float>(), reinterpret_cast<long long*>(out.data_ptr<int64_t>()), x.numel(), base, cur_stream()), "fix_precision");
  return out;
}
torch::Tensor float_precision(torch::Tensor x, double base) {
  TORCH_CHECK(x.is_cuda() && x.scalar_type() == at::kLong && x.is_contiguous(), "x must be contiguous CUDA int64");
  c10::cuda::CUDAGuard guard(x.device());
  auto out = torch::empty(x.sizes(), x.options().dtype(at::kFloat));
  check(launch_float_precision(reinterpret_cast<const long long*>(x.data_ptr<int64_t>()), out.data_ptr<float>(), x.numel(), 1.0 / base, cur_stream()), "float_precision");
  return out;
}
torch::Tensor ring_matmul(torch::Tensor a, torch::Tensor b) {
  TORCH_CHECK(a.is_cuda() && b.is_cuda() && a.scalar_type() == at::kLong && b.scalar_type() == at::kLong, "int64 CUDA tensors");
  TORCH_CHECK(a.dim() == 2 && b.dim() == 2 && a.size(1) == b.size(0) && a.is_contiguous() && b.is_contiguous(), "A[M,K] B[K,N] contiguous");
  c10::cuda::CUDAGuard guard(a.device());
  auto out = torch::empty({a.size(0), b.size(1)}, a.options());
  check(launch_ring_matmul(reinterpret_cast<const long long*>(a.data_ptr<int64_t>()), reinterpret_cast<const long long*>(b.data_ptr<int64_t>()),
                           reinterpret_cast<long long*>(out.data_ptr<int64_t>()), (int)a.size(0), (int)a.size(1), (int)b.size(1), cur_stream()), "ring_matmul");
  return out;
}
torch::Tensor bias_sgd_from_partials(c10::optional<torch::Tensor> bias, torch::Tensor partials, double lr) {
  CHECK_CUDA_F32(partials);
  TORCH_CHECK(partials.dim() == 2, "partials [rows, n]");
  c10::cuda::CUDAGuard guard(partials.device());
  const int rows = (int)partials.size(0), n = (int)partials.size(1);
  auto grad = torch::empty({n}, partials.options());
  float* b = nullptr;
  int nb = n;
  if (bias.has_value()) {
    TORCH_CHECK(bias->is_cuda() && bias->scalar_type() == at::kFloat && bias->is_contiguous() && bias->numel() <= n, "bias");
    b = bias->data_ptr<float>();
    nb = (int)bias->numel();
  }
  check(launch_bias_sgd_from_partials(b, partials.data_ptr<float>(), rows, n, partials.stride(0), (float)lr, grad.data_ptr<float>(), nb, cur_stream()), "bias_sgd_from_partials");
  return grad;
}
void l2_flush(torch::Tensor buf) {
  CHECK_CUDA_F32(buf);
  c10::cuda::CUDAGuard guard(buf.device());
  check(launch_l2_flush(buf.data_ptr<float>(), buf.numel(), cur_stream()), "l2_flush");
}

// ---- comm ---------------------------------------------------------------------------------------------
void star_round(int64_t theta, int64_t slots, int64_t slot_stride, int64_t arrive_flags, int64_t arrive_epoch,
                std::vector<int64_t> peer_inbox, std::vector<int64_t> peer_bcast_flag, int64_t bcast_epoch,
                int64_t mc_inbox, int64_t select_mask, double server_lr, int64_t n, bool do_reduce, bool do_bcast,
                int64_t grid_counter, int64_t n_blocks, double timeout_ms, std::vector<double> weights, int64_t decision) {
  StarRoundArgs a;
  std::memset(&a, 0, sizeof(a));
  a.theta = ptr_of<float>(theta);
  a.slots = ptr_of<const float>(slots);
  a.slot_stride = slot_stride;
  a.arrive_flags = ptr_of<const uint32_t>(arrive_flags);
  a.arrive_epoch = (uint32_t)arrive_epoch;
  a.world = (int)peer_inbox.size();
  TORCH_CHECK(a.world <= 16 && peer_bcast_flag.size() == peer_inbox.size(), "world");
  for (int k = 0; k < a.world; ++k) {
    a.peer_inbox[k] = ptr_of<float>(peer_inbox[k]);
    a.peer_bcast_flag[k] = ptr_of<uint32_t>(peer_bcast_flag[k]);
  }
  a.bcast_epoch = (uint32_t)bcast_epoch;
  a.mc_inbox = ptr_of<float>(mc_inbox);
  a.select_mask = (uint32_t)select_mask;
  a.server_lr = (float)server_lr;
  a.n = n;
  a.do_reduce = do_reduce ? 1 : 0;
  a.do_bcast = do_bcast ? 1 : 0;
  a.grid_counter = ptr_of<uint32_t>(grid_counter);
  a.timeout_ns = timeout_ms > 0 ? (unsigned long long)(timeout_ms * 1e6) : 0ull;
  for (size_t k = 0; k < weights.size() && k < 16; ++k) a.weights[k] = (float)weights[k];
  a.decision = ptr_of<uint32_t>(decision);
  TORCH_CHECK(a.timeout_ns == 0 || a.decision != nullptr, "a deadline needs the decision scratch buffer");
  check(launch_star_round(a, (int)n_blocks, cur_stream()), "star_round");
}

static TwoShotArgs make_twoshot_args(const std::vector<int64_t>& work, const std::vector<int64_t>& shadow, const std::vector<int64_t>& chunk_flags,
                    int64_t arrive_flags, int64_t weights, int64_t theta_prev, int64_t epoch, int64_t select_mask,
                    double server_lr, int64_t n, int64_t chunk_elems, int64_t rank,
                    const std::vector<int64_t>& peer_arrive, bool wait_all, int64_t mc_work, int64_t mc_shadow, int64_t produced,
                    double produced_timeout_s) {
  TwoShotArgs a;
  std::memset(&a, 0, sizeof(a));
  a.world = (int)work.size();
  TORCH_CHECK(a.world <= 16 && chunk_flags.size() == work.size(), "world");
  for (int k = 0; k < a.world; ++k) {
    a.work[k] = ptr_of<float>(work[k]);
    a.shadow_bf16[k] = shadow.empty() ? nullptr : ptr_of<void>(shadow[k]);
    a.chunk_flags[k] = ptr_of<uint32_t>(chunk_flags[k]);
  }
  a.arrive_flags = ptr_of<const uint32_t>(arrive_flags);
  a.weights = ptr_of<const float>(weights);
  a.theta_prev = ptr_of<float>(theta_prev);
  a.epoch = (uint32_t)epoch;
  a.select_mask = (uint32_t)select_mask;
  a.server_lr = (float)server_lr;
  a.n = n;
  a.chunk_elems = chunk_elems;
  a.rank = (int)rank;
  a.signal_arrive = peer_arrive.empty() ? 0 : 1;
  for (size_t k = 0; k < peer_arrive.size() && k < 16; ++k) a.peer_arrive[k] = ptr_of<uint32_t>(peer_arrive[k]);
  a.wait_all = wait_all ? 1 : 0;
  a.mc_work = ptr_of<float>(mc_work);
  a.mc_shadow = ptr_of<void>(mc_shadow);
  // overlapped form (fused wgrad GEMM -> FedAvg reduce): my [world, n_chunks] table of produced epochs
  a.produced = ptr_of<const uint32_t>(produced);
  a.produced_timeout_ns = produced_timeout_s > 0 ? (unsigned long long)(produced_timeout_s * 1e9) : 0ull;
  return a;
}

void twoshot_fedavg(std::vector<int64_t> work, std::vector<int64_t> shadow, std::vector<int64_t> chunk_flags,
                    int64_t arrive_flags, int64_t weights, int64_t theta_prev, int64_t epoch, int64_t select_mask,
                    double server_lr, int64_t n, int64_t chunk_elems, int64_t rank, int64_t n_blocks,
                    std::vector<int64_t> peer_arrive, bool wait_all, int64_t mc_work, int64_t mc_shadow, int64_t produced,
                    double produced_timeout_s) {
  TwoShotArgs a = make_twoshot_args(work, shadow, chunk_flags, arrive_flags, weights, theta_prev, epoch, select_mask, server_lr, n,
                                    chunk_elems, rank, peer_arrive, wait_all, mc_work, mc_shadow, produced, produced_timeout_s);
  check(launch_twoshot_fedavg(a, (int)n_blocks, cur_stream()), "twoshot_fedavg");
}

// two-shot FedAvg with failure detection (TwoShotArgs::deadline_ns): the coordinator's arrived-set decision travels through
// every rank's decision ring, the result is also pushed into every rank's second arena
void twoshot_fedavg_deadline(std::vector<int64_t> work, std::vector<int64_t> shadow, std::vector<int64_t> chunk_flags,
                             int64_t arrive_flags, int64_t weights, int64_t theta_prev, int64_t epoch, int64_t select_mask,
                             double server_lr, int64_t n, int64_t chunk_elems, int64_t rank, int64_t n_blocks,
                             std::vector<int64_t> peer_arrive, bool wait_all, int64_t mc_work, int64_t mc_shadow,
                             double deadline_ms, std::vector<int64_t> decision, std::vector<int64_t> global_copy) {
  TwoShotArgs a = make_twoshot_args(work, shadow, chunk_flags, arrive_flags, weights, theta_prev, epoch, select_mask, server_lr, n,
                                    chunk_elems, rank, peer_arrive, wait_all, mc_work, mc_shadow, 0, 0.0);
  TORCH_CHECK(deadline_ms > 0 && decision.size() == work.size() && global_copy.size() == work.size(),
              "deadline mode needs a decision ring and a second arena on every rank");
  a.deadline_ns = (unsigned long long)(deadline_ms * 1e6);
  a.true_weights = a.weights;
  for (int k = 0; k < a.world; ++k) {
    a.decision[k] = ptr_of<uint32_t>(decision[k]);
    a.global_copy[k] = ptr_of<float>(global_copy[k]);
  }
  check(launch_twoshot_fedavg(a, (int)n_blocks, cur_stream()), "twoshot_fedavg (deadline)");
}

void twoshot_resync(int64_t decision_ring, int64_t prev_epoch, int64_t rank, int64_t work, int64_t shadow, int64_t global_copy,
                    int64_t n, int64_t n_blocks) {
  check(launch_twoshot_resync(ptr_of<const uint32_t>(decision_ring), (uint32_t)prev_epoch, (int)rank, ptr_of<float>(work), ptr_of<void>(shadow),
                              ptr_of<const float>(global_copy), n, (int)n_blocks, cur_stream()), "twoshot_resync");
}

void reduce_push(int64_t slots, int64_t k, int64_t stride, int64_t n, int64_t dst, int64_t losses, int64_t loss_dst,
                 int64_t flag, int64_t value, int64_t counter, int64_t n_blocks) {
  check(launch_reduce_push(ptr_of<const float>(slots), (int)k, stride, n, ptr_of<float>(dst), ptr_of<const float>(losses),
                           ptr_of<float>(loss_dst), ptr_of<uint32_t>(flag), (uint32_t)value, ptr_of<uint32_t>(counter),
                           (int)n_blocks, cur_stream()), "reduce_push");
}
void set_flag(int64_t flag, int64_t value) { check(launch_set_flag(ptr_of<uint32_t>(flag), (uint32_t)value, cur_stream()), "set_flag"); }
void wait_flag(int64_t flag, int64_t value) { check(launch_wait_flag(ptr_of<const uint32_t>(flag), (uint32_t)value, cur_stream()), "wait_flag"); }
void wait_flags(int64_t flags, int64_t count, int64_t value) { check(launch_wait_flags(ptr_of<const uint32_t>(flags), (int)count, (uint32_t)value, cur_stream()), "wait_flags"); }
void wait_flags_dev(int64_t flags, int64_t count, int64_t value_ptr) { check(launch_wait_flags_dev(ptr_of<const uint32_t>(flags), (int)count, ptr_of<const uint32_t>(value_ptr), cur_stream()), "wait_flags_dev"); }
void signal_peers(std::vector<int64_t> flags, int64_t value) {
  PeerFlags f;
  std::memset(&f, 0, sizeof(f));
  TORCH_CHECK(flags.size() <= 16, "world");
  for (size_t k = 0; k < flags.size(); ++k) f.ptr[k] = ptr_of<uint32_t>(flags[k]);
  check(launch_signal_peers(f, (int)flags.size(), (uint32_t)value, cur_stream()), "signal_peers");
}
void p2p_copy(int64_t dst, int64_t src, int64_t n, int64_t flag, int64_t flag_value, int64_t n_blocks) {
  check(launch_p2p_copy(ptr_of<float>(dst), ptr_of<const float>(src), n, ptr_of<uint32_t>(flag), (uint32_t)flag_value, (int)n_blocks, cur_stream()), "p2p_copy");
}

// ---- symmetric memory via CUDA IPC (fallback when torch symmetric memory is unavailable) -----------------
int64_t ipc_alloc(int64_t bytes) {
  void* p = nullptr;
  check(cudaMalloc(&p, (size_t)bytes), "cudaMalloc");
  check(cudaMemset(p, 0, (size_t)bytes), "cudaMemset");
  return (int64_t)reinterpret_cast<uintptr_t>(p);
}
void ipc_free(int64_t p) { cudaFree(ptr_of<void>(p)); }
py::bytes ipc_get_handle(int64_t p) {
  cudaIpcMemHandle_t h;
  check(cudaIpcGetMemHandle(&h, ptr_of<void>(p)), "cudaIpcGetMemHandle");
  return py::bytes(reinterpret_cast<const char*>(&h), sizeof(h));
}
int64_t ipc_open_handle(py::bytes handle) {
  std::string s = handle;
  TORCH_CHECK(s.size() == sizeof(cudaIpcMemHandle_t), "bad handle size");
  cudaIpcMemHandle_t h;
  std::memcpy(&h, s.data(), sizeof(h));
  void* p = nullptr;
  check(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
  return (int64_t)reinterpret_cast<uintptr_t>(p);
}
void ipc_close_handle(int64_t p) { cudaIpcCloseMemHandle(ptr_of<void>(p)); }
bool can_access_peer(int64_t dev, int64_t peer) {
  int ok = 0;
  cudaDeviceCanAccessPeer(&ok, (int)dev, (int)peer);
  return ok != 0;
}
void enable_peer_access(int64_t peer) {
  cudaError_t e = cudaDeviceEnablePeerAccess((int)peer, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return; }
  check(e, "cudaDeviceEnablePeerAccess");
}
torch::Tensor tensor_from_ptr(int64_t p, int64_t numel, int64_t dtype_code, int64_t device_index) {
  at::ScalarType st = dtype_code == 0 ? at::kFloat : dtype_code == 1 ? at::kBFloat16 : dtype_code == 2 ? at::kInt : at::kByte;
  auto opts = torch::TensorOptions().dtype(st).device(torch::kCUDA, (int)device_index);
  return torch::from_blob(ptr_of<void>(p), {numel}, [](void*) {}, opts);
}

#include "produced_bindings.inc"
void produced_mark(int64_t sig, int64_t chunk_elems, int64_t lo, int64_t hi) {
  int shift = 0;
  while (((int64_t)1 << shift) < chunk_elems) ++shift;
  check(launch_produced_mark(ptr_of<const ProducedSignal>(sig), shift, lo, hi, cur_stream()), "produced_mark");
}

// ---- tcgen05 GEMM -----------------------------------------------------------------------------------------
void gemm_tcgen05(torch::Tensor A, torch::Tensor B, c10::optional<torch::Tensor> bias, bool relu,
                  c10::optional<torch::Tensor> relu_mask, c10::optional<torch::Tensor> out_bf16,
                  c10::optional<torch::Tensor> out_f32, c10::optional<torch::Tensor> out_bf16_t,
                  c10::optional<torch::Tensor> sgd_master, double sgd_lr, c10::optional<torch::Tensor> sgd_shadow,
                  c10::optional<torch::Tensor> sgd_shadow_t, c10::optional<torch::Tensor> colsum,
                  int64_t ready_flags, int64_t ready_epoch, int64_t ready_chunk_elems, int64_t ready_elem_offset, int64_t tile_n,
                  int64_t ready_epoch_ptr, int64_t cluster, int64_t split_k, c10::optional<torch::Tensor> split_out,
                  int64_t mn_m, bool b_kn, c10::optional<torch::Tensor> addend, std::vector<int64_t> conv,
                  std::vector<int64_t> produced) {
  TORCH_CHECK(A.is_cuda() && B.is_cuda() && A.scalar_type() == at::kBFloat16 && B.scalar_type() == at::kBFloat16, "A,B must be CUDA bf16");
  TORCH_CHECK(A.dim() == 2 && B.dim() == 2 && A.is_contiguous() && B.is_contiguous(), "A, B must be contiguous matrices");
  // mn_m > 0: "MN-major" operands A[K, a_cols], B[K, N] (C = A^T B, M = mn_m >= a_cols);
  // b_kn:     A[M, K] K-major, B[b_rows >= K, N] (C = A B[:K]);   else A[M, K], B[N, K] (C = A B^T)
  const bool mn = mn_m > 0;
  TORCH_CHECK(!(mn && b_kn), "mn_m and b_kn are exclusive");
  TORCH_CHECK(!conv.empty() || (mn ? A.size(0) == B.size(0) : (b_kn ? A.size(1) <= B.size(0) : A.size(1) == B.size(1))),
              mn ? "A[K,a_cols], B[K,N]" : (b_kn ? "A[M,K], B[>=K,N]" : "A[M,K], B[N,K]"));
  c10::cuda::CUDAGuard guard(A.device());
  // conv (implicit GEMM) = [mode, flip, C, KH, KW, pad, H, W, n_images, b_rows_per_tap, M, N, K, b_mn]: A is the NHWC activation
  // [n_images*H*W, C] read through a 4-D tensor map, B the other operand (mode 1: K-major weights; mode 2: dz [pixels, a_cols])
  const bool is_conv = !conv.empty();
  TORCH_CHECK(!is_conv || (conv.size() == 14 && !mn && !b_kn), "conv = 14 ints, exclusive with mn_m / b_kn");
  const int M = is_conv ? (int)conv[10] : (mn ? (int)mn_m : (int)A.size(0));
  const int N = is_conv ? (int)conv[11] : ((mn || b_kn) ? (int)B.size(1) : (int)B.size(0));
  const int K = is_conv ? (int)conv[12] : (mn ? (int)A.size(0) : (int)A.size(1));
  GemmEpilogue ep;
  std::memset(&ep, 0, sizeof(ep));
  auto chk = [&](const c10::optional<torch::Tensor>& t, at::ScalarType st, int64_t r, int64_t c, const char* name) -> void* {
    if (!t.has_value()) return nullptr;
    TORCH_CHECK(t->is_cuda() && t->scalar_type() == st && t->is_contiguous(), name, ": dtype/contiguity");
    TORCH_CHECK(t->numel() == r * c, name, ": numel");
    return t->data_ptr();
  };
  ep.bias = (const float*)chk(bias, at::kFloat, 1, N, "bias");
  ep.relu = relu ? 1 : 0;
  ep.relu_mask = chk(relu_mask, at::kBFloat16, M, N, "relu_mask");
  ep.out_bf16 = chk(out_bf16, at::kBFloat16, M, N, "out_bf16");
  ep.out_f32 = (float*)chk(out_f32, at::kFloat, M, N, "out_f32");
  ep.out_bf16_t = chk(out_bf16_t, at::kBFloat16, N, M, "out_bf16_t");
  ep.sgd_master = (float*)chk(sgd_master, at::kFloat, M, N, "sgd_master");
  ep.sgd_lr = (float)sgd_lr;
  ep.sgd_shadow = chk(sgd_shadow, at::kBFloat16, M, N, "sgd_shadow");
  ep.sgd_shadow_t = chk(sgd_shadow_t, at::kBFloat16, N, M, "sgd_shadow_t");
  ep.colsum = (float*)chk(colsum, at::kFloat, M / 32, N, "colsum (partials [M/32, N])");
  ep.ready_flags = ptr_of<const uint32_t>(ready_flags);
  ep.ready_epoch = (uint32_t)ready_epoch;
  ep.ready_epoch_ptr = ptr_of<const uint32_t>(ready_epoch_ptr);
  ep.ready_chunk_elems = ready_chunk_elems > 0 ? ready_chunk_elems : 1;
  ep.ready_elem_offset = ready_elem_offset;
  ep.tile_n = (int)tile_n;
  ep.cluster = (int)cluster;
  ep.pdl = pdl_enabled() ? 1 : 0;      // programmatic dependent launch (on unless COLEARN_PDL=0)
  // produced = [ProducedSignal* (device), arena element of sgd_master[0, 0], max_ctas]: fused wgrad -> FedAvg reduce
  if (!produced.empty()) {
    TORCH_CHECK(produced.size() == 3, "produced = [signal_ptr, elem_offset, max_ctas]");
    ep.produced = ptr_of<const ProducedSignal>(produced[0]);
    ep.produced_elem_offset = produced[1];
    ep.max_ctas = (int)produced[2];
  }
  if (split_k > 1) {
    TORCH_CHECK(split_out.has_value() && split_out->is_cuda() && split_out->scalar_type() == at::kFloat && split_out->is_contiguous() &&
                split_out->numel() >= split_k * (int64_t)M * N, "split_out must be a contiguous CUDA fp32 tensor with >= split_k*M*N elements");
    ep.split_k = (int)split_k;
    ep.split_out = split_out->data_ptr<float>();
  }
  ep.addend = chk(addend, at::kBFloat16, M, N, "addend");
  if (is_conv) {
    convops::ConvAddr& g = ep.conv;
    g.mode = (int)conv[0]; g.flip = (int)conv[1]; g.C = (int)conv[2]; g.KH = (int)conv[3]; g.KW = (int)conv[4]; g.pad = (int)conv[5];
    const int H = (int)conv[6], W = (int)conv[7];
    g.HW = H * W; g.n_images = (int)conv[8]; g.b_rows_per_tap = (int)conv[9]; g.b_mn = (int)conv[13];
    TORCH_CHECK(A.numel() == (int64_t)g.n_images * H * W * g.C, "activation must be [n_images*H*W, C]");
    static const int dbg_lbo = std::getenv("COLEARN_UMMA_MN_LBO") ? std::atoi(std::getenv("COLEARN_UMMA_MN_LBO")) : 0;
    static const int dbg_sbo = std::getenv("COLEARN_UMMA_MN_SBO") ? std::atoi(std::getenv("COLEARN_UMMA_MN_SBO")) : 0;
    ep.mn_lbo = dbg_lbo;
    ep.mn_sbo = dbg_sbo;
    cudaError_t e = launch_gemm_tcgen05_conv(A.data_ptr(), g.n_images, H, W, B.data_ptr(), (int)B.size(0), (int)B.size(1), M, N, K, ep, cur_stream());
    TORCH_CHECK(e == cudaSuccess, "gemm_tcgen05 (implicit conv): ", cudaGetErrorString(e), " (", gemm_tcgen05_last_error(), ")");
    return;
  }
  if (mn || b_kn) {
    static const int dbg_lbo = std::getenv("COLEARN_UMMA_MN_LBO") ? std::atoi(std::getenv("COLEARN_UMMA_MN_LBO")) : 0;
    static const int dbg_sbo = std::getenv("COLEARN_UMMA_MN_SBO") ? std::atoi(std::getenv("COLEARN_UMMA_MN_SBO")) : 0;
    ep.mn_lbo = dbg_lbo;
    ep.mn_sbo = dbg_sbo;
    cudaError_t e = launch_gemm_tcgen05_mn(A.data_ptr(), mn ? 1 : 0, (int)A.size(1), B.data_ptr(), (int)B.size(0), M, N, K, ep, cur_stream());
    TORCH_CHECK(e == cudaSuccess, "gemm_tcgen05 (mn-major): ", cudaGetErrorString(e), " (", gemm_tcgen05_last_error(), ")");
    return;
  }
  cudaError_t e = launch_gemm_tcgen05(A.data_ptr(), B.data_ptr(), M, N, K, ep, cur_stream());
  TORCH_CHECK(e == cudaSuccess, "gemm_tcgen05: ", cudaGetErrorString(e), " (", gemm_tcgen05_last_error(), ")");
}

// ---- NHWC conv / BatchNorm / pooling (convnet.cu); wrappers shared with the host emulator ------------------
struct ConvCudaExec {
  static constexpr bool kCuda = true;
  static void im2col(const convops::Im2colArgs& a) { check(launch_im2col(a, cur_stream()), "im2col"); }
  static void col2im(const convops::Col2imArgs& a) { check(launch_col2im(a, cur_stream()), "col2im"); }
  static void bn_reduce(const convops::BnReduceArgs& a) { check(launch_bn_reduce(a, cur_stream()), "bn_reduce"); }
  static void bn_finalize(const convops::BnFinalizeArgs& a) { check(launch_bn_finalize(a, cur_stream()), "bn_finalize"); }
  static void bn_reduce_finalize(const convops::BnFusedArgs& a) { check(launch_bn_reduce_finalize(a, cur_stream()), "bn_reduce_finalize"); }
  static void bn_apply(const convops::BnApplyArgs& a) { check(launch_bn_apply(a, cur_stream()), "bn_apply"); }
  static void bn_bwd(const convops::BnBwdArgs& a) { check(launch_bn_bwd(a, cur_stream()), "bn_bwd"); }
  static void maxpool_fwd(const convops::PoolArgs& a) { check(launch_maxpool_fwd(a, cur_stream()), "maxpool_fwd"); }
  static void maxpool_bwd(const convops::PoolArgs& a) { check(launch_maxpool_bwd(a, cur_stream()), "maxpool_bwd"); }
  static void avgpool_fwd(const convops::AvgPoolArgs& a) { check(launch_avgpool_fwd(a, cur_stream()), "avgpool_fwd"); }
  static void avgpool_bwd(const convops::AvgPoolArgs& a) { check(launch_avgpool_bwd(a, cur_stream()), "avgpool_bwd"); }
  static void pack(const convops::PackArgs& a) { check(launch_pack(a, cur_stream()), "pack"); }
  static void splitk_reduce(const convops::SplitKReduceArgs& a) { check(launch_splitk_reduce(a, cur_stream()), "splitk_reduce"); }
};

}  // namespace

#include "conv_bindings.inc"

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "colearn_federated_learning_b200 sm_100a kernels";
  m.def("make_client_desc", &make_client_desc);
  m.def("set_spin_limit", &set_spin_limit);
  m.def("scale_inplace", &scale_inplace);
  m.def("client_desc_size", &client_desc_size);
  m.def("mlp_local_sgd", &mlp_local_sgd);
  m.def("mlp_net_params", &mlp_net_params);
  m.def("mlp_smem_bytes", &mlp_smem_bytes);
  m.def("mlp_local_sgd_generic", &mlp_local_sgd_generic);
  m.def("mlp_generic_plan", &generic_plan);
  m.def("mlp_forward", &mlp_forward);
  m.def("sgd_step", &sgd_step);
  m.def("fedavg_apply", &fedavg_apply);
  m.def("fedavg_flat", &fedavg_flat);
  m.def("sigmoid_bce", &sigmoid_bce);
  m.def("sse_loss", &sse_loss);
  m.def("softmax_xent", &softmax_xent);
  m.def("softmax_xent_head", &softmax_xent_head);
  m.def("eval_binary", &eval_binary);
  m.def("argmax_rows", &argmax_rows);
  m.def("minmax_scale", &minmax_scale);
  m.def("feistel_permutation", &feistel_permutation);
  m.def("fp32_to_bf16", &fp32_to_bf16);
  m.def("fp32_to_bf16_into", &fp32_to_bf16_into);
  m.def("l2_flush", &l2_flush);
  m.def("bias_sgd_from_partials", &bias_sgd_from_partials);
  m.def("fix_precision", &fix_precision);
  m.def("float_precision", &float_precision);
  m.def("ring_matmul", &ring_matmul);
  m.def("transpose_bf16", &transpose_bf16);
  m.def("star_round", &star_round);
  m.def("twoshot_fedavg", &twoshot_fedavg);
  m.def("twoshot_fedavg_deadline", &twoshot_fedavg_deadline);
  m.def("twoshot_resync", &twoshot_resync);
  m.def("produced_signal_pack", &produced_signal_pack);
  m.def("produced_mark", &produced_mark);
  m.def("reduce_push", &reduce_push);
  m.def("set_flag", &set_flag);
  m.def("wait_flag", &wait_flag);
  m.def("wait_flags", &wait_flags);
  m.def("wait_flags_dev", &wait_flags_dev);
  m.def("signal_peers", &signal_peers);
  m.def("p2p_copy", &p2p_copy);
  m.def("ipc_alloc", &ipc_alloc);
  m.def("ipc_free", &ipc_free);
  m.def("ipc_get_handle", &ipc_get_handle);
  m.def("ipc_open_handle", &ipc_open_handle);
  m.def("ipc_close_handle", &ipc_close_handle);
  m.def("can_access_peer", &can_access_peer);
  m.def("enable_peer_access", &enable_peer_access);
  m.def("tensor_from_ptr", &tensor_from_ptr);
  m.def("gemm_tcgen05", &gemm_tcgen05);
  convbind::register_ops<ConvCudaExec>(m);
}
