// Python face of the SIMT-on-CPU build: mlp_persistent.cu (+ mlp_v2.inc), elementwise.cu and comm.cu — the kernel
// sources themselves — are compiled with g++ through host_shim.h (simt_mlp.cpp / simt_elementwise.cpp / simt_comm.cpp,
// one OS thread per CUDA thread) and driven here through the same launch_* entry points bindings.cpp uses on a GPU.
// Tests only (ops/build.py::build_simt_emul, tests/test_simt_emul.py).
#define COLEARN_HOST_SHIM 1
#include <torch/extension.h>

#include "colearn_kernels.h"

#include <cstring>

namespace py = pybind11;

namespace {
using torch::Tensor;

const float* fptr(const Tensor& t, const char* name) {
  TORCH_CHECK(!t.is_cuda() && t.scalar_type() == at::kFloat && t.is_contiguous(), name, ": contiguous CPU fp32");
  return t.data_ptr<float>();
}

// K clients (one emulated CTA each, run one after the other).  theta_outs[i] may alias theta_in.
// Returns losses [K, 2] = {last, mean}; flags (int32 [K], optional) receive signal_value = 7 + i.
Tensor mlp_local_sgd(int64_t net_kind, Tensor theta_in, std::vector<Tensor> theta_outs, std::vector<Tensor> xs, std::vector<Tensor> ys,
                     std::vector<c10::optional<Tensor>> perms, int64_t batch_size, int64_t epochs, int64_t max_steps, int64_t loss,
                     double lr, int64_t variant, std::vector<double> out_scales, bool delta_mode, c10::optional<Tensor> flags,
                     int64_t perm_seed, int64_t perm_row0, c10::optional<Tensor> perm_scratch) {
  const size_t K = xs.size();
  TORCH_CHECK(K >= 1 && ys.size() == K && perms.size() == K && theta_outs.size() == K && out_scales.size() == K, "one entry per client");
  const int P = colearn::mlp_net_num_params((int)net_kind);
  TORCH_CHECK(P > 0 && theta_in.numel() == P, "theta_in must hold ", P, " parameters");
  Tensor losses = torch::zeros({(int64_t)K, 2}, torch::kFloat);
  std::vector<colearn::ClientDesc> descs(K);
  for (size_t i = 0; i < K; ++i) {
    colearn::ClientDesc& d = descs[i];
    memset(&d, 0, sizeof(d));
    d.x = fptr(xs[i], "x");
    d.y = fptr(ys[i], "y");
    TORCH_CHECK(xs[i].dim() == 2 && ys[i].dim() == 2 && xs[i].size(0) == ys[i].size(0), "x [n, d_in], y [n, y_dim]");
    d.n = (int)xs[i].size(0);
    d.y_dim = (int)ys[i].size(1);
    d.perm_rows = 1;
    if (perms[i].has_value()) {
      const Tensor& p = *perms[i];
      TORCH_CHECK(!p.is_cuda() && p.scalar_type() == at::kInt && p.is_contiguous() && p.dim() == 2 && p.size(1) == d.n, "perm int32 [rows, n]");
      d.perm = p.data_ptr<int>();
      d.perm_rows = (int)p.size(0);
    } else if (perm_seed != 0) {                                   // in-kernel shuffle (ClientDesc::perm_seed): client i keys on seed + i
      d.perm_seed = (uint64_t)(perm_seed + (int64_t)i);
      d.perm_row0 = (int)perm_row0;
      if (perm_scratch.has_value()) {
        TORCH_CHECK(perm_scratch->scalar_type() == at::kInt && perm_scratch->is_contiguous() && perm_scratch->dim() == 2 &&
                    perm_scratch->size(0) == (int64_t)K && perm_scratch->size(1) >= epochs * (int64_t)d.n, "perm_scratch int32 [K, epochs * n]");
        d.perm_scratch = perm_scratch->data_ptr<int>() + (int64_t)i * perm_scratch->size(1);
      }
    }
    d.theta_in = fptr(theta_in, "theta_in");
    TORCH_CHECK(theta_outs[i].numel() == P, "theta_out size");
    d.theta_out = const_cast<float*>(fptr(theta_outs[i], "theta_out"));
    d.loss_out = losses.data_ptr<float>() + 2 * i;
    d.out_scale = (float)out_scales[i];
    d.delta_mode = delta_mode ? 1 : 0;
    if (flags.has_value()) {
      TORCH_CHECK(flags->scalar_type() == at::kInt && flags->is_contiguous() && flags->numel() >= (int64_t)K, "flags int32 [K]");
      d.signal_flag = reinterpret_cast<uint32_t*>(flags->data_ptr<int>()) + i;
      d.signal_value = 7u + (uint32_t)i;
    }
  }
  colearn::SgdHyper hp;
  hp.batch_size = (int)batch_size;
  hp.epochs = (int)epochs;
  hp.max_steps = (int)max_steps;
  hp.loss = (int)loss;
  hp.lr = (float)lr;
  hp.variant = (int)variant;
  {
    py::gil_scoped_release nogil;
    cudaError_t e = colearn::launch_mlp_local_sgd((int)net_kind, descs.data(), (int)K, hp, nullptr);
    TORCH_CHECK(e == cudaSuccess, "launch_mlp_local_sgd (host shim) failed");
  }
  return losses;
}

// mlp_generic.cu: descs is a CPU uint8 tensor of ClientDescs packed by make_client_desc from host pointers; the clusters run one
// after the other, the CTAs of a cluster concurrently.  Same arguments as the CUDA binding.
void mlp_local_sgd_generic(std::vector<int64_t> dims, bool sigmoid, Tensor descs, int64_t desc_offset, int64_t n_clients, int64_t batch_size,
                           int64_t epochs, int64_t max_steps, int64_t loss, double lr, int64_t cluster) {
  TORCH_CHECK(!descs.is_cuda() && descs.scalar_type() == at::kByte && descs.is_contiguous(), "descs must be CPU uint8");
  TORCH_CHECK((desc_offset + n_clients) * (int64_t)sizeof(colearn::ClientDesc) <= descs.numel(), "descs too small");
  TORCH_CHECK(dims.size() >= 2 && dims.size() <= 9, "dims: 2..9 widths");
  std::vector<int> d(dims.begin(), dims.end());
  colearn::SgdHyper hp;
  hp.batch_size = (int)batch_size; hp.epochs = (int)epochs; hp.max_steps = (int)max_steps;
  hp.loss = (int)loss; hp.lr = (float)lr; hp.variant = 0;
  const colearn::ClientDesc* p = reinterpret_cast<const colearn::ClientDesc*>(descs.data_ptr<uint8_t>()) + desc_offset;
  py::gil_scoped_release nogil;
  TORCH_CHECK(cudaSuccess == colearn::launch_mlp_local_sgd_generic(d.data(), (int)d.size() - 1, sigmoid ? 1 : 0, p, (int)n_clients, hp, (int)cluster, nullptr), "launch_mlp_local_sgd_generic (host shim) failed");
}
int64_t mlp_generic_plan(std::vector<int64_t> dims, int64_t batch_size, int64_t cluster) {
  if (dims.size() < 2 || dims.size() > 9) return -1;
  std::vector<int> d(dims.begin(), dims.end());
  return colearn::mlp_generic_plan(d.data(), (int)d.size() - 1, (int)batch_size, (int)cluster, nullptr);
}
#include "client_desc.inc"

Tensor mlp_forward(int64_t net_kind, Tensor theta, Tensor x, int64_t d_out) {
  TORCH_CHECK(x.dim() == 2, "x [n, d_in]");
  Tensor out = torch::zeros({x.size(0), d_out}, torch::kFloat);
  {
    py::gil_scoped_release nogil;
    cudaError_t e = colearn::launch_mlp_forward((int)net_kind, fptr(theta, "theta"), fptr(x, "x"), out.data_ptr<float>(), (int)x.size(0), nullptr);
    TORCH_CHECK(e == cudaSuccess, "launch_mlp_forward (host shim) failed");
  }
  return out;
}

// ---- elementwise.cu ---------------------------------------------------------------------------------------------
#define CK(expr) TORCH_CHECK((expr) == cudaSuccess, "launch failed: " #expr)
float* fmut(Tensor& t, const char* name) { return const_cast<float*>(fptr(t, name)); }

void sgd_step(Tensor p, Tensor g, double lr) { CK(colearn::launch_sgd_step(fmut(p, "p"), fptr(g, "g"), (float)lr, p.numel(), nullptr)); }
void fedavg_apply(Tensor theta, Tensor slots, Tensor w, double server_lr) {
  TORCH_CHECK(slots.dim() == 2 && slots.size(1) == theta.numel() && w.numel() == slots.size(0), "slots [K, P], weights [K]");
  CK(colearn::launch_fedavg_apply(fmut(theta, "theta"), fptr(slots, "slots"), slots.size(1), fptr(w, "w"), (int)slots.size(0),
                                  (float)server_lr, theta.numel(), nullptr));
}
Tensor fedavg_flat(Tensor slots, Tensor w) {
  Tensor out = torch::zeros({slots.size(1)}, torch::kFloat);
  CK(colearn::launch_fedavg_flat(out.data_ptr<float>(), fptr(slots, "slots"), slots.size(1), fptr(w, "w"), (int)slots.size(0), slots.size(1), nullptr));
  return out;
}
std::tuple<Tensor, Tensor> sigmoid_bce(Tensor z, Tensor y) {
  Tensor dz = torch::zeros_like(z), loss = torch::zeros({}, torch::kFloat);
  CK(colearn::launch_sigmoid_bce(fptr(z, "z"), fptr(y, "y"), dz.data_ptr<float>(), loss.data_ptr<float>(), z.numel(), nullptr));
  return {loss, dz};
}
std::tuple<Tensor, Tensor> sse_loss(Tensor out, Tensor y, double scale) {
  Tensor dz = torch::zeros_like(out), loss = torch::zeros({}, torch::kFloat);
  CK(colearn::launch_sse(fptr(out, "out"), fptr(y, "y"), dz.data_ptr<float>(), loss.data_ptr<float>(), out.numel(), (float)scale, nullptr));
  return {loss, dz};
}
std::tuple<Tensor, Tensor> softmax_xent(Tensor logits, Tensor labels) {
  TORCH_CHECK(logits.dim() == 2 && labels.scalar_type() == at::kLong && labels.numel() == logits.size(0), "logits [R, C], labels int64 [R]");
  Tensor dl = torch::zeros_like(logits), loss = torch::zeros({}, torch::kFloat);
  CK(colearn::launch_softmax_xent(fptr(logits, "logits"), 0, labels.data_ptr<int64_t>(), dl.data_ptr<float>(), nullptr, loss.data_ptr<float>(),
                                  (int)logits.size(0), (int)logits.size(1), nullptr));
  return {loss, dl};
}
Tensor softmax_xent_head(Tensor logits, Tensor labels, int64_t rows, int64_t cols, c10::optional<Tensor> dl_f32, c10::optional<Tensor> dl_bf16,
                         c10::optional<Tensor> db) {
  TORCH_CHECK(!logits.is_cuda() && logits.dim() == 2 && logits.stride(1) == 1 && labels.scalar_type() == at::kLong && labels.is_contiguous(), "operands");
  const bool bf16 = logits.scalar_type() == at::kBFloat16;
  Tensor loss = torch::zeros({}, torch::kFloat);
  CK(colearn::launch_softmax_xent_head(logits.data_ptr(), bf16 ? 1 : 0, (int)logits.stride(0), labels.data_ptr<int64_t>(),
                                       dl_f32.has_value() ? dl_f32->data_ptr<float>() : nullptr, dl_f32.has_value() ? (int)dl_f32->stride(0) : 0,
                                       dl_bf16.has_value() ? dl_bf16->data_ptr() : nullptr, dl_bf16.has_value() ? (int)dl_bf16->stride(0) : 0,
                                       db.has_value() ? db->data_ptr<float>() : nullptr, loss.data_ptr<float>(), (int)rows, (int)cols, nullptr));
  return loss;
}
std::tuple<Tensor, Tensor> eval_binary(Tensor p, Tensor y) {
  Tensor loss = torch::zeros({}, torch::kFloat), correct = torch::zeros({}, torch::kInt);
  CK(colearn::launch_eval_binary(fptr(p, "p"), fptr(y, "y"), loss.data_ptr<float>(), correct.data_ptr<int>(), p.numel(), nullptr));
  return {loss, correct};
}
Tensor argmax_rows(Tensor x) {
  Tensor out = torch::zeros({x.size(0), 1}, torch::kLong);
  CK(colearn::launch_argmax_rows(fptr(x, "x"), out.data_ptr<int64_t>(), (int)x.size(0), (int)x.size(1), nullptr));
  return out;
}
Tensor minmax_scale(Tensor x) {
  Tensor out = torch::zeros_like(x);
  CK(colearn::launch_minmax_scale(fptr(x, "x"), out.data_ptr<float>(), (int)x.size(0), (int)x.size(1), nullptr));
  return out;
}
Tensor feistel_permutation(int64_t n, int64_t rows, int64_t seed) {
  Tensor out = torch::zeros({rows, n}, torch::kInt);
  CK(colearn::launch_feistel_permutation(out.data_ptr<int>(), (int)n, (int)rows, (uint64_t)seed, nullptr));
  return out;
}
Tensor transpose_bf16(Tensor x) {
  TORCH_CHECK(x.scalar_type() == at::kBFloat16 && x.is_contiguous() && x.dim() == 2, "bf16 matrix");
  Tensor out = torch::zeros({x.size(1), x.size(0)}, x.options());
  CK(colearn::launch_transpose_bf16(x.data_ptr(), out.data_ptr(), (int)x.size(0), (int)x.size(1), nullptr));
  return out;
}
Tensor ring_matmul(Tensor a, Tensor b) {
  TORCH_CHECK(a.scalar_type() == at::kLong && b.scalar_type() == at::kLong && a.is_contiguous() && b.is_contiguous(), "int64 matrices");
  Tensor c = torch::zeros({a.size(0), b.size(1)}, torch::kLong);
  CK(colearn::launch_ring_matmul(reinterpret_cast<const long long*>(a.data_ptr<int64_t>()), reinterpret_cast<const long long*>(b.data_ptr<int64_t>()),
                                 reinterpret_cast<long long*>(c.data_ptr<int64_t>()), (int)a.size(0), (int)a.size(1), (int)b.size(1), nullptr));
  return c;
}

// ---- comm.cu: W emulated ranks = W sets of buffers in this process; kernels of different ranks run one after the other -----
// Coordinator-side star round: slots [W, P] (already holding w_k * theta_k), arrive flags int32 [W], inboxes [W, P] (row k =
// rank k's inbox), bcast flags int32 [W].  Returns the arrived mask (deadline mode) or the select mask.
int64_t star_round(Tensor theta, Tensor slots, Tensor arrive, int64_t arrive_epoch, Tensor inboxes, Tensor bcast_flags, int64_t bcast_epoch,
                   int64_t select_mask, double server_lr, bool do_reduce, bool do_bcast, int64_t n_blocks, double timeout_ms,
                   std::vector<double> weights) {
  const int W = (int)slots.size(0);
  colearn::StarRoundArgs a;
  memset(&a, 0, sizeof(a));
  a.theta = fmut(theta, "theta");
  a.slots = fptr(slots, "slots");
  a.slot_stride = slots.size(1);
  a.arrive_flags = reinterpret_cast<const uint32_t*>(arrive.data_ptr<int>());
  a.arrive_epoch = (uint32_t)arrive_epoch;
  for (int k = 0; k < W; ++k) {
    a.peer_inbox[k] = inboxes.data_ptr<float>() + (int64_t)k * inboxes.size(1);
    a.peer_bcast_flag[k] = reinterpret_cast<uint32_t*>(bcast_flags.data_ptr<int>()) + k;
    a.weights[k] = k < (int)weights.size() ? (float)weights[k] : 0.f;
  }
  a.bcast_epoch = (uint32_t)bcast_epoch;
  a.select_mask = (uint32_t)select_mask;
  a.world = W;
  a.server_lr = (float)server_lr;
  a.n = theta.numel();
  a.do_reduce = do_reduce ? 1 : 0;
  a.do_bcast = do_bcast ? 1 : 0;
  static uint32_t counter = 0, decision[2] = {0, 0};
  a.grid_counter = &counter;
  a.timeout_ns = (unsigned long long)(timeout_ms * 1e6);
  a.decision = decision;
  {
    py::gil_scoped_release nogil;
    CK(colearn::launch_star_round(a, (int)n_blocks, nullptr));
  }
  return timeout_ms > 0 && do_reduce ? (int64_t)decision[1] : select_mask;
}

// One rank's two-shot kernel (P2P path): works [W, n] (row k = rank k's fp32 arena), shadows [W, n] bf16 or none, chunk flags
// int32 [W, n_chunks]; `arrive` (this rank's int32 [W]) must already carry `epoch` for every selected rank.
void twoshot_fedavg(int64_t rank, Tensor works, c10::optional<Tensor> shadows, Tensor chunk_flags, Tensor arrive, Tensor weights,
                    c10::optional<Tensor> theta_prev, int64_t epoch, int64_t select_mask, double server_lr, int64_t chunk_elems, int64_t n_blocks,
                    c10::optional<Tensor> produced, double produced_timeout_s) {
  const int W = (int)works.size(0);
  colearn::TwoShotArgs a;
  memset(&a, 0, sizeof(a));
  for (int k = 0; k < W; ++k) {
    a.work[k] = works.data_ptr<float>() + (int64_t)k * works.size(1);
    a.shadow_bf16[k] = shadows.has_value() ? static_cast<void*>(static_cast<char*>(shadows->data_ptr()) + (int64_t)k * shadows->size(1) * 2) : nullptr;
    a.chunk_flags[k] = reinterpret_cast<uint32_t*>(chunk_flags.data_ptr<int>()) + (int64_t)k * chunk_flags.size(1);
  }
  a.arrive_flags = reinterpret_cast<const uint32_t*>(arrive.data_ptr<int>());
  a.weights = fptr(weights, "weights");
  a.theta_prev = theta_prev.has_value() ? theta_prev->data_ptr<float>() : nullptr;
  a.epoch = (uint32_t)epoch;
  a.select_mask = (uint32_t)select_mask;
  a.server_lr = (float)server_lr;
  a.n = works.size(1);
  a.chunk_elems = chunk_elems;
  a.world = W;
  a.rank = (int)rank;
  if (produced.has_value()) {      // [W (owner), W (producer), n_chunks] int32: this rank's table is produced[rank]
    TORCH_CHECK(produced->dim() == 3 && produced->size(0) == W && produced->size(1) == W && produced->is_contiguous(), "produced");
    a.produced = reinterpret_cast<const uint32_t*>(produced->data_ptr<int>()) + rank * W * produced->size(2);
    a.produced_timeout_ns = produced_timeout_s > 0 ? (unsigned long long)(produced_timeout_s * 1e9) : 0ull;
  }
  {
    py::gil_scoped_release nogil;
    CK(colearn::launch_twoshot_fedavg(a, (int)n_blocks, nullptr));
  }
}

// deadline mode of one emulated rank: decisions int32 [W, 16] (row k = rank k's ring), globals [W, n] (second arenas)
void twoshot_fedavg_deadline(int64_t rank, Tensor works, Tensor globals, Tensor chunk_flags, Tensor arrive, Tensor weights, int64_t epoch,
                             int64_t select_mask, int64_t chunk_elems, int64_t n_blocks, double deadline_ms, Tensor decisions) {
  const int W = (int)works.size(0);
  colearn::TwoShotArgs a;
  memset(&a, 0, sizeof(a));
  for (int k = 0; k < W; ++k) {
    a.work[k] = works.data_ptr<float>() + (int64_t)k * works.size(1);
    a.global_copy[k] = globals.data_ptr<float>() + (int64_t)k * globals.size(1);
    a.chunk_flags[k] = reinterpret_cast<uint32_t*>(chunk_flags.data_ptr<int>()) + (int64_t)k * chunk_flags.size(1);
    a.decision[k] = reinterpret_cast<uint32_t*>(decisions.data_ptr<int>()) + (int64_t)k * decisions.size(1);
  }
  a.arrive_flags = reinterpret_cast<const uint32_t*>(arrive.data_ptr<int>());
  a.weights = a.true_weights = fptr(weights, "weights");
  a.epoch = (uint32_t)epoch;
  a.select_mask = (uint32_t)select_mask;
  a.server_lr = 1.f;
  a.n = works.size(1);
  a.chunk_elems = chunk_elems;
  a.world = W;
  a.rank = (int)rank;
  a.wait_all = 0;      // (the emulated ranks run one after the other: nobody may wait for a later rank's chunks)
  a.deadline_ns = (unsigned long long)(deadline_ms * 1e6);
  py::gil_scoped_release nogil;
  CK(colearn::launch_twoshot_fedavg(a, (int)n_blocks, nullptr));
}

void twoshot_resync(Tensor decision_ring, int64_t prev_epoch, int64_t rank, Tensor work, Tensor global_copy) {
  py::gil_scoped_release nogil;
  CK(colearn::launch_twoshot_resync(reinterpret_cast<const uint32_t*>(decision_ring.data_ptr<int>()), (uint32_t)prev_epoch, (int)rank,
                                    work.data_ptr<float>(), nullptr, global_copy.data_ptr<float>(), work.numel(), 2, nullptr));
}

void reduce_push(Tensor slots, Tensor dst, Tensor losses, Tensor loss_dst, Tensor flag, int64_t value, int64_t n_blocks) {
  static uint32_t counter = 0;
  py::gil_scoped_release nogil;
  CK(colearn::launch_reduce_push(fptr(slots, "slots"), (int)slots.size(0), slots.size(1), slots.size(1), fmut(dst, "dst"), fptr(losses, "losses"),
                                 fmut(loss_dst, "loss_dst"), reinterpret_cast<uint32_t*>(flag.data_ptr<int>()), (uint32_t)value, &counter,
                                 (int)n_blocks, nullptr));
}

#include "produced_bindings.inc"
void produced_mark(int64_t sig, int64_t chunk_elems, int64_t lo, int64_t hi) {
  int shift = 0;
  while (((int64_t)1 << shift) < chunk_elems) ++shift;
  py::gil_scoped_release nogil;
  CK(colearn::launch_produced_mark(reinterpret_cast<const colearn::ProducedSignal*>(static_cast<uintptr_t>(sig)), shift, lo, hi, nullptr));
}

// ---- gemm_tcgen05.cu on the functional tcgen05 / TMA / mbarrier model (tcgen05_host_model.h) ---------------------------------
// Same argument meaning as bindings.cpp::gemm_tcgen05 (minus the cross-GPU ready flags and the cluster modes).
void gemm_tcgen05(Tensor A, Tensor B, c10::optional<Tensor> bias, bool relu, c10::optional<Tensor> relu_mask, c10::optional<Tensor> out_bf16,
                  c10::optional<Tensor> out_f32, c10::optional<Tensor> out_bf16_t, c10::optional<Tensor> sgd_master, double sgd_lr,
                  c10::optional<Tensor> sgd_shadow, c10::optional<Tensor> sgd_shadow_t, c10::optional<Tensor> colsum, int64_t tile_n,
                  int64_t split_k, c10::optional<Tensor> split_out, int64_t mn_m, bool b_kn, c10::optional<Tensor> addend,
                  std::vector<int64_t> conv, std::vector<int64_t> produced) {
  TORCH_CHECK(!A.is_cuda() && !B.is_cuda() && A.scalar_type() == at::kBFloat16 && B.scalar_type() == at::kBFloat16 && A.is_contiguous() &&
              B.is_contiguous() && A.dim() == 2 && B.dim() == 2, "A, B: contiguous CPU bf16 matrices");
  const bool mn = mn_m > 0, is_conv = !conv.empty();
  TORCH_CHECK(!is_conv || conv.size() == 14, "conv = 14 ints");
  const int M = is_conv ? (int)conv[10] : (mn ? (int)mn_m : (int)A.size(0));
  const int N = is_conv ? (int)conv[11] : ((mn || b_kn) ? (int)B.size(1) : (int)B.size(0));
  const int K = is_conv ? (int)conv[12] : (mn ? (int)A.size(0) : (int)A.size(1));
  colearn::GemmEpilogue ep;
  memset(&ep, 0, sizeof(ep));
  auto ptr = [&](const c10::optional<Tensor>& t, at::ScalarType st, int64_t numel, const char* name) -> void* {
    if (!t.has_value()) return nullptr;
    TORCH_CHECK(!t->is_cuda() && t->scalar_type() == st && t->is_contiguous() && t->numel() >= numel, name, ": dtype / size");
    return t->data_ptr();
  };
  ep.bias = (const float*)ptr(bias, at::kFloat, N, "bias");
  ep.relu = relu ? 1 : 0;
  ep.relu_mask = ptr(relu_mask, at::kBFloat16, (int64_t)M * N, "relu_mask");
  ep.out_bf16 = ptr(out_bf16, at::kBFloat16, (int64_t)M * N, "out_bf16");
  ep.out_f32 = (float*)ptr(out_f32, at::kFloat, (int64_t)M * N, "out_f32");
  ep.out_bf16_t = ptr(out_bf16_t, at::kBFloat16, (int64_t)M * N, "out_bf16_t");
  ep.sgd_master = (float*)ptr(sgd_master, at::kFloat, (int64_t)M * N, "sgd_master");
  ep.sgd_lr = (float)sgd_lr;
  ep.sgd_shadow = ptr(sgd_shadow, at::kBFloat16, (int64_t)M * N, "sgd_shadow");
  ep.sgd_shadow_t = ptr(sgd_shadow_t, at::kBFloat16, (int64_t)M * N, "sgd_shadow_t");
  ep.colsum = (float*)ptr(colsum, at::kFloat, (int64_t)(M / 32) * N, "colsum");
  ep.addend = ptr(addend, at::kBFloat16, (int64_t)M * N, "addend");
  ep.ready_chunk_elems = 1;
  ep.tile_n = (int)tile_n;
  if (!produced.empty()) {
    TORCH_CHECK(produced.size() == 3, "produced = [signal_ptr, elem_offset, max_ctas]");
    ep.produced = reinterpret_cast<const colearn::ProducedSignal*>(static_cast<uintptr_t>(produced[0]));
    ep.produced_elem_offset = produced[1];
    ep.max_ctas = (int)produced[2];
  }
  if (split_k > 1) {
    ep.split_k = (int)split_k;
    ep.split_out = (float*)ptr(split_out, at::kFloat, split_k * (int64_t)M * N, "split_out");
    TORCH_CHECK(ep.split_out != nullptr, "split_out");
  }
  cudaError_t e;
  {
    py::gil_scoped_release nogil;
    if (is_conv) {
      colearn::convops::ConvAddr& g = ep.conv;
      g.mode = (int)conv[0]; g.flip = (int)conv[1]; g.C = (int)conv[2]; g.KH = (int)conv[3]; g.KW = (int)conv[4]; g.pad = (int)conv[5];
      const int H = (int)conv[6], W = (int)conv[7];
      g.HW = H * W; g.n_images = (int)conv[8]; g.b_rows_per_tap = (int)conv[9]; g.b_mn = (int)conv[13];
      e = colearn::launch_gemm_tcgen05_conv(A.data_ptr(), g.n_images, H, W, B.data_ptr(), (int)B.size(0), (int)B.size(1), M, N, K, ep, nullptr);
    } else if (mn || b_kn) {
      e = colearn::launch_gemm_tcgen05_mn(A.data_ptr(), mn ? 1 : 0, (int)A.size(1), B.data_ptr(), (int)B.size(0), M, N, K, ep, nullptr);
    } else {
      e = colearn::launch_gemm_tcgen05(A.data_ptr(), B.data_ptr(), M, N, K, ep, nullptr);
    }
  }
  TORCH_CHECK(e == cudaSuccess, "gemm_tcgen05 (host model): ", colearn::gemm_tcgen05_last_error());
}

// ---- convnet.cu: the launchers themselves (grid mapping, two-phase blocks, the ticket-counter BatchNorm reduction) behind the
// torch-facing wrappers of conv_bindings.inc — a third instantiation next to the GPU one and the body emulator ----------------
inline void ck(cudaError_t e, const char* what) { TORCH_CHECK(e == cudaSuccess, what, " failed"); }
struct ConvSimtExec {
  static constexpr bool kCuda = false;
  static void im2col(const colearn::convops::Im2colArgs& a) { ck(colearn::launch_im2col(a, nullptr), "im2col"); }
  static void col2im(const colearn::convops::Col2imArgs& a) { ck(colearn::launch_col2im(a, nullptr), "col2im"); }
  static void bn_reduce(const colearn::convops::BnReduceArgs& a) { ck(colearn::launch_bn_reduce(a, nullptr), "bn_reduce"); }
  static void bn_finalize(const colearn::convops::BnFinalizeArgs& a) { ck(colearn::launch_bn_finalize(a, nullptr), "bn_finalize"); }
  static void bn_reduce_finalize(const colearn::convops::BnFusedArgs& a) { ck(colearn::launch_bn_reduce_finalize(a, nullptr), "bn_reduce_finalize"); }
  static void bn_apply(const colearn::convops::BnApplyArgs& a) { ck(colearn::launch_bn_apply(a, nullptr), "bn_apply"); }
  static void bn_bwd(const colearn::convops::BnBwdArgs& a) { ck(colearn::launch_bn_bwd(a, nullptr), "bn_bwd"); }
  static void maxpool_fwd(const colearn::convops::PoolArgs& a) { ck(colearn::launch_maxpool_fwd(a, nullptr), "maxpool_fwd"); }
  static void maxpool_bwd(const colearn::convops::PoolArgs& a) { ck(colearn::launch_maxpool_bwd(a, nullptr), "maxpool_bwd"); }
  static void avgpool_fwd(const colearn::convops::AvgPoolArgs& a) { ck(colearn::launch_avgpool_fwd(a, nullptr), "avgpool_fwd"); }
  static void avgpool_bwd(const colearn::convops::AvgPoolArgs& a) { ck(colearn::launch_avgpool_bwd(a, nullptr), "avgpool_bwd"); }
  static void pack(const colearn::convops::PackArgs& a) { ck(colearn::launch_pack(a, nullptr), "pack"); }
  static void splitk_reduce(const colearn::convops::SplitKReduceArgs& a) { ck(colearn::launch_splitk_reduce(a, nullptr), "splitk_reduce"); }
};
}  // namespace

#include "conv_bindings.inc"

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "the CUDA kernels of mlp_persistent.cu / elementwise.cu / comm.cu / convnet.cu compiled for the CPU through a SIMT shim (tests only)";
  convbind::register_ops<ConvSimtExec>(m);
  m.def("gemm_tcgen05", &gemm_tcgen05);
  m.def("mlp_local_sgd", &mlp_local_sgd, py::arg("net_kind"), py::arg("theta_in"), py::arg("theta_outs"), py::arg("xs"), py::arg("ys"), py::arg("perms"),
        py::arg("batch_size"), py::arg("epochs"), py::arg("max_steps"), py::arg("loss"), py::arg("lr"), py::arg("variant"), py::arg("out_scales"),
        py::arg("delta_mode"), py::arg("flags"), py::arg("perm_seed") = 0, py::arg("perm_row0") = 0, py::arg("perm_scratch") = py::none());
  m.def("mlp_forward", &mlp_forward);
  m.def("mlp_local_sgd_generic", &mlp_local_sgd_generic);
  m.def("mlp_generic_plan", &mlp_generic_plan);
  m.def("make_client_desc", &make_client_desc);
  m.def("mlp_net_params", [](int64_t kind) { return (int64_t)colearn::mlp_net_num_params((int)kind); });
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
  m.def("transpose_bf16", &transpose_bf16);
  m.def("ring_matmul", &ring_matmul);
  m.def("star_round", &star_round);
  m.def("twoshot_fedavg", &twoshot_fedavg);
  m.def("twoshot_fedavg_deadline", &twoshot_fedavg_deadline);
  m.def("twoshot_resync", &twoshot_resync);
  m.def("produced_signal_pack", &produced_signal_pack);
  m.def("produced_mark", &produced_mark);
  m.def("reduce_push", &reduce_push);
}
