// Shared declarations between the sm_100a kernels (.cu) and the torch bindings (bindings.cpp).
// The .cu files deliberately do NOT include torch headers: they compile in seconds and expose
// plain C++ launchers taking raw pointers + a cudaStream_t.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>

#include "conv_ops.cuh"

// The SIMT kernels that also run on the CPU for the test-suite (host_shim.h) declare their dynamic shared memory and
// launch through these two macros; for nvcc they expand to the plain CUDA forms.
#ifndef COLEARN_HOST_SHIM
#define COLEARN_NOINLINE __noinline__
#define COLEARN_DYN_SMEM(type, name) extern __shared__ __align__(16) type name[]
#define COLEARN_DYN_SMEM_UNALIGNED(type, name) extern __shared__ type name[]
#define COLEARN_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<grid, block, smem, stream>>>(__VA_ARGS__)
// Programmatic dependent launch (default; COLEARN_PDL=0 turns it off): a kernel variant compiled with the prologue
// first waits for the grids it depends on (full completion + memory visibility), then lets ITS dependents be scheduled, so
// the launch latency of kernel i+2 hides behind the execution of kernel i+1.  Both instructions are no-ops for a launch
// without the programmatic attribute.
#define COLEARN_PDL_PROLOGUE()                                          \
  do {                                                                  \
    asm volatile("griddepcontrol.wait;" ::: "memory");                  \
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");     \
  } while (0)
#else
#define COLEARN_PDL_PROLOGUE() ((void)0)
#endif

#include <cstdlib>
namespace colearn {
// Programmatic dependent launch is ON unless COLEARN_PDL=0 (measured: ResNet-18 step 1.069 -> 0.974 ms, bit-identical results)
inline bool pdl_enabled() {
  static const bool on = [] { const char* e = std::getenv("COLEARN_PDL"); return !(e != nullptr && e[0] == '0'); }();
  return on;
}
#if defined(__CUDACC__) && !defined(COLEARN_HOST_SHIM)
// one-argument kernels (the conv / BatchNorm / pooling family): plain launch, or the PDL variant with the attribute
template <class Arg>
inline cudaError_t launch_maybe_pdl(void (*plain)(const Arg), void (*pdl)(const Arg), dim3 grid, dim3 block, cudaStream_t s, const Arg& a) {
  if (!pdl_enabled()) {
    plain<<<grid, block, 0, s>>>(a);
    return cudaGetLastError();
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = 0;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, pdl, a);
}
#endif
}  // namespace colearn

namespace colearn {

// ---------------------------------------------------------------------------------------------
// Bounded cross-GPU flag wait.  Every "wait until a peer raised this flag to >= want" of the round protocol (broadcast flag
// in the worker kernels, arrive / chunk flags in the star and two-shot kernels, per-chunk ready flags in the GEMM's TMA
// producer) goes through spin_wait_ge: ld.acquire.sys + __nanosleep, and once the wait exceeds the limit — a peer that died or
// wedged never signals — it prints what it was waiting for and traps, so the launch FAILS (cudaErrorLaunchFailure on the
// host, the round raises) instead of hanging the box until some outer watchdog kills the job.  The limit is generous (120 s,
// COLEARN_SPIN_TIMEOUT_S at module load; 0 = wait forever): a coordinator legitimately waits for a whole local fit.
// One copy of the limit per translation unit (no relocatable device code): set_spin_limit_* in each .cu.
// ---------------------------------------------------------------------------------------------
#if defined(__CUDACC__) && !defined(COLEARN_HOST_SHIM)
static __device__ unsigned long long g_spin_limit_ns = 120ull * 1000000000ull;
__device__ __forceinline__ uint32_t spin_ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long spin_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
static __device__ __noinline__ void spin_wait_failed(const uint32_t* p, uint32_t want, uint32_t have, const char* what) {
  printf("colearn: %s: flag %p stayed at %u (< %u) beyond the spin limit: a peer never signalled; failing the launch "
         "(block %d, thread %d)\n", what, (const void*)p, have, want, (int)blockIdx.x, (int)threadIdx.x);
  __trap();
}
__device__ __forceinline__ void spin_wait_ge(const uint32_t* p, uint32_t want, unsigned sleep_ns, const char* what) {
  uint32_t v = spin_ld_acquire_sys(p);
  if (v >= want) return;
  const unsigned long long limit = g_spin_limit_ns, t0 = spin_globaltimer();
  unsigned it = 0;
  while ((v = spin_ld_acquire_sys(p)) < want) {
    __nanosleep(sleep_ns);
    if (limit != 0 && (++it & 1023u) == 0 && spin_globaltimer() - t0 > limit) spin_wait_failed(p, want, v, what);
  }
}
#define COLEARN_DEFINE_SPIN_LIMIT_SETTER(name)                                                         \
  cudaError_t name(unsigned long long ns) { return cudaMemcpyToSymbol(g_spin_limit_ns, &ns, sizeof(ns)); }
#else
inline void spin_wait_ge(const uint32_t* p, uint32_t want, unsigned, const char*) {
  while (__atomic_load_n(p, __ATOMIC_ACQUIRE) < want) {}
}
#define COLEARN_DEFINE_SPIN_LIMIT_SETTER(name) cudaError_t name(unsigned long long) { return cudaSuccess; }
#endif
cudaError_t set_spin_limit_comm(unsigned long long ns);
cudaError_t preload_comm_kernels();   // force the lazy loader for every kernel of comm.cu (see there)
cudaError_t set_spin_limit_mlp(unsigned long long ns);
cudaError_t set_spin_limit_gemm(unsigned long long ns);

// ---------------------------------------------------------------------------------------------
// Keyed bijection on [0, n) (SURVEY K14, shuffle=True of the reference's loaders): 4-round Feistel network over 2*hb bits
// with cycle walking.  Shared by feistel_perm_kernel (tabulates whole rows) and the persistent MLP kernel's gather
// (computes the index of the sample it is about to prefetch), so both produce the same order for the same (seed, row).
// ---------------------------------------------------------------------------------------------
#if defined(__CUDACC__) && !defined(COLEARN_HOST_SHIM)
#define COLEARN_HD __host__ __device__ __forceinline__
#else
#define COLEARN_HD inline
#endif
// The network is UNBALANCED when the index needs an odd number of bits (left half lb = bits / 2, right half rb = bits - lb;
// a round maps (l, r) -> (r, l ^ F(r)), so the two widths swap every round and are back after the 4th): the domain is
// exactly 2^bits < 2 n, i.e. no rejections at all for a power-of-two n and fewer than one per index otherwise.
struct FeistelDomain { int lb, rb; };
COLEARN_HD FeistelDomain feistel_domain(uint32_t n) {
  int bits = 1;
  while ((1u << bits) < n) ++bits;
  FeistelDomain d;
  d.lb = bits >> 1;
  d.rb = bits - d.lb;
  return d;
}
COLEARN_HD uint32_t feistel_mix32(uint32_t x, uint32_t k) {
  x ^= k; x *= 0x9E3779B1u; x ^= x >> 15; x *= 0x85EBCA77u; x ^= x >> 13; x *= 0xC2B2AE3Du; x ^= x >> 16;
  return x;
}
COLEARN_HD uint32_t feistel_index(uint32_t v, uint32_t n, FeistelDomain dom, uint64_t seed, int row) {
  const uint32_t k0 = (uint32_t)seed ^ (0x51ED270Bu * (uint32_t)(row + 1));
  const uint32_t k1 = (uint32_t)(seed >> 32) + 0x68E31DA4u * (uint32_t)(row + 1);
  const uint32_t ml = (1u << dom.lb) - 1u, mr = (1u << dom.rb) - 1u;
  do {
    uint32_t l = v >> dom.rb, r = v & mr;          // l: lb bits, r: rb bits
#pragma unroll
    for (int round = 0; round < 4; ++round) {
      // even rounds: l has lb bits; odd rounds: the halves have swapped widths
      const uint32_t f = feistel_mix32(r, (round & 1 ? k1 : k0) + 0x9E3779B9u * round) & ((round & 1) ? mr : ml);
      const uint32_t nl = r;
      r = l ^ f;
      l = nl;
    }
    v = (l << dom.rb) | r;
  } while (v >= n);
  return v;
}

// ---------------------------------------------------------------------------------------------
// Persistent whole-network local SGD (mlp_persistent.cu)
// ---------------------------------------------------------------------------------------------
enum LossKind : int { LOSS_BCE = 0, LOSS_SSE = 1, LOSS_XENT = 2, LOSS_MSE = 3 };
enum NetKind : int { NET_FFNN = 0, NET_MLP64 = 1, NET_TESTING_REMOTE = 2 };

// One descriptor per client (= one CTA).  A "client" is a federated worker: it starts from
// theta_in, runs its local SGD over its private shard and emits out_scale * theta_k (or the
// scaled delta) to theta_out — which may be a *peer GPU's* memory (model-gather leg, SURVEY K2).
struct ClientDesc {
  const float* x;          // [n, d_in] row-major features
  const float* y;          // [n, y_dim] targets (xent: class index stored as float, y_dim = 1)
  const int* perm;         // [perm_rows, n] sample order, or nullptr for identity
  const float* theta_in;   // flat arena to start from (state-dict order, unpadded)
  float* theta_out;        // where out_scale * theta_k (or delta) goes; may alias theta_in
  float* loss_out;         // [2]: {last batch loss, mean loss over all steps}; may be peer memory
  const uint32_t* wait_flag;  // if non-null: spin (ld.acquire.sys) until *wait_flag >= wait_value
  uint32_t* signal_flag;      // if non-null: st.release.sys signal_value after theta_out is written
  int n;
  int perm_rows;
  int y_dim;
  uint32_t wait_value;
  uint32_t signal_value;
  float out_scale;         // FedAvg weight w_k pre-applied by the producer (SURVEY K3)
  int delta_mode;          // 0: out = w*theta_k ; 1: out = w*(theta_k - theta_in)
  int perm_row0;           // in-kernel shuffle: epoch e of this fit uses permutation row perm_row0 + e
  uint64_t perm_seed;      // != 0 (and perm == nullptr): the kernel fills perm_scratch with feistel_index(pos, n, key(perm_seed,
                           // perm_row0 + epoch)) for every epoch of the fit before it waits for the broadcast — the bijection
                           // feistel_perm_kernel tabulates, without a separate launch
  int* perm_scratch;       // [epochs of this fit, n] ints owned by this client (device memory), used with perm_seed
};

struct SgdHyper {
  int batch_size;
  int epochs;
  int max_steps;   // <= 0: unlimited (PySyft max_nr_batches semantics)
  int loss;        // LossKind
  float lr;
  int variant;     // 0/2: register-resident weights, 256 threads; 3: 128 threads (default of ops/fused_mlp.py); 4: 64 threads; 5: 128 threads, blocked slices;
                   // 1: smem-resident weights (v1)
};

// Returns cudaError_t from the launch.  descs lives in device memory ([n_clients]).
cudaError_t launch_mlp_local_sgd(int net_kind, const ClientDesc* descs, int n_clients,
                                 SgdHyper hp, cudaStream_t stream);
int mlp_local_sgd_smem_bytes(int net_kind, int batch_size);
int mlp_net_num_params(int net_kind);

// Persistent local SGD for any small MLP (mlp_generic.cu): layer widths dims[0..L] at run time (L <= 8, dims[L] <= 32, ReLU
// hidden layers, sigmoid head if `sigmoid`), one client = one thread-block cluster of C in {1, 2, 4, 8} CTAs that splits the
// weights.  mlp_generic_plan returns the cluster size a launch uses — `cluster` if > 0 and it fits, else the smallest C whose
// per-CTA footprint fits 227 KB of shared memory — or -1 when none does; *smem_bytes (if non-null) gets its minimum footprint.
int mlp_generic_plan(const int* dims, int L, int batch_size, int cluster, int* smem_bytes);
cudaError_t launch_mlp_local_sgd_generic(const int* dims, int L, int sigmoid, const ClientDesc* descs, int n_clients, SgdHyper hp,
                                         int cluster, cudaStream_t stream);

// Forward-only batched inference/eval for the small nets: out[n, d_out] (post-activation).
cudaError_t launch_mlp_forward(int net_kind, const float* theta, const float* x, float* out,
                               int n, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// Elementwise / reduction kernels (elementwise.cu)
// ---------------------------------------------------------------------------------------------
cudaError_t launch_sgd_step(float* param, const float* grad, float lr, int64_t n, cudaStream_t s);
cudaError_t launch_scale_inplace(float* p, float scale, int64_t n, cudaStream_t s);   // p *= scale
cudaError_t launch_sgd_step_bf16grad(float* param, const void* grad_bf16, float lr, int64_t n,
                                     cudaStream_t s);
// theta <- theta + server_lr * (sum_k w[k] * slots[k*stride .. ] - theta)   (weights sum to 1)
cudaError_t launch_fedavg_apply(float* theta, const float* slots, int64_t slot_stride,
                                const float* weights, int k, float server_lr, int64_t n,
                                cudaStream_t s);
// out = sum_k w[k] * slots[k]
cudaError_t launch_fedavg_flat(float* out, const float* slots, int64_t slot_stride,
                               const float* weights, int k, int64_t n, cudaStream_t s);
// Fused loss forward+backward.  loss_out is a single float (mean or sum per LossKind).
cudaError_t launch_sigmoid_bce(const float* z, const float* y, float* dz, float* loss_out,
                               int64_t n, cudaStream_t s);
cudaError_t launch_sse(const float* out, const float* y, float* dz, float* loss_out, int64_t n,
                       float scale, cudaStream_t s);
cudaError_t launch_softmax_xent(const void* logits, int logits_is_bf16, const int64_t* labels,
                                float* dlogits, void* dlogits_bf16, float* loss_out, int rows,
                                int cols, cudaStream_t s);
// one-block loss head on padded operands: dl / dl_bf16 (either may be null) with their own row strides, db[cols] = column sums of
// dL/dlogits (may be null), *loss_out = mean loss; bit-reproducible (fixed summation order), cols <= 128
cudaError_t launch_softmax_xent_head(const void* logits, int logits_is_bf16, int ld_in, const int64_t* labels, float* dl, int ld_dl,
                                     void* dl_bf16, int ld_bf16, float* db, float* loss_out, int rows, int cols, cudaStream_t s);
// Eval: sum BCE + number of correct round(p) predictions (cf.py:233-253)
cudaError_t launch_eval_binary(const float* p, const float* y, float* loss_sum, int* correct,
                               int64_t n, cudaStream_t s);
cudaError_t launch_argmax_rows(const float* x, int64_t* out, int rows, int cols, cudaStream_t s);
// Column-wise min/max scaling to [0,1] (NetworkTrafficDataset preprocessing, ds.py:31-32)
cudaError_t launch_minmax_scale(const float* x, float* out, int rows, int cols, cudaStream_t s);
// Philox-keyed random permutation of [0, n): writes sort keys; caller argsorts? No — full device
// Fisher-Yates is serial; we use a keyed bijection (Feistel network over the next power of two,
// cycle-walking) so each index is computed independently in O(1).
cudaError_t launch_feistel_permutation(int* out, int n, int rows, uint64_t seed, cudaStream_t s);
cudaError_t launch_fp32_to_bf16(const float* in, void* out, int64_t n, cudaStream_t s);
cudaError_t launch_l2_flush(float* buf, int64_t n, cudaStream_t s);
// bias[n] -= lr * sum_r partials[r, n]   (also writes the summed gradient to grad_out if non-null)
cudaError_t launch_bias_sgd_from_partials(float* bias, const float* partials, int rows, int n, int64_t row_stride,
                                          float lr, float* grad_out, int n_bias, cudaStream_t s);
// SMPC ring ops (int64, arithmetic mod 2^64)
cudaError_t launch_fix_precision(const float* x, long long* out, int64_t n, double base, cudaStream_t s);
cudaError_t launch_float_precision(const long long* x, float* out, int64_t n, double inv_base, cudaStream_t s);
cudaError_t launch_ring_matmul(const long long* A, const long long* B, long long* C, int M, int K, int N, cudaStream_t s);
// out[C,R] = in[R,C]^T (bf16), 32x32 smem tiles
cudaError_t launch_transpose_bf16(const void* in, void* out, int rows, int cols, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
// Fused wgrad GEMM -> FedAvg reduce: per-chunk "produced" reports of the last local step (device side in produced.cuh)
// ---------------------------------------------------------------------------------------------
struct ProducedSignal {
  uint32_t* count;            // local [n_chunks] element counters, zero at rest (the completing add resets its chunk)
  uint32_t* flags[16];        // flags[o]: rank o's [world, n_chunks] table (peer pointers); I write row `rank`
  const uint32_t* epoch_ptr;  // published value = *epoch_ptr + epoch_add (device-resident so that CUDA graphs replay)
  int64_t n;                  // arena elements that get reported (every one exactly once per round)
  uint32_t epoch_add;
  int chunk_shift;            // chunk_elems = 1 << chunk_shift
  int world, rank, n_chunks;
};
// every element of arena range [lo, hi) is final (biases, padded edge layers, the tail): one thread per chunk
cudaError_t launch_produced_mark(const ProducedSignal* sig_dev, int chunk_shift, int64_t lo, int64_t hi, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
// Cross-GPU collectives over NVLink peer memory (comm.cu)
// ---------------------------------------------------------------------------------------------
// Coordinator-side "star" round step for small models:
//   wait until every selected worker k published w_k*theta_k into slots[k] (flag >= epoch),
//   theta <- theta + server_lr*(sum_k slots[k] - theta)  [weights already applied by producers],
//   then push theta into every selected peer's inbox and raise their bcast flag (= epoch+1).
// One kernel = FedAvg reduce + server apply + next-round broadcast (SURVEY K1+K2+K3+K4).
struct StarRoundArgs {
  float* theta;                 // coordinator's global model (local memory)
  const float* slots;           // [world, slot_stride] local slot buffer peers push into
  int64_t slot_stride;
  const uint32_t* arrive_flags; // [world] local flags raised by workers (value = round epoch)
  uint32_t arrive_epoch;
  float* peer_inbox[16];        // each rank's theta_in buffer (peer pointers; [rank]=local)
  uint32_t* peer_bcast_flag[16];
  uint32_t bcast_epoch;
  float* mc_inbox;              // multicast alias of the inbox (nullptr -> unicast P2P stores)
  uint32_t select_mask;         // bit k set = worker k participates this round
  int world;
  float server_lr;
  int64_t n;
  int do_reduce;                // 0: broadcast only (round 0)
  int do_bcast;                 // 0: reduce/apply only (last round)
  uint32_t* grid_counter;       // device scratch for the in-kernel grid barrier
  // failure detection: give up on a silent worker after timeout_ns (0 = wait forever).  weights[k]
  // are the FedAvg weights the producers pre-applied, so the sum can be renormalised over the
  // workers that actually arrived.  decision[0] = epoch flag, decision[1] = arrived mask (device).
  unsigned long long timeout_ns;
  float weights[16];
  uint32_t* decision;
};
cudaError_t launch_star_round(const StarRoundArgs& a, int n_blocks, cudaStream_t s);

// Bandwidth-optimal symmetric "two-shot" FedAvg for large models.  Chunk c of the arena is owned
// by rank (c % world): the owner pulls that chunk of theta_k from every selected peer's work
// arena (P2P ld), forms sum_k w_k*theta_k, applies the server update and writes the new chunk
// into every peer's fp32 work arena AND bf16 shadow arena (fp32->bf16 fused into the
// broadcast), then raises the chunk's ready flag on every peer.  The next round's first
// consumer GEMM polls those flags from its TMA producer warp (fused broadcast -> GEMM, SURVEY
// K1); non-GEMM consumers use launch_wait_flags.
struct TwoShotArgs {
  float* work[16];              // per-rank fp32 arenas (peer pointers; trained params in, theta out)
  void* shadow_bf16[16];        // per-rank bf16 shadows (peer pointers) or nullptr
  uint32_t* chunk_flags[16];    // per-rank [n_chunks] ready flags (peer pointers)
  const uint32_t* arrive_flags; // local [world]: rank k finished local training (value >= epoch)
  const float* weights;         // local device [world]: normalised FedAvg weights
  float* theta_prev;            // local previous global model (needed iff server_lr != 1) or null
  uint32_t epoch;
  uint32_t select_mask;
  float server_lr;
  int64_t n;                    // total elements (multiple of 4)
  int64_t chunk_elems;          // flag granularity (multiple of 4)
  int world;
  int rank;
  uint32_t* peer_arrive[16];    // if signal_arrive: my arrive slot on every rank (raised at kernel start)
  float* mc_work;               // NVLS multicast alias of the work arena: enables multimem.ld_reduce / multimem.st
  void* mc_shadow;              // multicast alias of the bf16 shadow arena (or nullptr)
  int signal_arrive;            // fold the "local training done" signal into this kernel
  int wait_all;                 // spin at the end until every chunk of MY arena carries `epoch`
  // overlapped mode (fused wgrad -> reduce): my [world, n_chunks] table of produced epochs.  The kernel runs NEXT TO the last
  // local step instead of after it and waits per chunk for table[k][c] >= epoch of every selected rank k, not for arrive_flags
  const uint32_t* produced;
  unsigned long long produced_timeout_ns;   // trap instead of hanging when a chunk never completes (0 = wait forever)
  // failure detection (deadline mode): rank 0's first CTA waits at most deadline_ns for the selected ranks' arrive flags and
  // publishes {epoch, arrived mask} into slot (epoch % 8) of EVERY rank's decision ring; all CTAs of all ranks then reduce over
  // exactly that set (weights renormalised), chunk ownership is dealt among the arrived ranks, and the result is also pushed into
  // every rank's second arena global_copy[k] — a rank that was late trains in place on a work arena that the owners overwrote
  // under it, so it restores its arena from global_copy before its next round (twoshot_resync_kernel)
  unsigned long long deadline_ns;
  uint32_t* decision[16];       // per-rank ring of 8 x {epoch, mask} words (peer pointers)
  float* global_copy[16];       // per-rank second fp32 arena (peer pointers) or nullptr
  const float* true_weights;    // local device [world]: the FedAvg weights to renormalise over the arrived set
};
cudaError_t launch_twoshot_fedavg(const TwoShotArgs& a, int n_blocks, cudaStream_t s);
// deadline mode, start of a round: if this rank was NOT in the arrived mask of `prev_epoch`, its work arena (and bf16 shadow) is
// restored from global_copy; a no-op otherwise
cudaError_t launch_twoshot_resync(const uint32_t* decision_ring, uint32_t prev_epoch, int rank, float* work, void* shadow_bf16,
                                  const float* global_copy, int64_t n, int n_blocks, cudaStream_t s);

// Many virtual clients per GPU: dst[j] = sum_c slots[c*stride + j] pushed to (peer) dst, mean losses to loss_dst,
// then flag <- value (release) by the last CTA.  counter: zero-initialised device scratch.
cudaError_t launch_reduce_push(const float* slots, int k, int64_t stride, int64_t n, float* dst, const float* losses,
                               float* loss_dst, uint32_t* flag, uint32_t value, uint32_t* counter, int n_blocks,
                               cudaStream_t s);

// Tiny helpers used by the host engine / tests.
cudaError_t launch_set_flag(uint32_t* flag, uint32_t value, cudaStream_t s);
cudaError_t launch_wait_flag(const uint32_t* flag, uint32_t value, cudaStream_t s);
cudaError_t launch_wait_flags(const uint32_t* flags, int count, uint32_t value, cudaStream_t s);
// same, but the value to wait for is read from device memory at kernel start (CUDA-graph friendly)
cudaError_t launch_wait_flags_dev(const uint32_t* flags, int count, const uint32_t* value_ptr, cudaStream_t s);
// raise flag_ptrs[k][0] = value on every rank k < world (release, system scope)
struct PeerFlags { uint32_t* ptr[16]; };
cudaError_t launch_signal_peers(const PeerFlags& flags, int world, uint32_t value, cudaStream_t s);
cudaError_t launch_p2p_copy(float* dst, const float* src, int64_t n, uint32_t* flag,
                            uint32_t flag_value, int n_blocks, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
// tcgen05 GEMM family (gemm_tcgen05.cu):  C[M,N] = A[M,K] * B[N,K]^T  (both operands K-major bf16)
// ---------------------------------------------------------------------------------------------
struct GemmEpilogue {
  const float* bias;        // [N] or nullptr
  int relu;                 // apply max(0, .)
  const void* relu_mask;    // bf16 [M,N]: multiply by (mask > 0) — dgrad through ReLU; or nullptr
  void* out_bf16;           // [M,N] bf16 or nullptr
  float* out_f32;           // [M,N] fp32 or nullptr
  void* out_bf16_t;         // [N,M] bf16 transposed copy or nullptr
  // fused SGD (wgrad epilogue): master[M,N] -= lr * acc ; shadow bf16 copies refreshed
  float* sgd_master;
  float sgd_lr;
  void* sgd_shadow;         // bf16 [M,N]
  void* sgd_shadow_t;       // bf16 [N,M]
  float* colsum;            // [M/32, N] per-32-row-block column sums of the epilogue output (bias gradient
                            // partials, reduced by launch_bias_sgd_from_partials); or nullptr
  // fused broadcast consumption: B is a view at element offset ready_elem_offset of a flat arena
  // whose chunk c (ready_chunk_elems elements each) is published by a peer GPU raising
  // ready_flags[c] >= ready_epoch.  Before loading B rows [n0, n0+BN) the TMA producer waits for
  // every chunk overlapping those rows (SURVEY K1).
  const uint32_t* ready_flags;
  uint32_t ready_epoch;
  const uint32_t* ready_epoch_ptr;  // if set, the epoch is read from device memory (CUDA-graph replays)
  int64_t ready_chunk_elems;
  int64_t ready_elem_offset;
  int tile_n;               // 0 = auto, 128 or 256 = force the N tile width
  int cluster;              // 3 = cta_group::2 (two SMs per 256x256 tile, UMMA M=256; needs M%256==0, N%256==0);
                            // 2 = pairs of CTAs + TMA multicast of the shared B tile (M%256==0, tile 256); else off
  // split-K (skinny problems: few output tiles, long reduction — the conv wgrads): the K range of every output tile
  // is cut into split_k slices that run as independent work units; slice s stores its raw fp32 accumulator to
  // split_out[s, M, N] and NO other epilogue op runs (launch_splitk_reduce sums the slices and applies the epilogue:
  // fused SGD or bf16 output).  split_k <= 1: off.  1-CTA kernel only; needs K/64 >= split_k.
  int split_k;
  float* split_out;         // fp32 [split_k, M, N]
  // debug overrides of the MN-major shared-memory descriptor fields (bytes; 0 = the kernel's layout: LBO 8192, SBO 1024)
  int mn_lbo, mn_sbo;
  // implicit-GEMM convolution: one operand is an NHWC activation read through a 4-D tensor map (conv_ops.cuh)
  convops::ConvAddr conv;
  const void* addend;       // bf16 [M,N] added to the accumulator before the bf16/fp32 outputs (residual gradient), or nullptr
  // fused wgrad -> FedAvg reduce (needs sgd_master): each epilogue warp reports the block of the master matrix it finished,
  // produced_elem_offset = arena element of master[0, 0] (see ProducedSignal)
  const ProducedSignal* produced;
  int64_t produced_elem_offset;
  int max_ctas;             // > 0: cap the persistent grid (leave SMs to a communication kernel running next to the GEMM)
  int pdl;                  // 1: launched with the programmatic-dependent-launch attribute; the kernel runs COLEARN_PDL_PROLOGUE
                            // after its own set-up (barrier init, TMEM allocation, tensor-map prefetch overlap the predecessor)
};
// A: [M,K] bf16 row-major, B: [N,K] bf16 row-major.  M%128==0, N%128==0, K%64==0.
cudaError_t launch_gemm_tcgen05(const void* A, const void* B, int M, int N, int K,
                                const GemmEpilogue& ep, cudaStream_t s);
// "MN-major" variants (operands whose reduction index runs over ROWS are read in place, no transposed copies):
//   a_mn = 1: C[M, N] = A^T * B  with A [K, a_cols], B [K, N]   (conv wgrad; a_cols <= M, missing columns = TMA zero fill)
//   a_mn = 0: C[M, N] = A * B    with A [M, K], B [b_rows >= K, N] (conv dgrad against the packed weights)
// M%128==0, N%128==0, K%64==0, a_cols%8==0.
cudaError_t launch_gemm_tcgen05_mn(const void* A, int a_mn, int a_cols, const void* B, int b_rows, int M, int N, int K,
                                   const GemmEpilogue& ep, cudaStream_t s);
// Implicit-GEMM convolution (stride 1, NHWC activation `act` [n_images, H, W, C] bf16, H*W in {1, 4, 16, 64}, C % 64 == 0).
//   ep.conv.mode = 1: C[M = n_images*H*W, N] = conv operand (A, K-major boxes) x `other` [N or rows, K] K-major weights
//   ep.conv.mode = 2: C[M, N] = other^T (A = dz [K = pixels, a_cols] MN-major) x conv operand (B, MN-major boxes)
cudaError_t launch_gemm_tcgen05_conv(const void* act, int n_images, int H, int W, const void* other, int other_rows, int other_cols,
                                     int M, int N, int K, const GemmEpilogue& ep, cudaStream_t s);
const char* gemm_tcgen05_last_error();

// ---------------------------------------------------------------------------------------------
// NHWC convolution / BatchNorm / pooling kernels (convnet.cu; bodies + argument structs in conv_ops.cuh)
// ---------------------------------------------------------------------------------------------
cudaError_t launch_im2col(const convops::Im2colArgs& a, cudaStream_t s);
cudaError_t launch_col2im(const convops::Col2imArgs& a, cudaStream_t s);
cudaError_t launch_bn_reduce(const convops::BnReduceArgs& a, cudaStream_t s);
cudaError_t launch_bn_finalize(const convops::BnFinalizeArgs& a, cudaStream_t s);
cudaError_t launch_bn_reduce_finalize(const convops::BnFusedArgs& a, cudaStream_t s);
cudaError_t launch_bn_apply(const convops::BnApplyArgs& a, cudaStream_t s);
cudaError_t launch_bn_bwd(const convops::BnBwdArgs& a, cudaStream_t s);
cudaError_t launch_maxpool_fwd(const convops::PoolArgs& a, cudaStream_t s);
cudaError_t launch_maxpool_bwd(const convops::PoolArgs& a, cudaStream_t s);
cudaError_t launch_avgpool_fwd(const convops::AvgPoolArgs& a, cudaStream_t s);
cudaError_t launch_avgpool_bwd(const convops::AvgPoolArgs& a, cudaStream_t s);
cudaError_t launch_pack(const convops::PackArgs& a, cudaStream_t s);
cudaError_t launch_splitk_reduce(const convops::SplitKReduceArgs& a, cudaStream_t s);

}  // namespace colearn
