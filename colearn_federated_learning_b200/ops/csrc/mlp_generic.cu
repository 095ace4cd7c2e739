// mlp_local_sgd_generic — the persistent local-SGD kernel for any small MLP, with the layer widths given at run time.
//
// Same contract as mlp_local_sgd_kernel / the v2 kernels (ClientDesc + SgdHyper, colearn_kernels.h): one launch runs the whole
// local fit of n_clients federated clients, each client waits for its broadcast flag, trains over its shard (epochs, max_steps,
// ragged last batch, perm table or in-kernel Feistel shuffle), writes out_scale * theta_k (or the scaled delta) into theta_out
// — possibly a peer GPU's slot — and raises signal_flag with st.release.sys.
//
// Network: L <= 8 layers, dims[0..L], ReLU on the hidden layers, sigmoid or no head, dims[L] <= 32 (loss and dz_L in one warp).
//
// One client = one thread-block cluster of C in {1, 2, 4, 8} CTAs, so that models up to ~8 x 50k parameters keep their weights
// in shared memory for the whole fit:
//   * Weights.  The output rows of every layer are split across the cluster in balanced contiguous ranges (a range may be
//     empty: a 1-wide head at C = 8 has 7 idle CTAs).  Each CTA keeps its rows + biases in fp32 shared memory with padded
//     row strides (stride == T mod 32, as in v1).  The thread that reads a weight in the forward pass is the thread that
//     updates it, so an update and the next sample's forward need no barrier between them; threads past the last
//     (row, lane) pair read nothing (the OWN_ONLY lesson of mlp_persistent.cu).
//   * Forward.  Each CTA computes its slice of a_{l+1} and pushes it into every peer's copy: every CTA then holds the whole
//     a_{l+1}, the head's a_L included, and computes the loss and dz_L redundantly with no further exchange.
//   * Backward.  dz_l = relu'(a_l) * W_l^T dz_{l+1} sums over rows that live in different CTAs: each CTA computes its partial
//     for every k, sends the partials of row range r to the CTA that owns range r in layer l-1, and that owner sums the C
//     partials in rank order (bitwise reproducible).  The rank-1 update of the CTA's own rows needs only local data.
//   * Exchange.  st.async.shared::cluster.mbarrier::complete_tx::bytes into the peer's buffer, completion observed on a local
//     mbarrier.  barrier.cluster runs only in the prologue and the epilogue: its arrive.release form (like fence.acq_rel.cluster)
//     compiles to a GPU-wide MEMBAR in front of UCGABAR_ARV, the st.async form to STAS + SYNCS.PHASECHK.TRANS64.TRYWAIT.
//   * Batch > 1 accumulates into a per-CTA fp32 gradient copy (sG, as v1) and applies it when the batch closes.
//   * Samples.  Every CTA gathers the full sample row (x, y) into its own ring of R rows (two stages of R/2), one stage
//     ahead with cp.async.
#include "colearn_kernels.h"

#include <math.h>
#include <string.h>

namespace colearn {
namespace {

constexpr int GNT = 256;              // threads per CTA
constexpr int GMAX_L = 8;             // layers
constexpr int GMAX_DOUT = 32;         // head width (one warp)
constexpr int GMAX_SMEM = 232448;     // 227 KB of dynamic shared memory per CTA on sm_100
constexpr int GMAX_RING = 128;        // sample ring rows (two stages of 64, the CHUNK of v1)
constexpr int GBAR_SLOTS = 16;        // mbarriers per parity: L forward + (L - 1) backward exchanges <= 15

// Launch-time description of the network and of the per-CTA shared-memory layout (offsets in floats after the mbarriers).
struct GenericNet {
  int L, sigmoid, C, ring;
  int dims[GMAX_L + 1];
  int T[GMAX_L];      // lanes per own row of layer l (forward + update: one mapping)
  int KP[GMAX_L];     // padded row stride of layer l
  int TB[GMAX_L];     // lanes per input k of layer l (backward partials)
  int rmax[GMAX_L];   // ceil(dims[l+1] / C): rows a CTA may own in layer l
  int woff[GMAX_L];   // layer l's rows (rmax x KP) then its rmax biases
  int aoff[GMAX_L + 1];   // a_l (l >= 1) inside one activation buffer
  int doff[GMAX_L];   // dz_{l+1} of the own rows of layer l
  int poff[GMAX_L];   // partials for the rows of layer l-1 (l >= 1): [C src ranks][rmax[l-1]]
  int sp, acts, dzs, parts, rowstride;
  int o_g, o_act, o_dz, o_part, o_misc, o_ring;   // section offsets (floats)
};

__host__ __device__ inline int gpow2_floor(int x) { int p = 1; while (p * 2 <= x) p *= 2; return p; }
__host__ __device__ inline int ggroup(int n_rows, int k_in) {
  int t = gpow2_floor(n_rows > 0 ? (GNT / n_rows > 0 ? GNT / n_rows : 1) : GNT);
  if (t > 32) t = 32;
  while (t > 1 && t > k_in) t /= 2;
  return t;
}
__host__ __device__ inline int gpad(int k, int t) { int s = k; while ((s % 32) != (t % 32)) ++s; return s; }
// first row of rank r in a layer of n rows (n <= 8 x 227 KB / 4 B rows, so n * r fits an int: no 64-bit division per step)
__host__ __device__ inline int row_lo(int n, int r, int C) { return n * r / C; }

// ---- cluster helpers: a PTX body for the GPU, a host_shim.h body for the CPU build ------------------------------------------
#ifdef COLEARN_HOST_SHIM
inline void g_st_release_sys(uint32_t* p, uint32_t v) { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
inline int cluster_rank() { return ::colearn_shim::cluster_rank(); }
inline void cluster_sync() { ::colearn_shim::cluster_sync(); }
inline void exchange_init(uint64_t* bar) { ::colearn_shim::mbar_init(bar); }
inline void push_to_peer(float* local_slot, float v, int peer, uint64_t* local_bar) {
  ::colearn_shim::push_to_peer(local_slot, v, peer, local_bar);
}
inline void wait_exchange(uint64_t* bar, uint32_t parity, uint32_t bytes, bool arrive) {
  ::colearn_shim::mbar_wait(bar, parity, bytes, arrive);
}
inline void copy_async4(float* dst, const float* src) { *dst = *src; }
inline void copy_async_wait() {}
#else
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void g_st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return (int)r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void exchange_init(uint64_t* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n\tfence.mbarrier_init.release.cluster;" ::"r"(smem_u32(bar)) : "memory");
}
// v -> the same offset in peer rank `peer`'s shared memory; completes 4 bytes of the transaction count of the peer's copy of
// local_bar
__device__ __forceinline__ void push_to_peer(float* local_slot, float v, int peer, uint64_t* local_bar) {
  uint32_t ra, rb;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(local_slot)), "r"(peer));
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rb) : "r"(smem_u32(local_bar)), "r"(peer));
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
               ::"r"(ra), "r"(__float_as_uint(v)), "r"(rb) : "memory");
}
// one thread (arrive) announces the bytes the peers send this phase; every caller then waits for the phase to complete
__device__ __forceinline__ void wait_exchange(uint64_t* bar, uint32_t parity, uint32_t bytes, bool arrive) {
  const uint32_t a = smem_u32(bar);
  if (arrive) asm volatile("mbarrier.arrive.expect_tx.release.cta.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
  uint32_t done = 0;
  while (!done) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(a), "r"(parity) : "memory");
  }
}
__device__ __forceinline__ void copy_async4(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void copy_async_wait() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_all;" ::: "memory");
}
#endif

// Loss + dz of the head for every output (warp 0; identical in every CTA of the cluster).  Semantics of loss_and_dz in
// mlp_persistent.cu with the head width at run time; dz lands in dz_head[j - lo] for the CTA's own head rows [lo, hi).
__device__ __forceinline__ float generic_loss(float* aL, int DO, bool sigmoid, const float* yrow, int loss, float inv_b,
                                              int lane, int lo, int hi, float* dz_own) {
  float value = 0.f;
  if (loss == LOSS_XENT) {
    const float z = lane < DO ? aL[lane] : -INFINITY;
    float m = z;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    const float e = lane < DO ? __expf(z - m) : 0.f;
    float s = e;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const int label = (int)yrow[0];
    const float zl = __shfl_sync(0xffffffffu, z, label & 31);
    value = (__logf(s) + m) - zl;
    if (lane >= lo && lane < hi) dz_own[lane - lo] = (e / s - (lane == label ? 1.f : 0.f)) * inv_b;
  } else {
    float contrib = 0.f;
    if (lane < DO) {
      const float z = aL[lane];
      const float y = yrow[lane];
      float out = z, dact = 1.f;
      if (sigmoid) { out = 1.f / (1.f + __expf(-z)); dact = out * (1.f - out); }
      const float inv_do = 1.f / (float)DO;
      float dz;
      if (loss == LOSS_BCE) {
        const float lp = fmaxf(__logf(out), -100.f), l1p = fmaxf(log1pf(-out), -100.f);
        contrib = -(y * lp + (1.f - y) * l1p) * inv_do;
        dz = (out - y) * inv_b * inv_do;
      } else {  // SSE / MSE
        const float d = out - y;
        contrib = d * d;
        dz = 2.f * d * dact * ((loss == LOSS_MSE) ? inv_b : 1.f);
      }
      if (lane >= lo && lane < hi) dz_own[lane - lo] = dz;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
    value = contrib;
  }
  return value;
}

__global__ void __launch_bounds__(GNT, 1)
mlp_local_sgd_generic_kernel(const ClientDesc* __restrict__ descs, SgdHyper hp, const GenericNet net) {
  COLEARN_DYN_SMEM(float, smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);               // [2 parities][GBAR_SLOTS]
  float* smem = smem_raw + 2 * GBAR_SLOTS * 2;
  const int C = net.C, L = net.L;
  const int rank = C > 1 ? cluster_rank() : 0;
  const ClientDesc d = descs[blockIdx.x / C];
  const int tid = threadIdx.x;
  const int B = hp.batch_size < 1 ? 1 : hp.batch_size;
  const bool accumulate = B > 1;
  const int DIN = net.dims[0], DOUT = net.dims[L];

  float* sP = smem;
  float* sG = smem + net.o_g;
  float* sAct = smem + net.o_act;     // 2 x acts (sample parity)
  float* sDz = smem + net.o_dz;
  float* sPart = smem + net.o_part;   // 2 x parts (sample parity)
  float* sMisc = smem + net.o_misc;   // [0] last loss, [1] loss sum
  float* sRing = smem + net.o_ring;   // ring rows x rowstride

  // (1) prologue: mbarriers, broadcast flag (rank 0 only), then the cluster barrier that also publishes the mbarrier inits
  if (C > 1 && tid == 0) {
    for (int i = 0; i < 2 * GBAR_SLOTS; ++i) exchange_init(bars + i);
  }
  if (d.wait_flag != nullptr && rank == 0 && tid == 0)
    spin_wait_ge(d.wait_flag, d.wait_value, 32, "mlp_local_sgd_generic: broadcast flag of this round");
  if (C > 1) cluster_sync();
  else __syncthreads();

  // (2) own rows of theta_in -> padded smem (L1 bypass: the arena may be peer-written)
  {
    int flat = 0;
    for (int l = 0; l < L; ++l) {
      const int K = net.dims[l], NO = net.dims[l + 1], KP = net.KP[l];
      const int lo = row_lo(NO, rank, C), nr = row_lo(NO, rank + 1, C) - lo;
      float* w = sP + net.woff[l];
      for (int i = tid; i < net.rmax[l] * KP; i += GNT) {
        const int n = i / KP, k = i - n * KP;
        w[i] = (n < nr && k < K) ? __ldcg(d.theta_in + flat + (size_t)(lo + n) * K + k) : 0.f;
      }
      for (int i = tid; i < net.rmax[l]; i += GNT) w[net.rmax[l] * KP + i] = i < nr ? __ldcg(d.theta_in + flat + NO * K + lo + i) : 0.f;
      flat += NO * K + NO;
    }
  }
  if (accumulate)
    for (int i = tid; i < net.sp; i += GNT) sG[i] = 0.f;
  if (tid < 2) sMisc[tid] = 0.f;

  // (3) step bookkeeping (as in mlp_local_sgd_kernel)
  const int n = d.n;
  const int ydim = d.y_dim;
  const int row = DIN + ydim;
  const int spe = (n + B - 1) / B;
  long long total_steps = (long long)hp.epochs * spe;
  if (hp.max_steps > 0 && hp.max_steps < total_steps) total_steps = hp.max_steps;
  long long Q;
  {
    const long long full_epochs = total_steps / spe;
    const long long rem_steps = total_steps - full_epochs * spe;
    long long rem_samples = rem_steps * B;
    if (rem_samples > n) rem_samples = n;
    Q = full_epochs * (long long)n + rem_samples;
  }
  const int S = net.ring / 2;                      // rows per stage
  const int n_stages = (int)((Q + S - 1) / S);
  const FeistelDomain fdom = feistel_domain((uint32_t)(n > 0 ? n : 1));
  auto gather = [&](int stage) {
    float* dst = sRing + (stage & 1) * S * net.rowstride;
    for (int e = tid; e < S * row; e += GNT) {
      const int i = e / row, c = e - i * row;
      const long long q = (long long)stage * S + i;
      if (q < Q) {
        const int ep = (int)(q / n);
        const int pos = (int)(q - (long long)ep * n);
        const int idx = d.perm ? __ldg(d.perm + (size_t)(ep % d.perm_rows) * n + pos)
                               : (d.perm_seed ? (int)feistel_index((uint32_t)pos, (uint32_t)n, fdom, d.perm_seed, d.perm_row0 + ep) : pos);
        copy_async4(dst + i * net.rowstride + c, (c < DIN) ? d.x + (size_t)idx * DIN + c : d.y + (size_t)idx * ydim + (c - DIN));
      }
    }
  };
  if (n_stages > 0) gather(0);
  copy_async_wait();
  __syncthreads();

  long long step = 0, it = 0;
  int pos_in_epoch = 0, in_batch = 0;
  int cur_batch = (n < B) ? n : B;
  float batch_loss = 0.f;   // rank 0, tid 0
  const float neg_lr = -hp.lr;

  for (int c = 0; c < n_stages; ++c) {
    if (c + 1 < n_stages) gather(c + 1);    // next stage flies during this stage's math
    const float* stage = sRing + (c & 1) * S * net.rowstride;
    const long long q0 = (long long)c * S;
    const int cnt = (int)((Q - q0) < S ? (Q - q0) : S);
    for (int i = 0; i < cnt; ++i, ++it) {
      const float* a0 = stage + i * net.rowstride;
      const float* yrow = a0 + DIN;
      const int par = (int)(it & 1);
      const uint32_t ph = (uint32_t)((it >> 1) & 1);
      float* acts = sAct + par * net.acts;
      float* parts = sPart + par * net.parts;
      uint64_t* bar = bars + par * GBAR_SLOTS;
      const float inv_b = 1.f / (float)cur_batch;

      // ---- forward: own rows of a_{l+1}, pushed into every peer's copy ----
      for (int l = 0; l < L; ++l) {
        const int K = net.dims[l], NO = net.dims[l + 1], T = net.T[l], KP = net.KP[l];
        const int lo = row_lo(NO, rank, C), nr = row_lo(NO, rank + 1, C) - lo;
        const float* a_in = l == 0 ? a0 : acts + net.aoff[l];
        float* a_out = acts + net.aoff[l + 1];
        const float* W = sP + net.woff[l];
        const float* bias = W + net.rmax[l] * KP;
        const bool relu = l + 1 < L;
        const int t = tid % T;
        for (int n0 = 0; n0 < nr; n0 += GNT / T) {
          const int r = n0 + tid / T;
          const bool valid = r < nr;
          float acc0 = 0.f, acc1 = 0.f;
          if (valid) {
            const float* w = W + r * KP;
            int k = t;
            for (; k + T < K; k += 2 * T) { acc0 = fmaf(w[k], a_in[k], acc0); acc1 = fmaf(w[k + T], a_in[k + T], acc1); }
            if (k < K) acc0 = fmaf(w[k], a_in[k], acc0);
          }
          float acc = acc0 + acc1;
          for (int o = T / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
          if (valid && t == 0) {
            const float z = acc + bias[r];
            const float a = relu ? fmaxf(z, 0.f) : z;
            a_out[lo + r] = a;
            for (int p = 1; p < C; ++p) {
              const int peer = rank + p < C ? rank + p : rank + p - C;
              push_to_peer(a_out + lo + r, a, peer, bar + l);
            }
          }
        }
        if (C > 1) wait_exchange(bar + l, ph, (uint32_t)(NO - nr) * 4u, tid == 0);
        __syncthreads();
      }

      // ---- loss + dz_L of the own head rows (every CTA holds the whole a_L) ----
      const int hlo = row_lo(DOUT, rank, C), hhi = row_lo(DOUT, rank + 1, C);
      if (tid < 32) {
        const float v = generic_loss(acts + net.aoff[L], DOUT, net.sigmoid != 0, yrow, hp.loss, inv_b, tid, hlo, hhi,
                                     sDz + net.doff[L - 1]);
        if (tid == 0) batch_loss += (hp.loss == LOSS_SSE) ? v : v * inv_b;
      }
      __syncthreads();

      // ---- backward ----
      for (int l = L - 1; l >= 0; --l) {
        const int K = net.dims[l], NO = net.dims[l + 1], KP = net.KP[l];
        const int lo = row_lo(NO, rank, C), nr = row_lo(NO, rank + 1, C) - lo;
        const float* a_in = l == 0 ? a0 : acts + net.aoff[l];
        const float* dz_out = sDz + net.doff[l];
        float* W = sP + net.woff[l];
        if (l > 0) {
          // partial[k] = sum over own rows n of W[n][k] dz_out[n], for every k; range r of layer l-1 goes to its owner
          const int TB = net.TB[l], t = tid % TB;
          float* my_part = parts + net.poff[l] + rank * net.rmax[l - 1];
          for (int k0 = 0; k0 < K; k0 += GNT / TB) {
            const int k = k0 + tid / TB;
            const bool valid = k < K;
            float acc0 = 0.f, acc1 = 0.f;
            if (valid) {
              int r = t;
              for (; r + TB < nr; r += 2 * TB) {
                acc0 = fmaf(W[r * KP + k], dz_out[r], acc0);
                acc1 = fmaf(W[(r + TB) * KP + k], dz_out[r + TB], acc1);
              }
              if (r < nr) acc0 = fmaf(W[r * KP + k], dz_out[r], acc0);
            }
            float acc = acc0 + acc1;
            for (int o = TB / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (valid && t == 0) {
              int owner = 0;
              while (row_lo(K, owner + 1, C) <= k) ++owner;
              float* slot = my_part + (k - row_lo(K, owner, C));
              if (owner == rank) *slot = acc;
              else push_to_peer(slot, acc, owner, bar + L + l - 1);
            }
          }
          __syncthreads();   // every read of W_l is done before its rows are updated
        }
        // rank-1 update of the own rows: same (row, lane) mapping as the forward pass
        {
          const int T = net.T[l], t = tid % T;
          float* tgt = accumulate ? sG + net.woff[l] : W;
          const float scale = accumulate ? 1.f : neg_lr;
          for (int n0 = 0; n0 < nr; n0 += GNT / T) {
            const int r = n0 + tid / T;
            if (r < nr) {
              const float g = scale * dz_out[r];
              float* w = tgt + r * KP;
              for (int k = t; k < K; k += T) w[k] = fmaf(g, a_in[k], w[k]);
              if (t == 0) tgt[net.rmax[l] * KP + r] += g;
            }
          }
        }
        if (l > 0) {
          // dz_l of my own rows of layer l-1: the C partials summed in rank order
          const int lo1 = row_lo(K, rank, C), nr1 = row_lo(K, rank + 1, C) - lo1;
          if (C > 1) wait_exchange(bar + L + l - 1, ph, (uint32_t)((C - 1) * nr1) * 4u, tid == 0);
          const float* pp = parts + net.poff[l];
          float* dz_in = sDz + net.doff[l - 1];
          for (int r = tid; r < nr1; r += GNT) {
            float s = 0.f;
            for (int src = 0; src < C; ++src) s += pp[src * net.rmax[l - 1] + r];
            dz_in[r] = a_in[lo1 + r] > 0.f ? s : 0.f;
          }
          __syncthreads();
        }
      }

      ++in_batch;
      ++pos_in_epoch;
      if (in_batch == cur_batch) {   // batch closes -> SGD step
        if (accumulate) {
          __syncthreads();
          for (int k = tid; k < net.sp; k += GNT) { sP[k] = fmaf(neg_lr, sG[k], sP[k]); sG[k] = 0.f; }
          __syncthreads();
        }
        if (tid == 0) { sMisc[0] = batch_loss; sMisc[1] += batch_loss; batch_loss = 0.f; }
        ++step;
        in_batch = 0;
        if (pos_in_epoch >= n) pos_in_epoch = 0;
        const int left = n - pos_in_epoch;
        cur_batch = left < B ? left : B;
      }
    }
    copy_async_wait();   // the next stage has landed
    __syncthreads();     // and everyone is done with this one before it is refilled
  }
  __syncthreads();

  // (4) epilogue: own rows of out_scale * theta_k (or the scaled delta) -> theta_out (possibly a peer GPU)
  {
    int flat = 0;
    for (int l = 0; l < L; ++l) {
      const int K = net.dims[l], NO = net.dims[l + 1], KP = net.KP[l];
      const int lo = row_lo(NO, rank, C), nr = row_lo(NO, rank + 1, C) - lo;
      const float* w = sP + net.woff[l];
      for (int i = tid; i < nr * K; i += GNT) {
        const int r = i / K, k = i - r * K;
        const size_t g = flat + (size_t)(lo + r) * K + k;
        float v = w[r * KP + k];
        if (d.delta_mode) v -= __ldcg(d.theta_in + g);
        d.theta_out[g] = d.out_scale * v;
      }
      for (int r = tid; r < nr; r += GNT) {
        const size_t g = flat + (size_t)NO * K + lo + r;
        float v = w[net.rmax[l] * KP + r];
        if (d.delta_mode) v -= __ldcg(d.theta_in + g);
        d.theta_out[g] = d.out_scale * v;
      }
      flat += NO * K + NO;
    }
  }
  if (rank == 0 && tid == 0 && d.loss_out != nullptr) {
    d.loss_out[0] = sMisc[0];
    d.loss_out[1] = step > 0 ? sMisc[1] / (float)step : 0.f;
  }
  // every CTA's slice is globally visible before the cluster barrier; only then does rank 0 raise the flag, so a coordinator
  // that sees the flag sees all C slices.  The barrier also keeps every CTA's shared memory alive until its peers are done.
  __threadfence_system();
  if (C > 1) cluster_sync();
  else __syncthreads();
  if (rank == 0 && tid == 0 && d.signal_flag != nullptr) g_st_release_sys(d.signal_flag, d.signal_value);
}

// Fills `net` for cluster size C; returns the bytes of dynamic shared memory with a ring of `ring` rows.
int generic_layout(const int* dims, int L, int sigmoid, int C, int batch_size, int ring, GenericNet* net) {
  GenericNet& g = *net;
  memset(&g, 0, sizeof(g));
  g.L = L; g.sigmoid = sigmoid; g.C = C; g.ring = ring;
  for (int i = 0; i <= L; ++i) g.dims[i] = dims[i];
  int off = 0, acts = 0, dzs = 0, parts = 0;
  for (int l = 0; l < L; ++l) {
    const int K = dims[l], NO = dims[l + 1];
    g.rmax[l] = (NO + C - 1) / C;
    g.T[l] = ggroup(g.rmax[l], K);
    g.KP[l] = gpad(K, g.T[l]);
    g.TB[l] = ggroup(K, g.rmax[l]);
    g.woff[l] = off;
    off += g.rmax[l] * g.KP[l] + g.rmax[l];
    g.aoff[l + 1] = acts;
    acts += NO;
    g.doff[l] = dzs;
    dzs += g.rmax[l];
    if (l > 0) { g.poff[l] = parts; parts += C * g.rmax[l - 1]; }
  }
  g.sp = off; g.acts = acts; g.dzs = dzs; g.parts = parts;
  g.rowstride = (dims[0] + dims[L] + 3) / 4 * 4;
  g.o_g = g.sp;
  g.o_act = g.o_g + (batch_size > 1 ? g.sp : 0);
  g.o_dz = g.o_act + 2 * acts;
  g.o_part = g.o_dz + dzs;
  g.o_misc = g.o_part + 2 * parts;
  g.o_ring = (g.o_misc + 4 + 3) / 4 * 4;
  return (2 * GBAR_SLOTS * 2 + g.o_ring + ring * g.rowstride) * (int)sizeof(float);
}

bool generic_cluster_legal(const int* dims, int L, int C) {
  if (L == 1) return C == 1;                    // no hidden layer: nothing to split but the head
  for (int l = 1; l < L; ++l)
    if (dims[l] < C) return false;              // every CTA owns hidden rows (the exchange protocol relies on it)
  return true;
}

}  // namespace

int mlp_generic_plan(const int* dims, int L, int batch_size, int cluster, int* smem_bytes) {
  if (L < 1 || L > GMAX_L || dims[L] > GMAX_DOUT) return -1;
  for (int i = 0; i <= L; ++i)
    if (dims[i] < 1) return -1;
  GenericNet net;
  for (int C = 1; C <= 8; C *= 2) {
    if (cluster > 0 && C != cluster) continue;
    if (!generic_cluster_legal(dims, L, C)) continue;
    const int bytes = generic_layout(dims, L, 0, C, batch_size, 2, &net);
    if (bytes <= GMAX_SMEM) {
      if (smem_bytes) *smem_bytes = bytes;
      return C;
    }
  }
  return -1;
}

cudaError_t launch_mlp_local_sgd_generic(const int* dims, int L, int sigmoid, const ClientDesc* descs, int n_clients, SgdHyper hp,
                                         int cluster, cudaStream_t stream) {
  int min_bytes = 0;
  const int C = mlp_generic_plan(dims, L, hp.batch_size, cluster, &min_bytes);
  if (C < 0 || n_clients < 1) return cudaErrorInvalidValue;
  GenericNet net;
  generic_layout(dims, L, sigmoid, C, hp.batch_size, 0, &net);
  const int ring_bytes = net.rowstride * (int)sizeof(float);
  int ring = (GMAX_SMEM - (min_bytes - 2 * ring_bytes)) / ring_bytes;
  ring = (ring > GMAX_RING ? GMAX_RING : ring) & ~1;
  const int bytes = generic_layout(dims, L, sigmoid, C, hp.batch_size, ring, &net);
#ifdef COLEARN_HOST_SHIM
  ::colearn_shim::launch_cluster(::colearn_shim::Dim3((unsigned)(n_clients * C)), (unsigned)C, ::colearn_shim::Dim3(GNT), (size_t)bytes,
                                 [&] { mlp_local_sgd_generic_kernel(descs, hp, net); });
  (void)stream;
  return cudaSuccess;
#else
  cudaError_t e = cudaFuncSetAttribute(mlp_local_sgd_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(n_clients * C));
  cfg.blockDim = dim3(GNT);
  cfg.dynamicSmemBytes = (size_t)bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int max_clusters = 0;
  e = cudaOccupancyMaxActiveClusters(&max_clusters, mlp_local_sgd_generic_kernel, &cfg);
  if (e != cudaSuccess) return e;
  if (max_clusters < 1) return cudaErrorInvalidConfiguration;
  e = cudaLaunchKernelEx(&cfg, mlp_local_sgd_generic_kernel, descs, hp, net);
  if (e != cudaSuccess) return e;
  return cudaGetLastError();
#endif
}

}  // namespace colearn
