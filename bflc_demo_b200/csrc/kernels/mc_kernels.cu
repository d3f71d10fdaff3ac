// Round kernels of the multi-client engine (engine/multiclient.py): C <= 32 virtual clients on
// one GPU, all state in local HBM (no symmetric heap, no flags).  See mc_round.h for the round.
#include <cuda_bf16.h>

#include "bflc_kernels.h"
#include "consensus_math.hpp"
#include "launch.cuh"
#include "mc_round.h"
#include "sm100_ptx.cuh"

namespace bflc {

namespace {

constexpr int kMcThreads = 256;

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

// 32-bit mix (murmur3 finaliser) of (seed, epoch, client): the simulated arrival key
__device__ __forceinline__ uint32_t arrival_key(uint32_t seed, uint32_t epoch, uint32_t c) {
  uint32_t h = seed * 0x9E3779B1u ^ (epoch + 0x7F4A7C15u) * 0x85EBCA77u ^ (c + 1u) * 0xC2B2AE3Du;
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h;
}

// ------------------------------------------------------------------ plan
// One warp: lane c prepares client c; lane 0 builds the committee list and the candidate list.
// Arrival order (first-K admission): the reference admits the first NEEDED_UPDATE_COUNT uploads in
// chain order (C:239-244), i.e. whoever finishes first.  Clients sharing one GPU train one after
// another, so there is no physical race to finish: the order is simulated as a permutation of the
// trainers keyed by (seed, epoch, client), with every straggler after every other trainer.
__global__ void k_mc_plan(McArgs a) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  McState* st = a.st;
  McPlan* p = a.plan;
  const int n = static_cast<int>(st->n_clients);
  const int c = threadIdx.x;
  if (c < kMcMaxClients) {
    const bool tr = c < n && (st->role[c] & ROLE_TRAINER);
    p->is_trainer[c] = tr ? 1 : 0;
    p->barrier[c] = 0u;
    p->opt_step[c] = p->opt_total[c];
    if (tr) p->opt_total[c] += a.clients->steps[c];
    p->loss_sum[c] = 0.f;
    p->train_correct[c] = 0u;
    for (int t = 0; t < kMcMaxClients; ++t) p->correct[c][t] = 0u;
  }
  if (c != 0) return;
  p->epoch = st->epoch;
  p->fedavg_blocks_done = 0u;
  p->digest_acc = 0ull;
  int n_comm = 0, n_tr = 0;
  int order[kMcMaxClients];
  uint32_t key[kMcMaxClients];
  for (int r = 0; r < n; ++r) {
    if (st->role[r] & ROLE_COMM) p->comm[n_comm++] = r;
    if (!(st->role[r] & ROLE_TRAINER)) continue;
    const uint32_t k = (arrival_key(st->seed, st->epoch, static_cast<uint32_t>(r)) >> 1) |
                       (((st->straggler_mask >> r) & 1u) << 31);
    int j = n_tr++;
    while (j > 0 && (key[j - 1] > k)) { key[j] = key[j - 1]; order[j] = order[j - 1]; --j; }
    key[j] = k; order[j] = r;
  }
  const int n_adm = static_cast<int>(st->n_needed) < n_tr ? static_cast<int>(st->n_needed) : n_tr;
  uint32_t m = 0;
  for (int z = 0; z < n_adm; ++z) { p->cand[z] = order[z]; m |= 1u << order[z]; }
  p->n_cand = n_adm;
  p->n_comm = n_comm;
  p->admitted_mask = m;
}

// ------------------------------------------------------------------ byzantine
struct McByzIds { int id[kMcMaxClients]; };

__global__ void __launch_bounds__(kMcThreads) k_mc_byzantine(McArgs a, McByzIds ids, float scale) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int c = ids.id[blockIdx.y];
  if (!a.plan->is_trainer[c]) return;
  float4* w = reinterpret_cast<float4*>(a.clients->master[c]);
  uint2* s = reinterpret_cast<uint2*>(a.clients->shadow[c]);
  const float4* g = reinterpret_cast<const float4*>(a.global_master);
  const long long nv = a.n_params / 4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nv;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 v = w[i];
    const float4 g0 = g[i];
    v.x = g0.x - scale * (v.x - g0.x); v.y = g0.y - scale * (v.y - g0.y);
    v.z = g0.z - scale * (v.z - g0.z); v.w = g0.w - scale * (v.w - g0.w);
    w[i] = v;
    s[i] = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
  }
}

// ------------------------------------------------------------------ consensus
struct McShared {
  ConsensusIn<kMcMaxClients> in;
  ConsensusOut<kMcMaxClients> out;
};

// One block: scores = correct / n_val of the scoring member, run_consensus<32> weighted by every
// trainer's own sample count, block record, ledger page.
__global__ void __launch_bounds__(kMcThreads)
k_mc_consensus(McArgs a, int weight_by_score) {
  __shared__ McShared sh;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  McState* st = a.st;
  McPlan* p = a.plan;
  const int n = static_cast<int>(st->n_clients);
  const uint32_t epoch = st->epoch;
  const uint32_t adm = p->admitted_mask;
  ConsensusIn<kMcMaxClients>& in = sh.in;
  McBlockRecord* rec = a.ring + (epoch % static_cast<uint32_t>(a.ring_slots));
  const McClients* cl = a.clients;
  for (int i = threadIdx.x; i < kMcMaxClients * kMcMaxClients; i += blockDim.x) {
    const int r = i / kMcMaxClients, t = i % kMcMaxClients;
    const bool ok = r < n && t < n && (st->role[r] & ROLE_COMM) && (st->role[t] & ROLE_TRAINER) && ((adm >> t) & 1u);
    in.scored[r][t] = ok ? 1 : 0;
    in.score[r][t] = ok ? static_cast<float>(p->correct[r][t]) * (1.f / static_cast<float>(cl->n_val[r])) : 0.f;
    rec->score_rows[r][t] = in.score[r][t];
  }
  if (threadIdx.x < kMcMaxClients) {
    const int r = threadIdx.x;
    const bool tr = r < n && (st->role[r] & ROLE_TRAINER);
    in.role[r] = r < n ? st->role[r] : 0u;
    in.admitted[r] = (tr && ((adm >> r) & 1u)) ? 1 : 0;
    in.n_samples[r] = tr ? cl->n_samples[r] : 0u;
    in.avg_cost[r] = tr ? p->loss_sum[r] / static_cast<float>(cl->steps[r] * cl->batch) : 0.f;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    in.n_ranks = n;
    in.n_comm = static_cast<int>(st->n_comm);
    in.n_aggregate = static_cast<int>(st->n_aggregate);
    in.weight_by_score = weight_by_score;
    run_consensus<kMcMaxClients>(in, sh.out);
    int k = 0;
    for (int r = 0; r < n; ++r)   // ascending client id = the fixed FedAvg order
      if (sh.out.selected[r]) { p->sel[k] = r; p->sel_w[k] = sh.out.weight[r]; ++k; }
    p->n_sel = k;
  }
  __syncthreads();
  const ConsensusOut<kMcMaxClients>& out = sh.out;
  if (threadIdx.x < kMcMaxClients) {
    const int r = threadIdx.x;
    uint32_t m = 0;
    for (int t = 0; t < kMcMaxClients; ++t)
      if (in.scored[r][t]) m |= 1u << t;
    rec->role_before[r] = in.role[r];
    rec->role_after[r] = r < n ? out.role_after[r] : 0u;
    rec->scored_mask[r] = m;
    rec->median[r] = r < n ? out.median[r] : 0.f;
    rec->n_samples[r] = in.n_samples[r];
    rec->avg_cost[r] = in.avg_cost[r];
    rec->weight[r] = r < n ? out.weight[r] : 0.f;
  }
  // every lane of warp 0 reads the role words before thread 0 rewrites them
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t sel = 0;
    for (int r = 0; r < n; ++r)
      if (out.selected[r]) sel |= 1u << r;
    rec->epoch = epoch;
    rec->n_clients = static_cast<uint32_t>(n);
    rec->n_comm = st->n_comm;
    rec->n_aggregate = st->n_aggregate;
    rec->admitted_mask = adm;
    rec->selected_mask = sel;
    rec->global_loss = out.global_loss;
    rec->weight_by_score = static_cast<uint32_t>(weight_by_score);
    // model_digest and seq are written by k_mc_fedavg once the new model exists
    for (int r = 0; r < n; ++r) {
      st->role[r] = out.role_after[r];
      st->last_median[r] = out.median[r];
    }
    st->admitted_mask = adm;
    st->selected_mask = sel;
    st->global_loss = out.global_loss;
    st->blocks_appended = st->blocks_appended + 1;
    st->epoch = epoch + 1;
  }
}

// ------------------------------------------------------------------ FedAvg
__device__ __forceinline__ unsigned long long digest_term(float v, long long idx) {
  // the same order-independent digest as k_consensus (fed_kernels.cu)
  return static_cast<unsigned long long>(__float_as_uint(v)) *
         (static_cast<unsigned long long>(2 * idx + 1) * 0x9E3779B97F4A7C15ull);
}

// Server optimizer constants as the kernel uses them (c1, c2 rounded on the host).
struct McServerK {
  float lr, b1, b2, c1, c2, tau;
  float* m; float* v;
};

// One element of the server step (mc_round.h): d = avg - g, state (m, v) updated in place,
// returns the new global value.
template <int MODE>
__device__ __forceinline__ float server_step(const McServerK& k, float avg, float g, float& m, float& v) {
  const float d = avg - g;
  if (MODE == MC_SERVER_MOMENTUM) {
    m = fmaf(k.b1, m, d);
    return fmaf(k.lr, m, g);
  }
  m = fmaf(k.b1, m, k.c1 * d);
  const float d2 = d * d;
  if (MODE == MC_SERVER_ADAM) {
    v = fmaf(k.b2, v, k.c2 * d2);
  } else {   // yogi: sign(v - d2), sign(0) = 0
    const float sg = v > d2 ? 1.f : (v < d2 ? -1.f : 0.f);
    v = v - (k.c2 * d2) * sg;
  }
  return g + k.lr * m / (sqrtf(v) + k.tau);
}

// new_global = sum_k w_k * master_k over the selected clients in ascending id, one fp32 fma per
// client per element (no atomics: bit-reproducible).  MODE != none: the average then takes the
// server optimizer step from the current global model (mc_round.h).  The result goes to the
// global model and to every client's next-round work master / shadow.  The last block finishes
// the block record.  MODE is a template parameter so that plain FedAvg compiles as before.
template <int MODE>
__global__ void __launch_bounds__(kMcThreads) k_mc_fedavg(McArgs a, int n_clients, McServerK sk) {
  __shared__ const float4* src[kMcMaxClients];
  __shared__ float w[kMcMaxClients];
  __shared__ float4* dst_m[kMcMaxClients];
  __shared__ uint2* dst_s[kMcMaxClients];
  __shared__ bool last;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  McPlan* p = a.plan;
  const int n_sel = p->n_sel;
  if (threadIdx.x < kMcMaxClients) {
    const int k = threadIdx.x;
    src[k] = k < n_sel ? reinterpret_cast<const float4*>(a.clients->master[p->sel[k]]) : nullptr;
    w[k] = k < n_sel ? p->sel_w[k] : 0.f;
    dst_m[k] = k < n_clients ? reinterpret_cast<float4*>(a.clients->master[k]) : nullptr;
    dst_s[k] = k < n_clients ? reinterpret_cast<uint2*>(a.clients->shadow[k]) : nullptr;
  }
  __syncthreads();
  float4* g_f32 = reinterpret_cast<float4*>(a.global_master);
  uint2* g_b16 = reinterpret_cast<uint2*>(a.global_shadow);
  const long long nv = a.n_params / 4;
  unsigned long long dig = 0ull;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nv;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n_sel == 0) {
      acc = g_f32[i];   // nothing admitted: the global model is unchanged
    } else {
      int k = 0;
      for (; k + 4 <= n_sel; k += 4) {   // four loads in flight, accumulation order unchanged
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldcs(src[k + u] + i);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float wk = w[k + u];
          acc.x = fmaf(wk, v[u].x, acc.x); acc.y = fmaf(wk, v[u].y, acc.y);
          acc.z = fmaf(wk, v[u].z, acc.z); acc.w = fmaf(wk, v[u].w, acc.w);
        }
      }
      for (; k < n_sel; ++k) {
        const float4 v = __ldcs(src[k] + i);
        const float wk = w[k];
        acc.x = fmaf(wk, v.x, acc.x); acc.y = fmaf(wk, v.y, acc.y);
        acc.z = fmaf(wk, v.z, acc.z); acc.w = fmaf(wk, v.w, acc.w);
      }
      if (MODE != MC_SERVER_NONE) {
        const float4 g = g_f32[i];
        float4 m = reinterpret_cast<const float4*>(sk.m)[i];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (MODE != MC_SERVER_MOMENTUM) v = reinterpret_cast<const float4*>(sk.v)[i];
        acc.x = server_step<MODE>(sk, acc.x, g.x, m.x, v.x);
        acc.y = server_step<MODE>(sk, acc.y, g.y, m.y, v.y);
        acc.z = server_step<MODE>(sk, acc.z, g.z, m.z, v.z);
        acc.w = server_step<MODE>(sk, acc.w, g.w, m.w, v.w);
        reinterpret_cast<float4*>(sk.m)[i] = m;
        if (MODE != MC_SERVER_MOMENTUM) reinterpret_cast<float4*>(sk.v)[i] = v;
      }
    }
    dig += digest_term(acc.x, 4 * i) + digest_term(acc.y, 4 * i + 1) + digest_term(acc.z, 4 * i + 2) +
           digest_term(acc.w, 4 * i + 3);
    const uint2 b = make_uint2(pack_bf16x2(acc.x, acc.y), pack_bf16x2(acc.z, acc.w));
    g_f32[i] = acc;
    g_b16[i] = b;
    for (int c = 0; c < n_clients; ++c) {
      __stcs(dst_m[c] + i, acc);
      __stcs(dst_s[c] + i, b);
    }
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) dig += __shfl_xor_sync(0xffffffffu, dig, off);
  if ((threadIdx.x & 31) == 0 && dig) atomicAdd(&p->digest_acc, dig);
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(&p->fedavg_blocks_done, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last || threadIdx.x != 0) return;
  __threadfence();
  const unsigned long long digest = *reinterpret_cast<volatile unsigned long long*>(&p->digest_acc);
  const uint32_t epoch = p->epoch;
  McBlockRecord* rec = a.ring + (epoch % static_cast<uint32_t>(a.ring_slots));
  rec->model_digest = digest;
  a.st->model_digest = digest;
  __threadfence();
  rec->seq = epoch + 1;
}

__global__ void __launch_bounds__(kMcThreads)
k_mc_bcast(const McArgs a, const uint4* __restrict__ src, long long n16) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  uint4* dst = reinterpret_cast<uint4*>(a.clients->blob[blockIdx.y]);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n16;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    dst[i] = src[i];
}

int mc_grid(long long n_vec, int cap) {
  long long b = (n_vec + kMcThreads - 1) / kMcThreads;
  if (b > cap) b = cap;
  return static_cast<int>(b < 1 ? 1 : b);
}

}  // namespace

cudaError_t mc_plan_round(const McArgs& a, cudaStream_t s) {
  note_launch();
  return launch_pdl(k_mc_plan, dim3(1), dim3(32), 0, s, a);
}

cudaError_t mc_byzantine(const McArgs& a, const int* ids, int n_ids, float scale, cudaStream_t s) {
  if (n_ids <= 0) return cudaSuccess;
  if (n_ids > kMcMaxClients || a.n_params % 4) return cudaErrorInvalidValue;
  McByzIds b{};
  for (int i = 0; i < n_ids; ++i) b.id[i] = ids[i];
  note_launch();
  return launch_pdl(k_mc_byzantine, dim3(mc_grid(a.n_params / 4, 64), n_ids), dim3(kMcThreads), 0, s, a, b, scale);
}

cudaError_t mc_consensus(const McArgs& a, int weight_by_score, cudaStream_t s) {
  note_launch();
  return launch_pdl(k_mc_consensus, dim3(1), dim3(kMcThreads), 0, s, a, weight_by_score);
}

cudaError_t mc_fedavg(const McArgs& a, int n_clients, cudaStream_t s, const McServerOpt& so) {
  if (n_clients <= 0 || n_clients > kMcMaxClients || a.n_params % 4) return cudaErrorInvalidValue;
  if (so.mode < MC_SERVER_NONE || so.mode > MC_SERVER_YOGI) return cudaErrorInvalidValue;
  if (so.mode != MC_SERVER_NONE &&
      (!(so.lr > 0.f) || !(so.beta1 >= 0.f && so.beta1 < 1.f) || !(so.beta2 >= 0.f && so.beta2 < 1.f) ||
       !(so.tau > 0.f) || so.m == nullptr || (so.mode != MC_SERVER_MOMENTUM && so.v == nullptr)))
    return cudaErrorInvalidValue;
  McServerK sk{so.lr, so.beta1, so.beta2, static_cast<float>(1.0 - static_cast<double>(so.beta1)),
               static_cast<float>(1.0 - static_cast<double>(so.beta2)), so.tau, so.m, so.v};
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const dim3 grid(mc_grid(a.n_params / 4, 4 * sms));
  note_launch();
  switch (so.mode) {
    case MC_SERVER_MOMENTUM: return launch_pdl(k_mc_fedavg<MC_SERVER_MOMENTUM>, grid, dim3(kMcThreads), 0, s, a, n_clients, sk);
    case MC_SERVER_ADAM: return launch_pdl(k_mc_fedavg<MC_SERVER_ADAM>, grid, dim3(kMcThreads), 0, s, a, n_clients, sk);
    case MC_SERVER_YOGI: return launch_pdl(k_mc_fedavg<MC_SERVER_YOGI>, grid, dim3(kMcThreads), 0, s, a, n_clients, sk);
    default: return launch_pdl(k_mc_fedavg<MC_SERVER_NONE>, grid, dim3(kMcThreads), 0, s, a, n_clients, sk);
  }
}

cudaError_t mc_broadcast_blob(const McArgs& a, const uint8_t* src, long long bytes, int n_clients,
                              cudaStream_t s) {
  if (bytes % 16 || n_clients <= 0 || n_clients > kMcMaxClients) return cudaErrorInvalidValue;
  note_launch();
  return launch_pdl(k_mc_bcast, dim3(mc_grid(bytes / 16, 16), n_clients), dim3(kMcThreads), 0, s, a,
                    reinterpret_cast<const uint4*>(src), bytes / 16);
}

}  // namespace bflc
