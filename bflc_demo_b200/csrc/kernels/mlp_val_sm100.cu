// Committee validation of the 2-layer MLP: "QueryAllUpdates" + per-candidate scoring
// (reference: CommitteePrecompiled.cpp:299-311, python-sdk/main.py:196-217 -- one TF graph +
// Session per candidate there) as ONE launch.  One CTA per (128 validation rows, candidate z):
//
//     fwd1 (K = in_dim, N = 256, TMEM cols [0,256)) -> +b1, relu -> A operand of fwd2 written
//     straight into 128B-swizzled smem -> fwd2 (N = 64, TMEM cols [256,320)) -> +b2, argmax ==
//     label -> one atomicAdd per warp into correct[z]
//
// Candidate z's weights are addressed through device-resident tensor maps selected by the round
// plan (local staging slots filled by k_pull, or a trainer's upload buffer in peer HBM); inactive
// candidates exit.  Neither logits nor hidden activations ever reach global memory.
//
// Two precisions: bf16 (kind::f16) and block-scaled fp8 (kind::mxf8f6f4.block_scale): e4m3 x
// with its UE8M0 scale chunks from the input kernel, candidates as Mx8MlpLayout blobs (e4m3
// weights + scale chunks + fp32 biases, 227 KB instead of 435 KB per candidate over NVLink); the
// relu epilogue quantises h per 32-column group (one thread owns a row -> one K-group per TMEM
// load) and writes its scale bytes into an smem chunk that tcgen05.cp moves to TMEM.
#include <cuda_bf16.h>

#include <cstring>

#include "bflc_kernels.h"
#include "epi_common.cuh"
#include "launch.cuh"
#include "mc_round.h"
#include "sm100_ptx.cuh"

namespace bflc {

namespace {

using epi::kSfChunk;
using epi::st_sw128;
__device__ __forceinline__ uint32_t pack2(float a, float b) { return epi::pack_bf16x2(a, b); }

constexpr int kBM = 128;
constexpr int kEpiWarps = 8;        // two per TMEM lane quarter: each owns 4 of the 8 hidden-column chunks
constexpr int kThreads = 64 + kEpiWarps * 32;
constexpr int kCStages = 3;
constexpr int kCA = kBM * 128, kCB = 256 * 128, kCStage = kCA + kCB;   // x tile 16 KB + W1 tile 32 KB
constexpr int kOffH = 0;                        // h tile (fwd2's A) aliases stage memory once fwd1 retired
constexpr int kOffW2K = kCStages * kCStage;     // W2 K-major, loaded up front
constexpr int kChainH = 256;
constexpr int kBarBytes = 512;
constexpr int kBiasFloats = 320;
constexpr int kTmemCols = 512;
constexpr uint32_t kTmemSfa = 320, kTmemSfb = 328;   // fp8: SFA 4 columns, SFB up to 8 (N = 256)
// fp8 scale chunks in smem: per stage [x 512 | W1 2 x 512], then W2 [2 x 512], then h [2 x 512]
constexpr int kSfStage = 3 * kSfChunk;
constexpr int kSfW2 = kCStages * kSfStage, kSfH = kSfW2 + 2 * kSfChunk, kSfBytes = kSfH + 2 * kSfChunk;
constexpr int kOffSf = kOffW2K + 32768;
constexpr int kOffBar = kOffSf + kSfBytes;
constexpr int kValSmem = kOffBar + kBarBytes + kBiasFloats * 4 + 1024;
static_assert(kValSmem <= 227 * 1024, "shared memory budget");

struct ValArgs {
  int n_val, in_dim, n_classes;
  const CUtensorMap* maps;               // table indexed by dyn{1,2}->map_index[z]
  const GemmDynamic* dyn1; const GemmDynamic* dyn2;
  const int32_t* labels; unsigned int* correct;
  const int* pred;
  // fp8
  const uint8_t* x_sf; const uint8_t* const* cand_blob; Mx8MlpLayout ql;
  // fused gather of the candidate blobs (see MlpValArgs)
  const uint8_t* const* cand_src; unsigned int* pull_cnt; long long blob_bytes;
  unsigned long long* stamps;
};

__device__ __forceinline__ void val_stamp(unsigned long long* stamps, int slot) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  atomicMax(stamps + slot, t);
}

// Shared-memory carve-up of one validation CTA (both kernels below).
struct ValSmem {
  uint8_t* smem; uint8_t* sf_smem;
  uint64_t* full; uint64_t* empty; uint64_t* w2k; uint64_t* acc_h; uint64_t* h_ready; uint64_t* acc_l;
  uint32_t* tmem_slot; float* sb;
};

__device__ __forceinline__ ValSmem val_smem(uint8_t* smem_raw) {
  ValSmem s;
  s.smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  s.sf_smem = s.smem + kOffSf;
  s.full = reinterpret_cast<uint64_t*>(s.smem + kOffBar);
  s.empty = s.full + kCStages;
  s.w2k = s.empty + kCStages;
  s.acc_h = s.w2k + 1;
  s.h_ready = s.acc_h + 1;
  s.acc_l = s.h_ready + 1;
  s.tmem_slot = reinterpret_cast<uint32_t*>(s.acc_l + 1);
  s.sb = reinterpret_cast<float*>(s.smem + kOffBar + kBarBytes);
  return s;
}

// mbarrier init + TMEM allocation (before griddepcontrol.wait); returns the TMEM base
__device__ __forceinline__ uint32_t val_setup(const ValSmem& S, const CUtensorMap* prefetch) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    if (prefetch != nullptr) ptx::tma_prefetch_desc(prefetch);
    for (int s = 0; s < kCStages; ++s) {
      ptx::mbar_init(&S.full[s], 1);
      ptx::mbar_init(&S.empty[s], 1);
    }
    ptx::mbar_init(S.w2k, 1); ptx::mbar_init(S.acc_h, 1); ptx::mbar_init(S.acc_l, 1);
    ptx::mbar_init(S.h_ready, kEpiWarps * 32);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc(S.tmem_slot, kTmemCols);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  return *S.tmem_slot;
}

__device__ __forceinline__ void val_teardown(uint32_t tmem_base) {
  __syncthreads();
  if ((threadIdx.x >> 5) == 1) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// What one CTA validates: 128 rows of x (map tx, row m0) against one candidate.
struct ChainJob {
  const CUtensorMap* tx; const CUtensorMap* m1; const CUtensorMap* m2;
  const float* b1; const float* b2;   // bf16 candidate biases (fp8: inside the blob)
  const uint8_t* blob;                // fp8 candidate (Mx8MlpLayout)
  const uint8_t* x_sf;                // fp8: scale chunks of x
  const int32_t* labels; unsigned int* correct;
  const uint32_t* wait_flag; uint32_t wait_value;   // optional: wait until *wait_flag >= wait_value
};

// The chain fwd1 -> relu -> fwd2 -> argmax == label of one (128 rows, candidate) tile, warp
// specialised: warp 0 TMA producer, warp 1 MMA issuer, warps 2..9 epilogue.
template <bool FP8>
__device__ __forceinline__ void val_chain(const ValSmem& S, uint32_t tmem_base, const ChainJob& j, int m0,
                                          int n_val, int in_dim, int n_classes, const Mx8MlpLayout& ql) {
  uint8_t* smem = S.smem;
  uint8_t* sf_smem = S.sf_smem;
  uint64_t* full = S.full;
  uint64_t* empty = S.empty;
  uint64_t* w2k = S.w2k;
  uint64_t* acc_h = S.acc_h;
  uint64_t* h_ready = S.h_ready;
  uint64_t* acc_l = S.acc_l;
  float* sb = S.sb;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kb_d = FP8 ? ql.kb1 : (in_dim + 63) / 64;
  const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
  const uint32_t base_lo = ptx::smem_u32(smem) >> 4;

  if (warp == 0) {
    if (j.wait_flag != nullptr) {   // candidate z's trainer has published its upload
      if (lane == 0) ptx::wait_flag_ge(j.wait_flag, j.wait_value);
      __syncwarp();
    }
    const CUtensorMap* m1 = j.m1;
    const CUtensorMap* m2 = j.m2;
    if (ptx::elect_one()) {
      if (FP8) {
        ptx::mbar_expect_tx(w2k, 2 * 8192 + 2 * kSfChunk);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb) {
          ptx::tma_load_3d(smem + kOffW2K + kb * 8192, m2, w2k, kb * 128, 0, 0);
          epi::bulk_g2s(sf_smem + kSfW2 + kb * kSfChunk, j.blob + ql.w2sf + kb * kSfChunk, kSfChunk, w2k);
        }
      } else {
        ptx::mbar_expect_tx(w2k, 32768);
#pragma unroll
        for (int kb = 0; kb < 4; ++kb) ptx::tma_load_3d(smem + kOffW2K + kb * 8192, m2, w2k, kb * 64, 0, 0);
      }
    }
    __syncwarp();
    for (int i = 0; i < kb_d; ++i) {
      const int s = i % kCStages;
      const uint32_t ph = (i / kCStages) & 1;
      ptx::mbar_wait(&empty[s], ph ^ 1);
      if (ptx::elect_one()) {
        uint8_t* sa = smem + s * kCStage;
        if (FP8) {
          uint8_t* sf = sf_smem + s * kSfStage;
          ptx::mbar_expect_tx(&full[s], kCStage + kSfStage);
          ptx::tma_load_3d(sa, j.tx, &full[s], i * 128, m0, 0);
          ptx::tma_load_3d(sa + kCA, m1, &full[s], i * 128, 0, 0);
          epi::bulk_g2s(sf, j.x_sf + (static_cast<long long>(m0 >> 7) * kb_d + i) * kSfChunk, kSfChunk, &full[s]);
          // W1: 256 rows = two 128-row blocks of scale chunks
          epi::bulk_g2s(sf + kSfChunk, j.blob + ql.w1sf + static_cast<long long>(i) * kSfChunk, kSfChunk, &full[s]);
          epi::bulk_g2s(sf + 2 * kSfChunk, j.blob + ql.w1sf + (static_cast<long long>(kb_d) + i) * kSfChunk, kSfChunk,
                        &full[s]);
        } else {
          ptx::mbar_expect_tx(&full[s], kCStage);
          ptx::tma_load_3d(sa, j.tx, &full[s], i * 64, m0, 0);
          ptx::tma_load_3d(sa + kCA, m1, &full[s], i * 64, 0, 0);
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    const uint32_t tsfa = tmem_base + kTmemSfa, tsfb = tmem_base + kTmemSfb;
    const uint32_t id1 = FP8 ? epi::make_idesc_mx8(kBM, 256) : ptx::make_idesc(1u, 0u, 0u, kBM, 256);
    for (int i = 0; i < kb_d; ++i) {
      const int s = i % kCStages;
      const uint32_t ph = (i / kCStages) & 1;
      ptx::mbar_wait(&full[s], ph);
      ptx::tc_fence_after_sync();
      if (ptx::elect_one()) {
        const uint32_t lo_a = (base_lo + static_cast<uint32_t>(s) * (kCStage >> 4)) | (1u << 16);
        const uint32_t lo_b = lo_a + (kCA >> 4);
        if (FP8) {
          const uint32_t sfs = ptx::smem_u32(sf_smem + s * kSfStage);
          epi::utccp_32x128b_warpx4(tsfa, epi::sf_desc(sfs));
          epi::utccp_32x128b_warpx4(tsfb, epi::sf_desc(sfs + kSfChunk));
          epi::utccp_32x128b_warpx4(tsfb + 4, epi::sf_desc(sfs + 2 * kSfChunk));
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k)
            epi::umma_mx8(tmem_base, (static_cast<uint64_t>(hi) << 32) | (lo_a + k * 2u),
                          (static_cast<uint64_t>(hi) << 32) | (lo_b + k * 2u), epi::idesc_mx8_k(id1, k),
                          (i > 0 || k > 0) ? 1u : 0u, tsfa, tsfb);
        } else {
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k)
            ptx::umma_f16(tmem_base, (static_cast<uint64_t>(hi) << 32) | (lo_a + k * 2u),
                          (static_cast<uint64_t>(hi) << 32) | (lo_b + k * 2u), id1, (i > 0 || k > 0) ? 1u : 0u);
        }
        ptx::umma_commit(&empty[s]);
      }
      __syncwarp();
    }
    if (ptx::elect_one()) ptx::umma_commit(acc_h);
    __syncwarp();
    ptx::mbar_wait(w2k, 0);
    ptx::mbar_wait(h_ready, 0);
    ptx::tc_fence_after_sync();
    if (ptx::elect_one()) {
      const uint32_t lo_a0 = (base_lo + (kOffH >> 4)) | (1u << 16);
      const uint32_t lo_b0 = (base_lo + (kOffW2K >> 4)) | (1u << 16);
      if (FP8) {
        const uint32_t id2 = epi::make_idesc_mx8(kBM, 64);
        const uint32_t sfs = ptx::smem_u32(sf_smem);
#pragma unroll
        for (uint32_t kb = 0; kb < 2; ++kb) {
          epi::utccp_32x128b_warpx4(tsfa, epi::sf_desc(sfs + kSfH + kb * kSfChunk));
          epi::utccp_32x128b_warpx4(tsfb, epi::sf_desc(sfs + kSfW2 + kb * kSfChunk));
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k)
            epi::umma_mx8(tmem_base + 256, (static_cast<uint64_t>(hi) << 32) | (lo_a0 + kb * (16384u >> 4) + k * 2u),
                          (static_cast<uint64_t>(hi) << 32) | (lo_b0 + kb * (8192u >> 4) + k * 2u),
                          epi::idesc_mx8_k(id2, k), (kb > 0 || k > 0) ? 1u : 0u, tsfa, tsfb);
        }
      } else {
        const uint32_t id2 = ptx::make_idesc(1u, 0u, 0u, kBM, 64);
#pragma unroll
        for (uint32_t kb = 0; kb < 4; ++kb)
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k)
            ptx::umma_f16(tmem_base + 256, (static_cast<uint64_t>(hi) << 32) | (lo_a0 + kb * (16384u >> 4) + k * 2u),
                          (static_cast<uint64_t>(hi) << 32) | (lo_b0 + kb * (8192u >> 4) + k * 2u), id2,
                          (kb > 0 || k > 0) ? 1u : 0u);
      }
      ptx::umma_commit(acc_l);
    }
    __syncwarp();
  } else {
    // warps 2..9: q = TMEM lane quarter, half = which four 32-column chunks of h this warp converts
    const int q = warp & 3, half = (warp - 2) >> 2, rl = q * 32 + lane, row = m0 + rl;
    const bool row_ok = row < n_val;
    const int C = n_classes;
    {
      const int et = threadIdx.x - 64;
      const float* b1 = FP8 ? reinterpret_cast<const float*>(j.blob + ql.b1) : j.b1;
      const float* b2 = FP8 ? reinterpret_cast<const float*>(j.blob + ql.b2) : j.b2;
      sb[et] = b1 != nullptr ? b1[et] : 0.f;            // kEpiWarps * 32 == kChainH
      if (et < 64) sb[kChainH + et] = (b2 != nullptr && et < C) ? b2[et] : 0.f;
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    ptx::mbar_wait(acc_h, 0);
    ptx::tc_fence_after_sync();
#pragma unroll 2
    for (int c = half * 4; c < half * 4 + 4; ++c) {
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c * 32, r);
      ptx::tmem_ld_wait();
      if (FP8) {
        // 32 hidden units of this row = one K-group of fwd2: quantise in registers, bytes into
        // K-block c / 4 of the swizzled A tile, the scale byte into that K-block's chunk
        float hv[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) hv[k] = fmaxf(__uint_as_float(r[k]) + sb[c * 32 + k], 0.f);
        uint32_t w[8];
        const int e = epi::mx8_quant32(hv, w);
        uint8_t* tile = smem + kOffH + (c >> 2) * 16384;
        st_sw128(tile, rl, (c & 3) * 2, make_uint4(w[0], w[1], w[2], w[3]));
        st_sw128(tile, rl, (c & 3) * 2 + 1, make_uint4(w[4], w[5], w[6], w[7]));
        sf_smem[kSfH + (c >> 2) * kSfChunk + epi::mx8_sf_off(rl, c & 3)] = static_cast<uint8_t>(e);
      } else {
        uint32_t pk[16];
#pragma unroll
        for (int k = 0; k < 32; k += 2)
          pk[k >> 1] = pack2(fmaxf(__uint_as_float(r[k]) + sb[c * 32 + k], 0.f),
                             fmaxf(__uint_as_float(r[k + 1]) + sb[c * 32 + k + 1], 0.f));
        uint8_t* tile = smem + kOffH + (c >> 1) * 16384;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj)
          st_sw128(tile, rl, (c & 1) * 4 + jj, make_uint4(pk[4 * jj], pk[4 * jj + 1], pk[4 * jj + 2], pk[4 * jj + 3]));
      }
    }
    ptx::fence_proxy_async_smem();
    ptx::tc_fence_before_sync();
    ptx::mbar_arrive(h_ready);
    if (half == 0) {     // the 64 logits of a row: one thread
    ptx::mbar_wait(acc_l, 0);
    ptx::tc_fence_after_sync();
    const int32_t label = row_ok ? j.labels[row] : -1;
    float vmax = -INFINITY;
    int amax = -1;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + 256 + c * 32, r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const int n = c * 32 + k;
        const float x = __uint_as_float(r[k]) + sb[kChainH + n];
        if (n < C && x > vmax) { vmax = x; amax = n; }
      }
    }
    const unsigned cnt = __popc(__ballot_sync(0xffffffffu, row_ok && amax == label));
    if (lane == 0 && cnt) atomicAdd(j.correct, cnt);
    }
    ptx::tc_fence_before_sync();
  }
}

template <bool FP8>
__global__ void __launch_bounds__(kThreads, 1)
mlp_val_kernel(const __grid_constant__ CUtensorMap tmX, const ValArgs v) {
  extern __shared__ uint8_t smem_raw[];
  const ValSmem S = val_smem(smem_raw);
  ptx::pdl_launch_dependents();
  const int warp = threadIdx.x >> 5;
  const int z = blockIdx.y, m0 = blockIdx.x * kBM;
  const uint32_t tmem_base = val_setup(S, &tmX);
  ptx::pdl_wait();
  const bool inactive = (v.pred != nullptr && *v.pred == 0) || z >= v.dyn1->active_batches;
  if (inactive) {
    if (warp == 1) ptx::tmem_dealloc(tmem_base, kTmemCols);
    return;
  }
  const uint8_t* blob = FP8 ? v.cand_blob[z] : nullptr;

  if (FP8 && v.cand_src != nullptr) {
    // ---- fused gather (reference: QueryAllUpdates, CommitteePrecompiled.cpp:299-311).  The
    // gridDim.x CTAs that validate candidate z each copy 1/gridDim.x of z's blob out of the
    // trainer's HBM with 16-byte P2P loads as soon as its FLAG_TRAINED is up, publish their share
    // (device-scope fence + counter), wait for the others' shares and only then start the TMA /
    // bulk loads of the local copy.  Every candidate crosses NVLink once per committee rank, and
    // there is no pull kernel in front of the validation.
    if (threadIdx.x == 0 && v.stamps != nullptr && blockIdx.x == 0 && z == 0) val_stamp(v.stamps, STAMP_PULL_BEGIN);
    if (threadIdx.x == 0 && v.dyn1->wait_flag[z] != nullptr)
      ptx::wait_flag_ge(v.dyn1->wait_flag[z], v.dyn1->wait_value);
    __syncthreads();
    const float4* src = reinterpret_cast<const float4*>(v.cand_src[z]);
    float4* dst = reinterpret_cast<float4*>(const_cast<uint8_t*>(blob));
    const long long n16 = v.blob_bytes >> 4;
    const long long per = (n16 + gridDim.x - 1) / gridDim.x;
    const long long lo = per * blockIdx.x, hi = lo + per < n16 ? lo + per : n16;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) dst[i] = ptx::ld_peer_f4(src + i);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
      atomicAdd(v.pull_cnt + z, 1u);
      unsigned long long spins = 0;
      unsigned int have;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(have) : "l"(v.pull_cnt + z) : "memory");
        if (have >= gridDim.x) break;
        __nanosleep(20);
      } while (++spins < (1ull << 26));
      if (have < gridDim.x) __trap();   // a sibling CTA never arrived: co-residency assumption broken
      if (v.stamps != nullptr && blockIdx.x == 0) val_stamp(v.stamps, STAMP_PULL_END);
    }
    __syncthreads();
    ptx::fence_proxy_async_all();   // the others' generic-proxy stores -> this CTA's TMA / bulk loads
  }

  ChainJob j;
  j.tx = &tmX;
  j.m1 = v.maps + v.dyn1->map_index[z];
  j.m2 = v.maps + v.dyn2->map_index[z];
  j.b1 = FP8 ? nullptr : v.dyn1->bias[z];
  j.b2 = FP8 ? nullptr : v.dyn2->bias[z];
  j.blob = blob; j.x_sf = v.x_sf;
  j.labels = v.labels; j.correct = v.correct + z;
  j.wait_flag = v.dyn1->wait_flag[z]; j.wait_value = v.dyn1->wait_value;
  val_chain<FP8>(S, tmem_base, j, m0, v.n_val, v.in_dim, v.n_classes, v.ql);
  val_teardown(tmem_base);
}

// Multi-client committee validation (engine/multiclient.py): CTA (m-tile, candidate slot z,
// committee slot k).  Who is candidate z and member k comes from the round plan; the candidate is
// read in place from its client's buffers (bf16 work shadow + fp32 biases, or the fp8 blob), the
// rows are the first n_val[member] rows of the member's own shard.  Members may hold different
// row counts: the grid spans the largest one, tiles past a member's n_val exit.
struct McVal {
  int in_dim, n_classes;
  const McPlan* plan; unsigned int* correct;
  const CUtensorMap* x_maps; const CUtensorMap* w_maps;
  const McClients* clients; long long b1_off, b2_off;
  Mx8MlpLayout ql;
};

template <bool FP8>
__global__ void __launch_bounds__(kThreads, 1)
mc_val_kernel(const McVal v) {
  extern __shared__ uint8_t smem_raw[];
  const ValSmem S = val_smem(smem_raw);
  ptx::pdl_launch_dependents();
  const int warp = threadIdx.x >> 5;
  const int z = blockIdx.y, k = blockIdx.z, m0 = blockIdx.x * kBM;
  const uint32_t tmem_base = val_setup(S, nullptr);
  ptx::pdl_wait();
  const int member = k < v.plan->n_comm ? v.plan->comm[k] : 0;
  const int n_val = v.clients->n_val[member];
  if (z >= v.plan->n_cand || k >= v.plan->n_comm || m0 >= n_val) {
    if (warp == 1) ptx::tmem_dealloc(tmem_base, kTmemCols);
    return;
  }
  const int cand = v.plan->cand[z];
  ChainJob j;
  j.tx = v.x_maps + member;
  j.m1 = v.w_maps + cand;
  j.m2 = v.w_maps + kMcMaxClients + cand;
  j.b1 = FP8 ? nullptr : v.clients->master[cand] + v.b1_off;
  j.b2 = FP8 ? nullptr : v.clients->master[cand] + v.b2_off;
  j.blob = FP8 ? v.clients->blob[cand] : nullptr;
  j.x_sf = FP8 ? v.clients->x_sf[member] : nullptr;
  j.labels = v.clients->labels[member];
  j.correct = v.correct + member * kMcMaxClients + cand;
  j.wait_flag = nullptr; j.wait_value = 0u;
  val_chain<FP8>(S, tmem_base, j, m0, n_val, v.in_dim, v.n_classes, v.ql);
  val_teardown(tmem_base);
}

}  // namespace

cudaError_t mlp_val_sm100(const MlpValArgs& r, cudaStream_t stream) {
  bind_context_once();
  if (r.hidden != kChainH || r.n_classes > 64 || r.in_dim % 8 || r.n_val <= 0 || r.max_cand <= 0)
    return cudaErrorInvalidValue;
  if (r.fp8 && (r.x_sf == nullptr || r.cand_blob == nullptr || r.in_dim % 16)) return cudaErrorInvalidValue;
  CUtensorMap tx;
  GemmOperand op{r.x, r.ldx, 0, false};
  cudaError_t e = gemm_make_operand_map(&tx, op, r.fp8 ? DType::FP8_E4M3 : DType::BF16, r.n_val, r.in_dim, 1, kBM);
  if (e != cudaSuccess) return e;
  ValArgs v{};
  v.n_val = r.n_val; v.in_dim = r.in_dim; v.n_classes = r.n_classes;
  v.maps = r.maps; v.dyn1 = r.dyn1; v.dyn2 = r.dyn2;
  v.labels = r.labels; v.correct = r.correct;
  v.pred = r.pred ? r.pred : current_predicate();
  v.x_sf = r.x_sf; v.cand_blob = r.cand_blob; v.ql = mx8_mlp_layout(r.in_dim, r.hidden);
  if (r.cand_src != nullptr) {
    // every CTA of a candidate must be able to run while its siblings spin on the counter
    if (!r.fp8 || r.pull_cnt == nullptr || r.blob_bytes <= 0 || r.blob_bytes % 16 != 0 ||
        (r.n_val + kBM - 1) / kBM > 128)
      return cudaErrorInvalidValue;
    v.cand_src = r.cand_src; v.pull_cnt = r.pull_cnt; v.blob_bytes = r.blob_bytes;
    v.stamps = r.stamps;
  }
  static bool configured[2] = {false, false};
  if (!configured[r.fp8 ? 1 : 0]) {
    e = r.fp8 ? cudaFuncSetAttribute(mlp_val_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kValSmem)
              : cudaFuncSetAttribute(mlp_val_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kValSmem);
    if (e != cudaSuccess) return e;
    configured[r.fp8 ? 1 : 0] = true;
  }
  note_launch();
  const dim3 grid((r.n_val + kBM - 1) / kBM, r.max_cand);
  if (r.fp8) return launch_pdl(mlp_val_kernel<true>, grid, dim3(kThreads), kValSmem, stream, tx, v);
  return launch_pdl(mlp_val_kernel<false>, grid, dim3(kThreads), kValSmem, stream, tx, v);
}

cudaError_t mc_val_sm100(const McValArgs& r, cudaStream_t stream) {
  bind_context_once();
  if (r.hidden != kChainH || r.n_classes > 64 || r.in_dim % 8 || r.max_n_val <= 0 || r.max_cand <= 0 ||
      r.max_cand > kMcMaxClients || r.max_comm <= 0 || r.max_comm > kMcMaxClients || r.plan == nullptr ||
      r.correct == nullptr || r.x_maps == nullptr || r.w_maps == nullptr || r.clients == nullptr)
    return cudaErrorInvalidValue;
  if (r.fp8 && r.in_dim % 16) return cudaErrorInvalidValue;
  McVal v{};
  v.in_dim = r.in_dim; v.n_classes = r.n_classes;
  v.plan = r.plan; v.correct = r.correct; v.x_maps = r.x_maps; v.w_maps = r.w_maps;
  v.clients = r.clients; v.b1_off = r.b1_off; v.b2_off = r.b2_off;
  v.ql = mx8_mlp_layout(r.in_dim, r.hidden);
  static bool configured[2] = {false, false};
  cudaError_t e;
  if (!configured[r.fp8 ? 1 : 0]) {
    e = r.fp8 ? cudaFuncSetAttribute(mc_val_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kValSmem)
              : cudaFuncSetAttribute(mc_val_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kValSmem);
    if (e != cudaSuccess) return e;
    configured[r.fp8 ? 1 : 0] = true;
  }
  note_launch();
  const dim3 grid((r.max_n_val + kBM - 1) / kBM, r.max_cand, r.max_comm);
  if (r.fp8) return launch_pdl(mc_val_kernel<true>, grid, dim3(kThreads), kValSmem, stream, v);
  return launch_pdl(mc_val_kernel<false>, grid, dim3(kThreads), kValSmem, stream, v);
}

}  // namespace bflc
