// One persistent kernel for a trainer's whole local-training pass of the 2-layer MLP:
// every mini-batch step (forward, softmax-xent, both weight gradients, the hidden gradient
// and the optimizer) runs inside ONE launch; phases are separated by a device-wide barrier
// instead of kernel boundaries -- and the LAST step's optimizer epilogue is also the
// UploadLocalUpdate of the protocol (reference: CommitteePrecompiled.cpp:215-258): it writes the
// peer-readable upload buffers and CTA 0 releases FLAG_TRAINED on every peer.
//
//   per step:  P1  h  = relu(x W1^T + b1)                       K = 784
//              X   per 128 batch rows, 4 CTAs: fwd2 -> softmax-xent -> dh = (dlogits W2) relu'(h)
//              B   dW1 = dh^T x  ||  dW2 = dlogits^T h  as 64 x 64 tiles (UMMA M = 64) on 57 CTAs,
//                  optimizer (SGD / Adam) applied to the fp32 master straight from the
//                  accumulator tile (E_OPT) + compute-copy refresh
//
// Precision.  bf16 mode: every GEMM is tcgen05.mma.kind::f16 on bf16 shadows.  fp8 mode
// (BASELINE.json config #2, "block-scaled fp8"): fwd1 and fwd2 are
// tcgen05.mma.kind::mxf8f6f4.block_scale -- x arrives as e4m3 + UE8M0 scales from the input
// kernel (elementwise_optim.cu), the E_OPT epilogue re-quantises every updated weight tile (one
// thread per 32-element K-group of the staged tile: amax, one scale byte, 32 e4m3 bytes) and
// the fwd1 epilogue quantises h; scale chunks reach TMEM through tcgen05.cp.  The hidden/weight
// gradients stay bf16, masters and Adam moments fp32.  Measured limits of the block-scaled
// UMMA on sm_100a: M = 64 per CTA is an illegal instruction, and a scale-factor TMEM address
// at an odd column (32-wide tiles) faults with `misaligned address` -- so fwd1 is 128 x 64.
//
// Warp roles (384 threads = three warpgroups): warpgroup 0 = warp 0 TMA producer, warp 1 TMEM
// owner + single-thread MMA issuer (warps 2-3 idle); warpgroups 1-2 = eight epilogue warps.  A
// warp may only touch the TMEM lane quarter (warp % 4); two warps share a quarter and split a
// tile's 64 columns -- "half" h owns columns [32h, 32h+32).  Measured before the split (4
// epilogue warps = one warp per SM sub-partition, every dependent instruction exposes its full
// latency): epilogues were 9.8 of a 23 us step.  Registers follow the work: `setmaxnreg` shrinks
// warpgroup 0 to 56 registers per thread and grows the epilogue warpgroups to 224.
//
// Each GEMM tile is the same tcgen05 / TMEM / TMA pipeline as gemm_sm100.cu (7-stage
// 128B-swizzled ring, staged coalesced epilogue); the smem ring, its mbarriers and the TMEM
// allocation persist across tiles, phases and steps.
//
// Why: at this problem size every stand-alone GEMM launch costs 6-12 us of which only a
// fraction is math (launch, prologue, first-TMA latency, drain) -- six launches per step,
// 48 per round.  Inside one kernel the fixed costs are paid once and a phase boundary is a
// ~2 us grid barrier.  (Reference step: python-sdk/main.py:141-148, three sess.run calls;
// Adam: the commented alternative at python-sdk/main.py:126.)
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "bflc_kernels.h"
#include "epi_common.cuh"
#include "fed_admit.cuh"
#include "launch.cuh"
#include "sm100_ptx.cuh"

namespace bflc {

namespace {

using epi::kStgLd;
using epi::kSfChunk;
using epi::stage_put;
using epi::stage_get;
using epi::col_sum32;
using epi::st_sw128;
__device__ __forceinline__ uint32_t pack2(float a, float b) { return epi::pack_bf16x2(a, b); }

constexpr int kBM = 128, kBN = 64, kStages = 7;
constexpr int kABytes = kBM * 128, kBBytes = kBN * 128, kStageBytes = kABytes + kBBytes;
constexpr int kTileBytes = kStages * kStageBytes;
constexpr int kSfStage = 2 * kSfChunk;              // per ring stage: [SFA chunk | SFB chunk]
constexpr int kSfBytes = kStages * kSfStage;        // fp8 only; the chain uses the first 4 chunks
constexpr int kBarBytes = 512;
constexpr int kEpiWarps = 8;       // two per TMEM lane quarter: warp (q, half) owns 32 of a tile's 64 columns
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kStgAll = kEpiWarps * 32 * kStgLd * 4;
constexpr int kBiasFloats = 320;   // chain: b1[256] | b2[64]; tile jobs use the first kBN
constexpr int kXchFloats = 4 * 2 * 128;   // chain E2: per-row partials exchanged by the two halves
constexpr int kSmemTotal = kTileBytes + kSfBytes + kBarBytes + kStgAll + (kBiasFloats + kXchFloats) * 4 + 1024;
static_assert(kSmemTotal <= 227 * 1024, "shared memory budget");
constexpr int kEpiT0 = 128;        // first epilogue thread (warpgroup 0 = producer / MMA / 2 idle warps)
constexpr int kThreads = kEpiT0 + kEpiThreads;
constexpr int kRegsLow = 56, kRegsHigh = 224;   // (168 - 56) * 128 == (224 - 168) * 256
constexpr int kGrid = 32;

// ---- fused chain (hidden == 256): the ring memory re-cut as
//   [0, 64 KB) h tile = fwd2's A operand | [64, 96 KB) W2 K-major (fwd2's B) | [96, 104 KB) this
//   CTA's 64-column slice of W2 MN-major (dh's B) | [104, 120 KB) dlogits (dh's A).
//   fp8: h is 2 x 16 KB of e4m3 at [0, 32 KB), W2 K-major 2 x 8 KB at [64, 80 KB).
constexpr int kOffH = 0;
constexpr int kOffW2K = 64 * 1024;
constexpr int kOffW2MN = 96 * 1024;
constexpr int kOffDL = 104 * 1024;
static_assert(kOffDL + 16384 <= kTileBytes, "chain smem layout");
constexpr int kChainH = 256;
constexpr int kDefaultPlan = 3;    // phase plan when neither the caller nor BFLC_MLP_CHAIN picks one (0 | 3)
constexpr int kTmemCols = 512;     // chain: dh accumulator [0,64) + logits [256,320) + scales
constexpr uint32_t kTmemSfa = 320, kTmemSfb = 328;   // fp8: scale-factor columns (4 + up to 4)

enum EpiMode : int { E_BIAS_RELU_BF16 = 0, E_XENT = 1, E_F32 = 2, E_MASK_COLSUM_BF16 = 3,
                     E_OPT = 4 };  // E_OPT: the tile IS the gradient -> optimizer applied in the epilogue

struct Maps {  // TMA descriptors, SWIZZLE_128B
  CUtensorMap x_k, w1_k, h_k, w2_k, dl_mn, h_mn, dl_k, w2_mn, dh_mn, x_mn;   // bf16
  CUtensorMap xq_k, w1q_k, hq_k, w2q_k;   // fp8 (e4m3 as u8): x 128-row box, W1 64, h 128, W2 64
};

struct Args {
  int B, steps, in_dim, hidden, n_classes, ncp;  // ncp = dlogits row stride (padded classes)
  int chain;                     // 0: P1|P2|P3 as separate phases   3: P1 | fwd2->xent->dh chained
  int epiopt;                    // optimizer applied in the weight-gradient epilogues (no P5)
  unsigned long long* dbg;       // optional %globaltimer stamps [steps][32] written by CTA 0
  const unsigned int* x_ready;   // optional input pipeline: step s may read x once x_ready[s] >= *round_seq + 1
  const unsigned int* round_seq;
  long long n_params;
  const int* pred;               // whole kernel is a no-op when *pred == 0 (non-trainer rank)
  unsigned int* barrier;         // device-wide phase barrier counter (zeroed before launch)
  // parameters / optimizer state
  float* master; const float* b1; const float* b2;
  float* grad; float* gw1; float* gb1; float* gw2; float* gb2;
  __nv_bfloat16* shadow;
  float* adam_m; float* adam_v;
  int adam; float lr, beta1, beta2, eps; const int* step_base;
  // activations
  __nv_bfloat16* h; __nv_bfloat16* dlogits; __nv_bfloat16* dh;
  const int32_t* labels;
  float* loss_sum; unsigned int* correct;
  // fp8 forward
  const uint8_t* x_sf; uint8_t* work_q; uint8_t* h_q; uint8_t* h_sf;
  Mx8MlpLayout ql;
  int bm_w;                      // weight-gradient tile height: 64 (default) or 128
  // fused upload
  int has_fed; FedArgs f; long long upq_off[2];
  int n_samples, n_loss_terms, byz_mode; float byz_scale; int straggle_us;
  // FedProx (PROX instantiations only): g' = mu (w - anchor) + g before the optimizer
  const float* prox_anchor; float prox_mu;
};

struct Job {  // one output tile (bm rows x 64 columns)
  const CUtensorMap* ta; const CUtensorMap* tb;
  int a_mn, b_mn;
  int a_c0, a_c1, b_c0, b_c1;   // TMA coordinates of K-block 0 (c0 = innermost)
  int n_kb;
  int m0, n0, M, N;             // output tile origin / logical extent
  int bm;                       // tile height: 128, or 64 (UMMA M = 64, kind::f16 only)
  int mode;
  long long ldd;
  void* d;                      // output
  const float* bias;            // E_BIAS_RELU_BF16 / E_XENT
  const __nv_bfloat16* aux;     // E_MASK_COLSUM_BF16: relu mask source, same shape as d
  float* colsum;
  const int32_t* labels;        // E_XENT (already offset to this step's rows)
  float grad_scale;
  float bc1, bc2;               // E_OPT + Adam: bias corrections of this step
  // ---- fp8 operands (K-major e4m3, K-blocks of 128 elements)
  int fp8;
  const uint8_t* sfa; const uint8_t* sfb;   // scale chunk of K-block 0 of this tile's row block
  uint32_t sfb_col;                         // column of the tile's first W row inside the 4-column chunk
  // ---- E_OPT in fp8 mode: where the re-quantised tile goes (byte offsets inside a model blob)
  int q_off, qsf_off, ldq, q_nkb;
  int last;                     // last step of the round: E_OPT also publishes the upload
  unsigned long long* dbg;      // this step's stamp slots (CTA 0): [dbg_slot] accumulator ready, [+1] epilogue done
  int dbg_slot;
};

struct Pipe {  // persistent pipeline state of one role
  uint32_t it;    // K-blocks processed so far (ring slot / parity)
  uint32_t tile;  // tiles processed so far (accumulator barrier parity)
};
struct ChainBars {
  uint64_t* h;                       // h tile (+ scale chunks) landed
  uint64_t* w2k; uint64_t* w2mn;     // W2 operand tiles landed
  uint64_t* acc_l; uint64_t* dl_ready; uint64_t* acc_dh;
};

template <typename T>
__device__ __forceinline__ T* heap_at(char* base, long long off) {
  return reinterpret_cast<T*>(base + off);
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// Where the last step's optimizer epilogue publishes (resolved from the ledger page: the upload
// buffers are double-buffered by epoch parity).
struct UploadDst {
  float* master;            // fp32 upload (FedAvg operand)
  __nv_bfloat16* shadow;    // bf16 upload (bf16-mode validation operand); null in fp8 mode
  uint8_t* blob;            // fp8 mode: Mx8MlpLayout blob the committee validates
  const float* global;      // Byzantine fault injection: upload global - s * (w - global)
  float byz_scale;
};
template <bool FP8>
__device__ __forceinline__ UploadDst upload_dst(const Args& a) {
  char* me = a.f.peers.base[a.f.rank];
  const RoundState* st = heap_at<const RoundState>(me, a.f.lay.state_off);
  const uint32_t par = st->epoch & 1u;
  UploadDst u;
  u.master = heap_at<float>(me, a.f.lay.upload_master_off[par]);
  u.shadow = FP8 ? nullptr : heap_at<__nv_bfloat16>(me, a.f.lay.upload_shadow_off[par]);
  u.blob = FP8 ? heap_at<uint8_t>(me, a.upq_off[par]) : nullptr;
  u.global = a.byz_mode == 1 ? heap_at<const float>(me, a.f.lay.global_off) : nullptr;
  u.byz_scale = a.byz_scale;
  return u;
}

// ---------------------------------------------------------------- producer / MMA / epilogue
template <bool FP8>
__device__ __forceinline__ void produce_tile(const Job& j, uint8_t* smem, uint8_t* sf_smem,
                                             uint64_t* full_bar, uint64_t* empty_bar, Pipe& pp) {
  const uint32_t a_bytes = static_cast<uint32_t>(j.bm) * 128u;
  for (int i = 0; i < j.n_kb; ++i, ++pp.it) {
    const int s = pp.it % kStages;
    const uint32_t ph = (pp.it / kStages) & 1;
    ptx::mbar_wait(&empty_bar[s], ph ^ 1);
    uint8_t* sa = smem + s * kStageBytes;
    uint8_t* sb = sa + kABytes;
    if (ptx::elect_one()) {
      if (FP8 && j.fp8) {
        // e4m3 tiles (K-block = 128 bytes) + the two 512-byte scale chunks of this K-block
        ptx::mbar_expect_tx(&full_bar[s], static_cast<uint32_t>(kABytes + kBBytes + kSfStage));
        ptx::tma_load_3d(sa, j.ta, &full_bar[s], j.a_c0 + i * 128, j.a_c1, 0);
        ptx::tma_load_3d(sb, j.tb, &full_bar[s], j.b_c0 + i * 128, j.b_c1, 0);
        epi::bulk_g2s(sf_smem + s * kSfStage, j.sfa + static_cast<long long>(i) * kSfChunk, kSfChunk, &full_bar[s]);
        epi::bulk_g2s(sf_smem + s * kSfStage + kSfChunk, j.sfb + static_cast<long long>(i) * kSfChunk, kSfChunk,
                      &full_bar[s]);
      } else {
        ptx::mbar_expect_tx(&full_bar[s], a_bytes + kBBytes);
        if (!j.a_mn) {
          ptx::tma_load_3d(sa, j.ta, &full_bar[s], j.a_c0 + i * 64, j.a_c1, 0);
        } else {
          // MN-major A: one 64-element (128-byte) chunk of M per box
          ptx::tma_load_3d(sa, j.ta, &full_bar[s], j.a_c0, j.a_c1 + i * 64, 0);
          if (j.bm == kBM) ptx::tma_load_3d(sa + 64 * 128, j.ta, &full_bar[s], j.a_c0 + 64, j.a_c1 + i * 64, 0);
        }
        if (!j.b_mn)
          ptx::tma_load_3d(sb, j.tb, &full_bar[s], j.b_c0 + i * 64, j.b_c1, 0);
        else
          ptx::tma_load_3d(sb, j.tb, &full_bar[s], j.b_c0, j.b_c1 + i * 64, 0);
      }
    }
    __syncwarp();
  }
}

template <bool FP8>
__device__ __forceinline__ void mma_tile(const Job& j, uint8_t* smem, uint8_t* sf_smem, uint64_t* full_bar,
                                         uint64_t* empty_bar, uint64_t* accum_bar,
                                         uint32_t tmem_base, Pipe& pp) {
  const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO = 1024, v1, SWIZZLE_128B
  const uint32_t base_lo = ptx::smem_u32(smem) >> 4;
  if (FP8 && j.fp8) {
    const uint32_t idesc0 = epi::make_idesc_mx8(kBM, kBN);
    const uint32_t lo_a0 = base_lo | (1u << 16);
    const uint32_t lo_b0 = (base_lo + (kABytes >> 4)) | (1u << 16);
    const uint32_t tsfa = tmem_base + kTmemSfa, tsfb = tmem_base + kTmemSfb;
    for (int i = 0; i < j.n_kb; ++i, ++pp.it) {
      const int s = pp.it % kStages;
      const uint32_t ph = (pp.it / kStages) & 1;
      ptx::mbar_wait(&full_bar[s], ph);
      ptx::tc_fence_after_sync();
      const uint32_t so = static_cast<uint32_t>(s) * (kStageBytes >> 4);
      if (ptx::elect_one()) {
        // tcgen05.cp and tcgen05.mma execute in issue order: the one scale region in TMEM is
        // rewritten per K-block without any extra barrier
        const uint32_t sfs = ptx::smem_u32(sf_smem + s * kSfStage);
        epi::utccp_32x128b_warpx4(tsfa, epi::sf_desc(sfs));
        epi::utccp_32x128b_warpx4(tsfb, epi::sf_desc(sfs + kSfChunk));
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
          const uint64_t ad = (static_cast<uint64_t>(hi) << 32) | (lo_a0 + so + k * 2u);
          const uint64_t bd = (static_cast<uint64_t>(hi) << 32) | (lo_b0 + so + k * 2u);
          epi::umma_mx8(tmem_base, ad, bd, epi::idesc_mx8_k(idesc0, k), (i > 0 || k > 0) ? 1u : 0u,
                        tsfa, tsfb + j.sfb_col);
        }
        ptx::umma_commit(&empty_bar[s]);
      }
      __syncwarp();
    }
  } else {
    const uint32_t idesc = ptx::make_idesc(1u, j.a_mn ? 1u : 0u, j.b_mn ? 1u : 0u,
                                           static_cast<uint32_t>(j.bm), kBN);
    const uint32_t lbo_a = j.a_mn ? (8192u >> 4) : 1u, lbo_b = j.b_mn ? (8192u >> 4) : 1u;
    const uint32_t lo_a0 = base_lo | (lbo_a << 16);
    const uint32_t lo_b0 = (base_lo + (kABytes >> 4)) | (lbo_b << 16);
    const uint32_t ks_a = (j.a_mn ? 2048u : 32u) >> 4, ks_b = (j.b_mn ? 2048u : 32u) >> 4;
    for (int i = 0; i < j.n_kb; ++i, ++pp.it) {
      const int s = pp.it % kStages;
      const uint32_t ph = (pp.it / kStages) & 1;
      ptx::mbar_wait(&full_bar[s], ph);
      ptx::tc_fence_after_sync();
      const uint32_t so = static_cast<uint32_t>(s) * (kStageBytes >> 4);
      if (ptx::elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint64_t ad = (static_cast<uint64_t>(hi) << 32) | (lo_a0 + so + k * ks_a);
          const uint64_t bd = (static_cast<uint64_t>(hi) << 32) | (lo_b0 + so + k * ks_b);
          ptx::umma_f16(tmem_base, ad, bd, idesc, (i > 0 || k > 0) ? 1u : 0u);
        }
        ptx::umma_commit(&empty_bar[s]);
      }
      __syncwarp();
    }
  }
  if (ptx::elect_one()) ptx::umma_commit(accum_bar);
  __syncwarp();
  ++pp.tile;
}

// SGD / Adam on n (<= 4) consecutive parameters starting at flat index pi, gradient in g0[]:
// fp32 master, bf16 shadow (and the Adam moments) are updated in place; the new values are
// returned in w[].  Coherent loads: other CTAs of this kernel wrote these buffers in earlier phases.
// PROX: the gradient becomes fmaf(mu, w - anchor, g) with w the master before this update (the
// anchor is read-only for the whole launch).
template <bool PROX>
__device__ __forceinline__ void opt_apply(const Args& a, long long pi, int n, const float* g0,
                                          float bc1, float bc2, float (&w)[4]) {
  float m[4], v[4], g[4], an[4];
  const bool vec = n == 4 && (pi & 3) == 0;
  if (vec) {
    const float4 w4 = __ldcg(reinterpret_cast<const float4*>(a.master + pi));
    w[0] = w4.x; w[1] = w4.y; w[2] = w4.z; w[3] = w4.w;
    if (PROX) {
      const float4 a4 = __ldg(reinterpret_cast<const float4*>(a.prox_anchor + pi));
      an[0] = a4.x; an[1] = a4.y; an[2] = a4.z; an[3] = a4.w;
    }
    if (a.adam) {
      const float4 m4 = __ldcg(reinterpret_cast<const float4*>(a.adam_m + pi));
      const float4 v4 = __ldcg(reinterpret_cast<const float4*>(a.adam_v + pi));
      m[0] = m4.x; m[1] = m4.y; m[2] = m4.z; m[3] = m4.w;
      v[0] = v4.x; v[1] = v4.y; v[2] = v4.z; v[3] = v4.w;
    }
  } else {
    for (int k = 0; k < n; ++k) {
      w[k] = __ldcg(a.master + pi + k);
      if (PROX) an[k] = __ldg(a.prox_anchor + pi + k);
      if (a.adam) { m[k] = __ldcg(a.adam_m + pi + k); v[k] = __ldcg(a.adam_v + pi + k); }
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k >= n) break;
    g[k] = PROX ? fmaf(a.prox_mu, w[k] - an[k], g0[k]) : g0[k];
    if (a.adam) {
      m[k] = a.beta1 * m[k] + (1.f - a.beta1) * g[k];
      v[k] = a.beta2 * v[k] + (1.f - a.beta2) * g[k] * g[k];
      w[k] -= a.lr * (m[k] / bc1) / (sqrtf(v[k] / bc2) + a.eps);
    } else {
      w[k] -= a.lr * g[k];
    }
  }
  if (vec) {
    *reinterpret_cast<float4*>(a.master + pi) = make_float4(w[0], w[1], w[2], w[3]);
    *reinterpret_cast<uint2*>(a.shadow + pi) = make_uint2(pack2(w[0], w[1]), pack2(w[2], w[3]));
    if (a.adam) {
      *reinterpret_cast<float4*>(a.adam_m + pi) = make_float4(m[0], m[1], m[2], m[3]);
      *reinterpret_cast<float4*>(a.adam_v + pi) = make_float4(v[0], v[1], v[2], v[3]);
    }
  } else {
    for (int k = 0; k < n; ++k) {
      a.master[pi + k] = w[k];
      a.shadow[pi + k] = __float2bfloat16(w[k]);
      if (a.adam) { a.adam_m[pi + k] = m[k]; a.adam_v[pi + k] = v[k]; }
    }
  }
}

// Accumulator rows of lane quarter q: UMMA M = 128 -> rows 32q .. 32q+31 in lanes 0..31;
// UMMA M = 64 -> row m lives in TMEM lane (m % 16) + 32 * (m / 16): rows 16q .. 16q+15 in the
// quarter's first 16 lanes.
__device__ __forceinline__ int rows_per_quarter(int bm) { return bm == 64 ? 16 : 32; }

// E_OPT: the accumulator tile IS the weight gradient.  Per (row, 4 columns) thread: optimizer on
// the fp32 master (+ moments), bf16 shadow refresh -- master / moments of this thread's elements
// are fetched BEFORE the accumulator wait, so the update pays no exposed load latency (Adam
// without the prefetch: +4.3 us per step, measured).  fp8 mode: the updated tile is parked in
// the staging buffer and re-quantised one K-group (32 columns of a row) per thread.  On the last
// step the values (optionally Byzantine-transformed) also go to the upload buffers the committee
// and the FedAvg kernel read.  PROX: the anchor's float4s are prefetched with the master (same
// reason) and the gradient becomes fmaf(mu, w - anchor, g) before SGD / Adam.
template <bool FP8, bool PROX>
__device__ __forceinline__ void epilogue_opt(const Job& j, const Args& a, int q, int half, int lane,
                                             uint64_t* accum_bar, uint32_t tmem_base, float* stg,
                                             Pipe& pp) {
  const int rpq = rows_per_quarter(j.bm);
  const int n_it = rpq / 4;                      // staged store iterations: 4 rows each
  const int row_base = j.m0 + q * rpq;
  const int cr = lane >> 3, cg = (lane & 7) * 4;
  const int nc = j.n0 + half * 32;               // this warp's 32 columns
  const long long pbase = reinterpret_cast<float*>(j.d) - a.master;
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + half * 32;
  float4 wpre[8], mpre[8], vpre[8], apre[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int rw = row_base + it * 4 + cr, col = nc + cg;
    const bool ok = it < n_it && rw < j.M && col + 3 < j.N;
    const long long pi = pbase + static_cast<long long>(rw) * j.ldd + col;
    wpre[it] = ok ? __ldcg(reinterpret_cast<const float4*>(a.master + pi)) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (PROX)
      apre[it] = ok ? __ldg(reinterpret_cast<const float4*>(a.prox_anchor + pi)) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.adam) {
      mpre[it] = ok ? __ldcg(reinterpret_cast<const float4*>(a.adam_m + pi)) : make_float4(0.f, 0.f, 0.f, 0.f);
      vpre[it] = ok ? __ldcg(reinterpret_cast<const float4*>(a.adam_v + pi)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  const bool up = j.last && a.has_fed;
  UploadDst ud{};
  if (up) ud = upload_dst<FP8>(a);
  uint8_t* qblob = (FP8 && up) ? ud.blob : a.work_q;
  ptx::mbar_wait(accum_bar, pp.tile & 1);
  ptx::tc_fence_after_sync();
  ++pp.tile;
  const bool stampit = j.dbg != nullptr && blockIdx.x == 0 && threadIdx.x == kEpiT0;
  if (stampit) j.dbg[j.dbg_slot] = globaltimer_ns();
  {
    uint32_t r[32];
    ptx::tmem_ld_32x32b_x32(taddr, r);
    ptx::tmem_ld_wait();
    float v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(r[k]);
    stage_put(stg, lane, v);
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      if (it >= n_it) break;
      const int rr = it * 4 + cr, rw = row_base + rr, col = nc + cg;
      const bool valid = rw < j.M && col + 3 < j.N;
      const long long pi = pbase + static_cast<long long>(rw) * j.ldd + col;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid) {
        float4 g = *reinterpret_cast<const float4*>(stg + rr * kStgLd + cg);
        w = wpre[it];
        if (PROX) {
          const float mu = a.prox_mu;
          g.x = fmaf(mu, w.x - apre[it].x, g.x); g.y = fmaf(mu, w.y - apre[it].y, g.y);
          g.z = fmaf(mu, w.z - apre[it].z, g.z); g.w = fmaf(mu, w.w - apre[it].w, g.w);
        }
        if (a.adam) {
          float4 m = mpre[it], s = vpre[it];
          const float b1 = a.beta1, b2 = a.beta2, c1 = 1.f - a.beta1, c2 = 1.f - a.beta2;
          m.x = b1 * m.x + c1 * g.x; m.y = b1 * m.y + c1 * g.y; m.z = b1 * m.z + c1 * g.z; m.w = b1 * m.w + c1 * g.w;
          s.x = b2 * s.x + c2 * g.x * g.x; s.y = b2 * s.y + c2 * g.y * g.y;
          s.z = b2 * s.z + c2 * g.z * g.z; s.w = b2 * s.w + c2 * g.w * g.w;
          w.x -= a.lr * (m.x / j.bc1) / (sqrtf(s.x / j.bc2) + a.eps);
          w.y -= a.lr * (m.y / j.bc1) / (sqrtf(s.y / j.bc2) + a.eps);
          w.z -= a.lr * (m.z / j.bc1) / (sqrtf(s.z / j.bc2) + a.eps);
          w.w -= a.lr * (m.w / j.bc1) / (sqrtf(s.w / j.bc2) + a.eps);
          *reinterpret_cast<float4*>(a.adam_m + pi) = m;
          *reinterpret_cast<float4*>(a.adam_v + pi) = s;
        } else {
          w.x -= a.lr * g.x; w.y -= a.lr * g.y; w.z -= a.lr * g.z; w.w -= a.lr * g.w;
        }
        *reinterpret_cast<float4*>(a.master + pi) = w;
        *reinterpret_cast<uint2*>(a.shadow + pi) = make_uint2(pack2(w.x, w.y), pack2(w.z, w.w));
        if (up) {
          if (ud.global != nullptr) {   // Byzantine client (fault injection, SURVEY.md 5.3)
            const float4 g0 = __ldcg(reinterpret_cast<const float4*>(ud.global + pi));
            w.x = g0.x - ud.byz_scale * (w.x - g0.x); w.y = g0.y - ud.byz_scale * (w.y - g0.y);
            w.z = g0.z - ud.byz_scale * (w.z - g0.z); w.w = g0.w - ud.byz_scale * (w.w - g0.w);
          }
          *reinterpret_cast<float4*>(ud.master + pi) = w;
          if (!FP8) *reinterpret_cast<uint2*>(ud.shadow + pi) = make_uint2(pack2(w.x, w.y), pack2(w.z, w.w));
        }
      }
      // fp8: park the updated values in the staging tile (over the gradient this thread just
      // consumed); they are re-quantised row-wise below
      if (FP8) *reinterpret_cast<float4*>(stg + rr * kStgLd + cg) = w;
    }
    if (FP8) {
      // One thread per row of the staged sub-tile: its 32 columns are exactly one K-group of the
      // weight matrix -> amax, UE8M0 byte and 32 e4m3 bytes without any shuffle, two 16-byte
      // stores (a shuffle-per-4-columns version cost 3.7 us per step, measured).
      __syncwarp();
      const int rw = row_base + lane;
      const int nv = j.N - nc < 32 ? j.N - nc : 32;          // valid columns of this group (multiple of 4)
      if (lane < rpq && rw < j.M && nv > 0) {
        float x[32];
        stage_get(stg, lane, x);
        uint32_t w8[8];
        const int e = epi::mx8_quant32(x, w8);
        uint4* qd = reinterpret_cast<uint4*>(qblob + j.q_off + static_cast<long long>(rw) * j.ldq + nc);
        qd[0] = make_uint4(w8[0], w8[1], w8[2], w8[3]);
        if (nv > 16) qd[1] = make_uint4(w8[4], w8[5], w8[6], w8[7]);
        qblob[j.qsf_off + epi::mx8_sf_index(rw, nc >> 5, j.q_nkb)] = static_cast<uint8_t>(e);
      }
    }
    __syncwarp();
  }
  ptx::tc_fence_before_sync();
  if (stampit) j.dbg[j.dbg_slot + 1] = globaltimer_ns();
}

// epilogue warps 4..11: q = TMEM lane quarter, half = which 32 of the tile's 64 columns
template <bool FP8, bool PROX>
__device__ __forceinline__ void epilogue_tile(const Job& j, const Args& a, int q, int half, int lane,
                                              uint64_t* accum_bar, uint32_t tmem_base,
                                              float* stg, float* sbias, Pipe& pp) {
  {
    const int et = threadIdx.x - kEpiT0;
    // coherent (L2) loads: the biases are rewritten by the optimizer phase of this same kernel
    if (et < kBN) sbias[et] = (j.bias != nullptr && j.n0 + et < j.N) ? __ldcg(j.bias + j.n0 + et) : 0.f;
    epi_bar();
  }
  if (j.mode == E_OPT) {
    epilogue_opt<FP8, PROX>(j, a, q, half, lane, accum_bar, tmem_base, stg, pp);
    return;
  }
  const int rpq = rows_per_quarter(j.bm);
  const int row_base = j.m0 + q * rpq;
  const int row = row_base + lane;
  const bool row_ok = lane < rpq && row < j.M;
  const int cr = lane >> 3, cg = (lane & 7) * 4;
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  ptx::mbar_wait(accum_bar, pp.tile & 1);
  ptx::tc_fence_after_sync();
  ++pp.tile;
  const bool stampit = j.dbg != nullptr && blockIdx.x == 0 && threadIdx.x == kEpiT0;
  if (stampit) j.dbg[j.dbg_slot] = globaltimer_ns();

  if (j.mode != E_XENT) {
    const int c = half;
    const int nc = j.n0 + c * 32;
    if (nc < j.N) {
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c * 32, r);
      ptx::tmem_ld_wait();
      float v[32];
#pragma unroll
      for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(r[k]) + sbias[c * 32 + k];
      if (j.mode == E_BIAS_RELU_BF16) {
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] = fmaxf(v[k], 0.f);
        if (FP8 && j.fp8 && row_ok) {
          // fwd2's A operand: this thread's 32 columns of h are exactly one K-group
          uint32_t w[8];
          const int e = epi::mx8_quant32(v, w);
          uint4* hq = reinterpret_cast<uint4*>(a.h_q + static_cast<long long>(row) * a.hidden + nc);
          hq[0] = make_uint4(w[0], w[1], w[2], w[3]);
          hq[1] = make_uint4(w[4], w[5], w[6], w[7]);
          a.h_sf[epi::mx8_sf_index(row, nc >> 5, a.ql.kb2)] = static_cast<uint8_t>(e);
        }
      } else if (j.mode == E_MASK_COLSUM_BF16) {
        // coalesced (L2-coherent) load of the mask tile through the staging buffer
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int rr = it * 4 + cr, rw = row_base + rr, col = nc + cg;
          float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
          if (rr < rpq && rw < j.M && col + 3 < j.N) {
            const uint2 u = __ldcg(reinterpret_cast<const uint2*>(j.aux + static_cast<long long>(rw) * j.ldd + col));
            const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
            const float2 hi2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
            x = make_float4(lo.x, lo.y, hi2.x, hi2.y);
          }
          *reinterpret_cast<float4*>(stg + rr * kStgLd + cg) = x;
        }
        __syncwarp();
        float m[32];
        stage_get(stg, lane, m);
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] = m[k] > 0.f ? v[k] : 0.f;
      }
      stage_put(stg, lane, v);
      __syncwarp();
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int rr = it * 4 + cr, rw = row_base + rr, col = nc + cg;
        if (rr >= rpq || rw >= j.M || col >= j.N) continue;
        const float4 x = *reinterpret_cast<const float4*>(stg + rr * kStgLd + cg);
        const long long off = static_cast<long long>(rw) * j.ldd + col;
        if (j.mode == E_F32) {
          float* d = reinterpret_cast<float*>(j.d) + off;
          if (col + 3 < j.N) *reinterpret_cast<float4*>(d) = x;
          else {
            const float xs[4] = {x.x, x.y, x.z, x.w};
            for (int k = 0; k < 4; ++k) if (col + k < j.N) d[k] = xs[k];
          }
        } else {
          __nv_bfloat16* d = reinterpret_cast<__nv_bfloat16*>(j.d) + off;
          *reinterpret_cast<uint2*>(d) = make_uint2(pack2(x.x, x.y), pack2(x.z, x.w));
        }
      }
      if (j.colsum != nullptr) {
        const float tot = col_sum32(stg, lane, min(rpq, j.M - row_base));
        if (nc + lane < j.N) atomicAdd(j.colsum + nc + lane, tot);
      }
      __syncwarp();
    }
  } else if (half == 0) {
    // softmax cross-entropy over the N (<= 64) logits of each row (plan 0 only: general hidden
    // sizes; one thread owns a whole row, the second half of the epilogue warps idles)
    const int32_t label = row_ok ? j.labels[row] : -1;
    float vmax = -INFINITY, zlab = 0.f;
    int amax = -1;
    float z[64];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c * 32, r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const int n = c * 32 + k;
        const float x = __uint_as_float(r[k]) + sbias[n];
        z[n] = x;
        if (n < j.N) {
          if (x > vmax) { vmax = x; amax = n; }
          if (n == label) zlab = x;
        }
      }
    }
    float sum = 0.f;
#pragma unroll
    for (int n = 0; n < 64; ++n)
      if (n < j.N) sum += __expf(z[n] - vmax);
    const float inv = 1.f / sum;
    float loss = row_ok ? (__logf(sum) + vmax - zlab) : 0.f;
    const bool hit = row_ok && (amax == label);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      float v[32];
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const int n = c * 32 + k;
        v[k] = (n < j.N && row_ok)
                   ? (__expf(z[n] - vmax) * inv - (n == label ? 1.f : 0.f)) * j.grad_scale
                   : 0.f;
      }
      stage_put(stg, lane, v);
      __syncwarp();
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int rr = it * 4 + cr, rw = row_base + rr, col = c * 32 + cg;
        if (rw >= j.M || col >= j.ldd) continue;
        const float4 x = *reinterpret_cast<const float4*>(stg + rr * kStgLd + cg);
        __nv_bfloat16* d = reinterpret_cast<__nv_bfloat16*>(j.d) + static_cast<long long>(rw) * j.ldd + col;
        *reinterpret_cast<uint2*>(d) = make_uint2(pack2(x.x, x.y), pack2(x.z, x.w));
      }
      if (j.colsum != nullptr) {
        const float tot = col_sum32(stg, lane, 32);
        if (c * 32 + lane < j.N) atomicAdd(j.colsum + c * 32 + lane, tot);
      }
      __syncwarp();
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, off);
    const unsigned cnt = __popc(__ballot_sync(0xffffffffu, hit));
    if (lane == 0) {
      atomicAdd(a.loss_sum, loss);
      if (cnt) atomicAdd(a.correct, cnt);
    }
  }
  ptx::tc_fence_before_sync();
  if (stampit) j.dbg[j.dbg_slot + 1] = globaltimer_ns();
}

// ---------------------------------------------------------------- fused chain of one 128-row tile
//   (h was produced by P1 and arrives by TMA -- bf16, or e4m3 + scale chunks)
//   fwd2  logits[128 x 64] = h W2^T          (A, B from smem)                    TMEM cols [256,320)
//   E2    softmax-xent per row -> dlogits -> smem (dh's A operand) + global
//   dh    acc[128 x 64 slice] = dlogits W2   (B = W2 MN-major)                   TMEM cols [0,64)
//   E3    dh = acc * relu'(h) -> bf16 global, db1
// logits / dlogits never make the global -> TMA round trip; the three GEMMs cost one grid barrier.
// Four CTAs per M-tile: all redo the cheap fwd2 + xent so that the dh GEMM and its epilogue run
// 4-wide (64 hidden columns each); loss, db2 and the global dlogits copy are done by one of them.
template <bool FP8>
__device__ __forceinline__ void chain_produce(const Maps& maps, const Args& a, uint8_t* smem, uint8_t* sf_smem,
                                              const ChainBars& cb, int m0, int slice) {
  if (ptx::elect_one()) {
    if (FP8) {
      // e4m3: two K-blocks of 128 hidden units each, plus their scale chunks
      ptx::mbar_expect_tx(cb.w2k, 2 * 8192 + 2 * kSfChunk);
      ptx::mbar_expect_tx(cb.h, 2 * 16384 + 2 * kSfChunk);
      ptx::mbar_expect_tx(cb.w2mn, 8192);
#pragma unroll
      for (int kb = 0; kb < 2; ++kb) {
        ptx::tma_load_3d(smem + kOffH + kb * 16384, &maps.hq_k, cb.h, kb * 128, m0, 0);
        epi::bulk_g2s(sf_smem + kb * kSfChunk,
                      a.h_sf + (static_cast<long long>(m0 >> 7) * a.ql.kb2 + kb) * kSfChunk, kSfChunk, cb.h);
      }
#pragma unroll
      for (int kb = 0; kb < 2; ++kb) {
        ptx::tma_load_3d(smem + kOffW2K + kb * 8192, &maps.w2q_k, cb.w2k, kb * 128, 0, 0);
        epi::bulk_g2s(sf_smem + (2 + kb) * kSfChunk, a.work_q + a.ql.w2sf + kb * kSfChunk, kSfChunk, cb.w2k);
      }
      ptx::tma_load_3d(smem + kOffW2MN, &maps.w2_mn, cb.w2mn, slice * 64, 0, 0);
    } else {
      ptx::mbar_expect_tx(cb.w2k, 32768);
      ptx::mbar_expect_tx(cb.h, 65536);
      ptx::mbar_expect_tx(cb.w2mn, 8192);
      // in the order the chain consumes them: h and W2 (fwd2) first, W2^T (dh) last
#pragma unroll
      for (int kb = 0; kb < 4; ++kb)
        ptx::tma_load_3d(smem + kOffH + kb * 16384, &maps.h_k, cb.h, kb * 64, m0, 0);
#pragma unroll
      for (int kb = 0; kb < 4; ++kb)
        ptx::tma_load_3d(smem + kOffW2K + kb * 8192, &maps.w2_k, cb.w2k, kb * 64, 0, 0);
      ptx::tma_load_3d(smem + kOffW2MN, &maps.w2_mn, cb.w2mn, slice * 64, 0, 0);
    }
  }
  __syncwarp();
}

template <bool FP8>
__device__ __forceinline__ void chain_mma(uint8_t* smem, uint8_t* sf_smem, const ChainBars& cb,
                                          uint32_t tmem_base, uint32_t par) {
  const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
  const uint32_t base_lo = ptx::smem_u32(smem) >> 4;
  // fwd2: 128 x 64 x 256, A = h (TMA), B = W2 K-major
  ptx::mbar_wait(cb.w2k, par);
  ptx::mbar_wait(cb.h, par);
  ptx::tc_fence_after_sync();
  if (ptx::elect_one()) {
    const uint32_t lo_a0 = (base_lo + (static_cast<uint32_t>(kOffH) >> 4)) | (1u << 16);
    const uint32_t lo_b0 = (base_lo + (static_cast<uint32_t>(kOffW2K) >> 4)) | (1u << 16);
    if (FP8) {
      const uint32_t idq = epi::make_idesc_mx8(kBM, 64);
      const uint32_t tsfa = tmem_base + kTmemSfa, tsfb = tmem_base + kTmemSfb;
      const uint32_t sfs = ptx::smem_u32(sf_smem);
#pragma unroll
      for (uint32_t kb = 0; kb < 2; ++kb) {
        epi::utccp_32x128b_warpx4(tsfa, epi::sf_desc(sfs + kb * kSfChunk));
        epi::utccp_32x128b_warpx4(tsfb, epi::sf_desc(sfs + (2 + kb) * kSfChunk));
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k)
          epi::umma_mx8(tmem_base + 256, (static_cast<uint64_t>(hi) << 32) | (lo_a0 + kb * (16384u >> 4) + k * 2u),
                        (static_cast<uint64_t>(hi) << 32) | (lo_b0 + kb * (8192u >> 4) + k * 2u),
                        epi::idesc_mx8_k(idq, k), (kb > 0 || k > 0) ? 1u : 0u, tsfa, tsfb);
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
    ptx::umma_commit(cb.acc_l);
  }
  __syncwarp();
  // dh: 128 x 64 x 64, A = dlogits (smem, written by the epilogue warps), B = W2 MN-major slice
  ptx::mbar_wait(cb.w2mn, par);
  ptx::mbar_wait(cb.dl_ready, par);
  ptx::tc_fence_after_sync();
  if (ptx::elect_one()) {
    const uint32_t id3 = ptx::make_idesc(1u, 0u, 1u, kBM, 64);
    const uint32_t lo_a0 = (base_lo + (static_cast<uint32_t>(kOffDL) >> 4)) | (1u << 16);
    const uint32_t lo_b0 = (base_lo + (static_cast<uint32_t>(kOffW2MN) >> 4)) | ((8192u >> 4) << 16);
#pragma unroll
    for (uint32_t k = 0; k < 4; ++k)
      ptx::umma_f16(tmem_base, (static_cast<uint64_t>(hi) << 32) | (lo_a0 + k * 2u),
                    (static_cast<uint64_t>(hi) << 32) | (lo_b0 + k * (2048u >> 4)), id3, k > 0 ? 1u : 0u);
    ptx::umma_commit(cb.acc_dh);
  }
  __syncwarp();
}

// Epilogue of the chain.  Thread (q, half, lane) owns row rl = 32q + lane of the M-tile and the
// column half `half`: logits [32 half, +32) in E2, hidden columns [32 half, +32) of this CTA's
// 64-column dh slice in E3.  The two threads of a row combine their softmax partials through a
// small smem exchange (xch) around two 256-thread named barriers.
template <bool FP8>
__device__ __forceinline__ void chain_epilogue(const Args& a, uint8_t* smem, const ChainBars& cb,
                                               uint32_t tmem_base, int q, int half, int lane, float* stg,
                                               float* sb, float* xch, uint32_t par, int m0, int r0, int slice,
                                               unsigned long long* dbg) {
  auto stampc = [&](int slot) {
    if (dbg != nullptr && blockIdx.x == 0 && threadIdx.x == kEpiT0) dbg[slot] = globaltimer_ns();
  };
  const int rl = q * 32 + lane;        // row inside the tile == TMEM lane
  const int row = m0 + rl;             // row inside the mini-batch
  const bool row_ok = row < a.B;
  const int32_t label = row_ok ? __ldg(a.labels + r0 + row) : -1;   // issued early: needed by E2
  const int C = a.n_classes;
  {
    const int et = threadIdx.x - kEpiT0;   // coherent loads: the optimizer of this kernel rewrites the biases
    sb[et] = __ldcg(a.b1 + et);        // kEpiThreads == kChainH == 256
    if (et < 64) sb[kChainH + et] = et < C ? __ldcg(a.b2 + et) : 0.f;
    epi_bar();
  }
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  float* xmax = xch + half * 128;            const float* omax = xch + (1 - half) * 128;
  float* xidx = xch + 256 + half * 128;      const float* oidx = xch + 256 + (1 - half) * 128;
  float* xzl = xch + 512 + half * 128;       const float* ozl = xch + 512 + (1 - half) * 128;
  float* xsum = xch + 768 + half * 128;      const float* osum = xch + 768 + (1 - half) * 128;

  // ---- E1: relu mask of this thread's 32 hidden columns [64 slice + 32 half, +32), read back
  //          through the swizzle from the h tile the TMA dropped into the A-operand slots
  uint32_t mk = 0u;
  ptx::mbar_wait(cb.h, par);
  stampc(6);
  {
    const uint8_t* hs = smem + kOffH;
    if (FP8) {
      // e4m3: K-block (slice / 2) holds hidden units [128 * (slice / 2), +128), one byte each
      const uint8_t* tile = hs + (slice >> 1) * 16384;
#pragma unroll
      for (int jj = 0; jj < 2; ++jj) {
        const uint4 u = epi::ld_sw128(tile, rl, (slice & 1) * 4 + half * 2 + jj);
        const uint32_t wds[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int e = 0; e < 4; ++e)
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const uint32_t byte = (wds[e] >> (8 * b)) & 0xFFu;   // e4m3 > 0  <=>  sign clear, not zero
            mk |= ((byte != 0u && (byte & 0x80u) == 0u) ? 1u : 0u) << (jj * 16 + e * 4 + b);
          }
      }
    } else {
      const int c = 2 * slice + half;       // 32-column chunk of the 256 hidden units
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const uint4 u = epi::ld_sw128(hs + (c >> 1) * 16384, rl, (c & 1) * 4 + jj);
        const uint32_t wds[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          // bf16 > 0  <=>  sign clear and not zero
          mk |= (((wds[e] & 0xFFFFu) != 0u && (wds[e] & 0x8000u) == 0u) ? 1u : 0u) << (jj * 8 + e * 2);
          mk |= (((wds[e] >> 16) != 0u && (wds[e] & 0x80000000u) == 0u) ? 1u : 0u) << (jj * 8 + e * 2 + 1);
        }
      }
    }
  }
  stampc(7);

  // ---- E2: softmax cross-entropy of the row, 32 logits per thread
  ptx::mbar_wait(cb.acc_l, par);
  ptx::tc_fence_after_sync();
  stampc(8);
  {
    float z[32];
    {
      uint32_t ra[32];
      ptx::tmem_ld_32x32b_x32(taddr + 256 + half * 32, ra);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int k = 0; k < 32; ++k) z[k] = __uint_as_float(ra[k]) + sb[kChainH + half * 32 + k];
    }
    const int nb = half * 32;
    float pm[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    int pi[4] = {-1, -1, -1, -1};
    float zlab = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      if (nb + k < C) {
        if (z[k] > pm[k & 3]) { pm[k & 3] = z[k]; pi[k & 3] = nb + k; }
        if (nb + k == label) zlab = z[k];
      }
    }
    float vmax = pm[0];
    int amax = pi[0];
#pragma unroll
    for (int jq = 1; jq < 4; ++jq)   // first maximum wins, as in a serial scan
      if (pm[jq] > vmax || (pm[jq] == vmax && pi[jq] >= 0 && pi[jq] < amax)) { vmax = pm[jq]; amax = pi[jq]; }
    xmax[rl] = vmax; xidx[rl] = __int_as_float(amax); xzl[rl] = zlab;
    epi_bar();
    {
      const float ov = omax[rl];
      const int oi = __float_as_int(oidx[rl]);
      // the lower half holds the lower class indices: it wins ties
      const bool take = half == 0 ? (ov > vmax) : (ov >= vmax && oi >= 0);
      if (take) { vmax = ov; amax = oi; }
      zlab += ozl[rl];
    }
    stampc(12);
    float ps[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 32; ++k) {   // z <- exp(z - max): each exponential is evaluated once
      z[k] = nb + k < C ? __expf(z[k] - vmax) : 0.f;
      ps[k & 3] += z[k];
    }
    const float psum = (ps[0] + ps[1]) + (ps[2] + ps[3]);
    xsum[rl] = psum;
    epi_bar();
    const float sum = psum + osum[rl];
    const float inv = 1.f / sum;
    const float gs = 1.f / static_cast<float>(a.B);
    // the 4 slice-CTAs of an M-tile all need dlogits in smem, but the bookkeeping is done once:
    const bool do_colsum = slice == 1, do_global = slice == 2, do_loss = slice == 3 && half == 0;
    uint8_t* dls = smem + kOffDL;
    {
      float v[32];
#pragma unroll
      for (int k = 0; k < 32; ++k)
        v[k] = (nb + k < C && row_ok) ? (z[k] * inv - (nb + k == label ? 1.f : 0.f)) * gs : 0.f;
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const uint4 u = make_uint4(pack2(v[8 * jj], v[8 * jj + 1]), pack2(v[8 * jj + 2], v[8 * jj + 3]),
                                   pack2(v[8 * jj + 4], v[8 * jj + 5]), pack2(v[8 * jj + 6], v[8 * jj + 7]));
        st_sw128(dls, rl, half * 4 + jj, u);
      }
      if (do_colsum) {
        stage_put(stg, lane, v);
        __syncwarp();
        const float tot = col_sum32(stg, lane, 32);
        if (nb + lane < C) atomicAdd(a.gb2 + nb + lane, tot);
        __syncwarp();
      }
    }
    // hand the tile to the dh MMA first, then finish the bookkeeping underneath it
    stampc(13);
    ptx::fence_proxy_async_smem();
    ptx::tc_fence_before_sync();
    ptx::mbar_arrive(cb.dl_ready);
    stampc(14);
    // dlogits -> global for dW2, read back out of the swizzled tile: one store instruction covers
    // 8 rows x this half's 64 bytes (a row-per-thread store touches 32 lines per instruction)
    __syncwarp();
    if (do_global) {
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int rt = q * 32 + it * 8 + (lane >> 2), ch = half * 4 + (lane & 3);
        const uint4 u = epi::ld_sw128(dls, rt, ch);
        if (m0 + rt < a.B && ch * 8 < a.ncp)
          *reinterpret_cast<uint4*>(a.dlogits + static_cast<long long>(m0 + rt) * a.ncp + ch * 8) = u;
      }
    }
    if (do_loss) {
      float loss = row_ok ? (__logf(sum) + vmax - zlab) : 0.f;
      const bool hit = row_ok && (amax == label);
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, off);
      const unsigned cnt = __popc(__ballot_sync(0xffffffffu, hit));
      if (lane == 0) {
        atomicAdd(a.loss_sum, loss);
        if (cnt) atomicAdd(a.correct, cnt);
      }
    }
  }
  stampc(9);

  // ---- E3: dh = (dlogits W2) * relu'(h), db1 -- 32 hidden columns per thread
  ptx::mbar_wait(cb.acc_dh, par);
  ptx::tc_fence_after_sync();
  stampc(10);
  {
    // The h tile at kOffH is dead (fwd2 retired before acc_l, the mask is in registers): its first
    // 16 KB become a bf16 staging tile (128 rows x 128 bytes) so that dh leaves the SM 8 rows x 64
    // bytes per store instruction instead of 32 scattered 16-byte pieces.
    uint8_t* ds = smem + kOffH;
    uint32_t r[32];
    ptx::tmem_ld_32x32b_x32(taddr + half * 32, r);
    ptx::tmem_ld_wait();
    float v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = ((mk >> k) & 1u) ? __uint_as_float(r[k]) : 0.f;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
      st_sw128(ds, rl, half * 4 + jj,
               make_uint4(pack2(v[8 * jj], v[8 * jj + 1]), pack2(v[8 * jj + 2], v[8 * jj + 3]),
                          pack2(v[8 * jj + 4], v[8 * jj + 5]), pack2(v[8 * jj + 6], v[8 * jj + 7])));
    stage_put(stg, lane, v);
    __syncwarp();
    const float tot = col_sum32(stg, lane, 32);
    atomicAdd(a.gb1 + (2 * slice + half) * 32 + lane, tot);
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int rt = q * 32 + it * 8 + (lane >> 2), ch = half * 4 + (lane & 3);
      const uint4 u = epi::ld_sw128(ds, rt, ch);
      if (m0 + rt < a.B)
        *reinterpret_cast<uint4*>(a.dh + static_cast<long long>(m0 + rt) * a.hidden + slice * 64 + ch * 8) = u;
    }
    __syncwarp();
  }
  ptx::tc_fence_before_sync();
  stampc(11);
}

// Device-wide barrier between phases.  All CTAs are co-resident (one per SM), the counter
// only grows.  Writers: bar.sync orders every thread's writes before thread 0's gpu-scope
// fence (cumulative release); readers: acquire, then a proxy fence so the next phase's TMA
// (async proxy) observes what other CTAs stored with ordinary instructions.  `sys`: the writes
// of this phase are about to be published to peer GPUs (last step's upload) -- fence at system
// scope instead.
__device__ __forceinline__ void grid_barrier(unsigned int* counter, unsigned int& epoch, bool sys = false) {
  ++epoch;
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (threadIdx.x == 0) {
    ptx::fence_proxy_async_all();
    if (sys) __threadfence_system(); else __threadfence();
    atomicAdd(counter, 1u);
    const unsigned int target = epoch * gridDim.x;
    unsigned long long spins = 0;
    while (true) {
      unsigned int v;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (v >= target) break;
      if (++spins > (1ull << 27)) __trap();  // a lost CTA traps within seconds instead of hanging
    }
    ptx::fence_proxy_async_all();
  }
  __syncthreads();
  ptx::tc_fence_after_sync();
}

// PROX: FedProx term in every optimizer update.  A template parameter, not a runtime branch, so
// that the default instantiations keep their register allocation.
template <bool FP8, bool PROX>
__global__ void __launch_bounds__(kThreads, 1)
mlp_round_kernel(const __grid_constant__ Maps maps, const Args a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sf_smem = smem + kTileBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kTileBytes + kSfBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* accum_bar = empty_bar + kStages;
  uint64_t* cbar = accum_bar + 1;      // chain barriers
  ChainBars cb{cbar, cbar + 1, cbar + 2, cbar + 3, cbar + 4, cbar + 5};
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(cbar + 6);
  float* stage_base = reinterpret_cast<float*>(smem + kTileBytes + kSfBytes + kBarBytes);
  float* sbias = stage_base + kEpiWarps * 32 * kStgLd;
  float* xch = sbias + kBiasFloats;

  ptx::pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    ptx::mbar_init(accum_bar, 1);
    ptx::mbar_init(cb.h, 1); ptx::mbar_init(cb.w2k, 1); ptx::mbar_init(cb.w2mn, 1);
    ptx::mbar_init(cb.acc_l, 1); ptx::mbar_init(cb.acc_dh, 1);
    ptx::mbar_init(cb.dl_ready, kEpiThreads);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc(tmem_slot, kTmemCols);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  ptx::pdl_wait();
  if (a.pred != nullptr && *a.pred == 0) {
    if (warp == 1) ptx::tmem_dealloc(tmem_base, kTmemCols);
    return;
  }

  Pipe pp{0u, 0u};
  uint32_t chains = 0;        // chains processed by this CTA (parity of the once-per-chain barriers)
  bool x_all_ready = false;   // input pipeline: every chunk of this round has been converted
  unsigned int bar_epoch = 0;
  const int t = blockIdx.x;
  const int q = warp & 3, half = (warp - 4) >> 2;       // epilogue warps 4..11
  float* stg = stage_base + (warp >= 4 ? warp - 4 : 0) * (32 * kStgLd);
  const int B = a.B, H = a.hidden, C = a.n_classes, D = a.in_dim;
  const int mt_b = (B + kBM - 1) / kBM;                 // M-tiles over the batch
  const int nt_h = (H + kBN - 1) / kBN;                 // N-tiles over hidden
  const int nt_d = (D + kBN - 1) / kBN;                 // N-tiles over in_dim
  const int bm_w = a.bm_w;                              // weight-gradient tile height (64 | 128)
  const int mt_hw = (H + bm_w - 1) / bm_w;              // M-tiles over hidden (dW1)
  const int kb_d = (D + 63) / 64, kb_h = (H + 63) / 64, kb_b = (B + 63) / 64, kb_c = (C + 63) / 64;
  const int p1_tiles = mt_b * nt_h;

  // The step loop exists twice, specialised per role group, so that each side of the
  // `setmaxnreg` split is compiled against its own register budget: EPI = false is warpgroup 0
  // (TMA producer, MMA issuer, two idle warps), EPI = true the eight epilogue warps.  Both copies
  // execute the same sequence of CTA-wide barriers.
  auto round_loop = [&](auto epi_tag) {
  constexpr bool EPI = decltype(epi_tag)::value;
  auto run = [&](const Job& j) {
    if constexpr (EPI) {
      epilogue_tile<FP8, PROX>(j, a, q, half, lane, accum_bar, tmem_base, stg, sbias, pp);
    } else {
      if (warp == 0) produce_tile<FP8>(j, smem, sf_smem, full_bar, empty_bar, pp);
      else if (warp == 1) mma_tile<FP8>(j, smem, sf_smem, full_bar, empty_bar, accum_bar, tmem_base, pp);
    }
  };

  // Phase plan of one step (a.chain, a.epiopt pick the variant; all are numerically equivalent):
  //   chain 3:  P1 fwd1 | [fwd2 -> xent -> dh chained per M-tile]             | B
  //   chain 0:  P1 | P2 xent | P3 dh                                          | B   (any hidden size)
  //   B = dW1 || dW2 (+ SGD/Adam in the epilogue and a bias CTA when epiopt, else a flat P5)
  auto stamp = [&](int step, int slot) {
    if (a.dbg != nullptr && blockIdx.x == 0 && threadIdx.x == kEpiT0) a.dbg[step * 32 + slot] = globaltimer_ns();
  };
  for (int step = 0; step < a.steps; ++step) {
    const int r0 = step * B;
    const bool last = step == a.steps - 1;
    float bc1 = 1.f, bc2 = 1.f;
    if (a.adam) {
      const int tt = (a.step_base ? *a.step_base : 0) + step + 1;
      bc1 = 1.f - powf(a.beta1, static_cast<float>(tt));
      bc2 = 1.f - powf(a.beta2, static_cast<float>(tt));
    }
    const bool eo = a.epiopt != 0;
    unsigned long long* sdbg = a.dbg != nullptr ? a.dbg + step * 32 : nullptr;
    stamp(step, 0);
    // ---- P1: h = relu(x W1^T + b1)
    if (t < p1_tiles) {
      if (!EPI && a.x_ready != nullptr && warp == 0 && !x_all_ready) {
        // input pipeline: this step's rows are converted by the side-branch kernel as soon as
        // their H2D copy lands; only the TMA producer has to wait (phase B reads them later).
        // Once the LAST chunk is seen ready nothing is checked any more.
        int all = 0;
        if (lane == 0) {
          const unsigned int want = __ldcg(a.round_seq) + 1u;   // bumped by k_consensus at round end
          unsigned int v;
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(a.x_ready + a.steps - 1) : "memory");
          all = static_cast<int>(v - want) >= 0 ? 1 : 0;
          unsigned long long spins = 0;
          while (!all) {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(a.x_ready + step) : "memory");
            if (static_cast<int>(v - want) >= 0) break;
            if (++spins > (1ull << 28)) __trap();   // the input kernel gives up (error word) long before this
            __nanosleep(32);
          }
        }
        x_all_ready = __shfl_sync(0xffffffffu, all, 0) != 0;
        ptx::fence_proxy_async_all();   // their generic stores -> this warp's TMA (async proxy) loads
      }
      Job j{};
      j.mode = E_BIAS_RELU_BF16; j.d = a.h; j.ldd = H; j.bias = a.b1; j.M = B; j.N = H; j.bm = kBM;
      j.dbg = sdbg; j.dbg_slot = 16;
      j.m0 = (t / nt_h) * kBM; j.n0 = (t % nt_h) * kBN;
      if (FP8) {
        // e4m3 x tile against a 64-row tile of e4m3 W1; scale chunks are per 128-row block, the
        // W1 tile's rows start at TMEM column (row % 128) / 32 of the 4-column chunk (0 or 2)
        const int kbq = a.ql.kb1;
        const int xr = r0 + j.m0;
        j.fp8 = 1; j.n_kb = kbq;
        j.ta = &maps.xq_k; j.tb = &maps.w1q_k;
        j.a_c0 = 0; j.a_c1 = xr; j.b_c0 = 0; j.b_c1 = j.n0;
        j.sfa = a.x_sf + static_cast<long long>(xr >> 7) * kbq * kSfChunk;
        j.sfb = a.work_q + a.ql.w1sf + static_cast<long long>(j.n0 >> 7) * kbq * kSfChunk;
        j.sfb_col = static_cast<uint32_t>((j.n0 & 127) >> 5);
      } else {
        j.ta = &maps.x_k; j.tb = &maps.w1_k; j.a_mn = 0; j.b_mn = 0;
        j.a_c0 = 0; j.a_c1 = r0 + j.m0; j.b_c0 = 0; j.b_c1 = j.n0; j.n_kb = kb_d;
      }
      run(j);
    }
    grid_barrier(a.barrier, bar_epoch);
    stamp(step, 1);
    if (a.chain != 0) {
      // ---- chained tail of the forward/backward pass per 128-row tile: four CTAs per M-tile, each
      // redoes fwd2 + xent (cheap) and owns a 64-column slice of dh
      if (t < mt_b * 4) {
        const int m0 = (t / 4) * kBM, slice = t % 4;
        const uint32_t par = chains & 1;
        if constexpr (EPI) {
          chain_epilogue<FP8>(a, smem, cb, tmem_base, q, half, lane, stg, sbias, xch, par, m0, r0, slice, sdbg);
        } else {
          if (warp == 0) chain_produce<FP8>(maps, a, smem, sf_smem, cb, m0, slice);
          else if (warp == 1) chain_mma<FP8>(smem, sf_smem, cb, tmem_base, par);
        }
        ++chains;
      }
      grid_barrier(a.barrier, bar_epoch);
      stamp(step, 2);
    } else {
      // ---- P2: logits -> dlogits / loss / db2
      if (t < mt_b) {
        Job j{};
        j.ta = &maps.h_k; j.tb = &maps.w2_k; j.a_mn = 0; j.b_mn = 0; j.bm = kBM;
        j.m0 = t * kBM; j.n0 = 0; j.M = B; j.N = C;
        j.a_c0 = 0; j.a_c1 = j.m0; j.b_c0 = 0; j.b_c1 = 0; j.n_kb = kb_h;
        j.mode = E_XENT; j.d = a.dlogits; j.ldd = a.ncp; j.bias = a.b2; j.colsum = a.gb2;
        j.labels = a.labels + r0; j.grad_scale = 1.f / static_cast<float>(B);
        run(j);
      }
      grid_barrier(a.barrier, bar_epoch);
      // ---- P3: dh = (dlogits W2) * relu'(h), db1
      if (t < mt_b * nt_h) {
        Job j{};
        j.ta = &maps.dl_k; j.tb = &maps.w2_mn; j.a_mn = 0; j.b_mn = 1; j.bm = kBM;
        j.m0 = (t / nt_h) * kBM; j.n0 = (t % nt_h) * kBN; j.M = B; j.N = H;
        j.a_c0 = 0; j.a_c1 = j.m0; j.b_c0 = j.n0; j.b_c1 = 0; j.n_kb = kb_c;
        j.mode = E_MASK_COLSUM_BF16; j.d = a.dh; j.ldd = H; j.aux = a.h; j.colsum = a.gb1;
        run(j);
      }
      grid_barrier(a.barrier, bar_epoch);
      stamp(step, 2);
    }
    // ---- B: dW1 = dh^T x (tiles [0, mt_hw*nt_d))  ||  dW2 = dlogits^T h (next nt_h tiles)  || biases
    if (t < mt_hw * nt_d) {
      Job j{};
      j.ta = &maps.dh_mn; j.tb = &maps.x_mn; j.a_mn = 1; j.b_mn = 1; j.bm = bm_w;
      j.m0 = (t / nt_d) * bm_w; j.n0 = (t % nt_d) * kBN; j.M = H; j.N = D;
      j.a_c0 = j.m0; j.a_c1 = 0; j.b_c0 = j.n0; j.b_c1 = r0; j.n_kb = kb_b;
      j.mode = eo ? E_OPT : E_F32; j.d = eo ? a.master + (a.gw1 - a.grad) : a.gw1; j.ldd = D;
      j.bc1 = bc1; j.bc2 = bc2; j.last = last ? 1 : 0;
      j.dbg = sdbg; j.dbg_slot = 18;
      j.q_off = a.ql.w1q; j.qsf_off = a.ql.w1sf; j.ldq = D; j.q_nkb = a.ql.kb1;
      run(j);
    } else if (t < mt_hw * nt_d + nt_h) {
      const int u = t - mt_hw * nt_d;
      Job j{};
      j.ta = &maps.dl_mn; j.tb = &maps.h_mn; j.a_mn = 1; j.b_mn = 1; j.bm = bm_w;
      j.m0 = 0; j.n0 = u * kBN; j.M = C; j.N = H;
      j.a_c0 = 0; j.a_c1 = 0; j.b_c0 = j.n0; j.b_c1 = 0; j.n_kb = kb_b;
      j.mode = eo ? E_OPT : E_F32; j.d = eo ? a.master + (a.gw2 - a.grad) : a.gw2; j.ldd = H;
      j.bc1 = bc1; j.bc2 = bc2; j.last = last ? 1 : 0;
      j.q_off = a.ql.w2q; j.qsf_off = a.ql.w2sf; j.ldq = H; j.q_nkb = a.ql.kb2;
      run(j);
    } else if (eo && t == mt_hw * nt_d + nt_h) {
      // biases: their gradients were accumulated by column sums earlier in the step; consume + re-zero
      const bool up = last && a.has_fed;
      UploadDst ud{};
      if (up) ud = upload_dst<FP8>(a);
      for (int i = threadIdx.x; i < H + C; i += blockDim.x) {
        float* gp = i < H ? a.gb1 + i : a.gb2 + (i - H);
        const float g = __ldcg(gp);
        *gp = 0.f;
        float w[4];
        const long long pi = gp - a.grad;
        opt_apply<PROX>(a, pi, 1, &g, bc1, bc2, w);
        if (up) {
          float wu = w[0];
          if (ud.global != nullptr) { const float g0 = __ldcg(ud.global + pi); wu = g0 - ud.byz_scale * (wu - g0); }
          ud.master[pi] = wu;
          if (!FP8) ud.shadow[pi] = __float2bfloat16(wu);
          else *reinterpret_cast<float*>(ud.blob + (i < H ? a.ql.b1 + 4 * i : a.ql.b2 + 4 * (i - H))) = wu;
        }
      }
    }
    stamp(step, 3);
    grid_barrier(a.barrier, bar_epoch, last && a.has_fed);
    stamp(step, 4);
    if (eo) continue;   // the optimizer ran in the epilogues
    // ---- P5: optimizer over the flat buffer (all threads of all CTAs)
    {
      const long long nv = a.n_params / 4;
      const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
      for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nv; i += stride) {
        const float4 g4 = __ldcg(reinterpret_cast<const float4*>(a.grad) + i);
        const float g[4] = {g4.x, g4.y, g4.z, g4.w};
        float w[4];
        opt_apply<PROX>(a, 4 * i, 4, g, bc1, bc2, w);
        reinterpret_cast<float4*>(a.grad)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    grid_barrier(a.barrier, bar_epoch);
    stamp(step, 5);
  }

  };   // round_loop
  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsLow));
    round_loop(std::false_type{});
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsHigh));
    round_loop(std::true_type{});
  }

  // ---- UploadLocalUpdate, second half: every CTA's upload stores were fenced at system scope
  // before the last barrier; CTA 0 pushes the meta record into every replica's ledger page and
  // raises FLAG_TRAINED on every peer (C:246-253).
  if (a.has_fed && a.epiopt && blockIdx.x == 0) {
    char* me = a.f.peers.base[a.f.rank];
    const RoundState* st = heap_at<const RoundState>(me, a.f.lay.state_off);
    RoundPlan* plan = heap_at<RoundPlan>(me, a.f.lay.plan_off);
    const uint32_t epoch = st->epoch;
    const uint32_t par = epoch & 1u;
    if (threadIdx.x == 0) atomicMax(&plan->t_stamp[STAMP_UPLOAD_BEGIN], globaltimer_ns());
    // first-K-wins admission (C:239-244): one ticket per trainer and round from the counter on
    // rank 0's page; a ticket beyond NEEDED_UPDATE_COUNT publishes nothing (update dropped)
    __shared__ int ticket;
    const bool fk = admit::first_k(st);
    if (threadIdx.x == 0) {
      admit::straggle(a.straggle_us);
      int tk = fk ? admit::take_ticket(&admit::page(a.f.peers.base[0], a.f.lay, par)->ticket, epoch) : 0;
      if (fk && tk >= static_cast<int>(st->n_needed)) tk = -1;
      ticket = tk;
    }
    __syncthreads();
    if (ticket >= 0 && threadIdx.x < a.f.n_ranks) {
      const int r = threadIdx.x;
      UploadMeta* meta = heap_at<UploadMeta>(a.f.peers.base[r], a.f.lay.meta_off) + par * kMaxRanks + a.f.rank;
      UploadMeta m;
      m.n_samples = static_cast<uint32_t>(a.n_samples);
      m.avg_cost = __ldcg(a.loss_sum) / static_cast<float>(a.n_loss_terms > 0 ? a.n_loss_terms : 1);
      *meta = m;
      __threadfence_system();
      if (fk)
        ptx::st_release_sys(&admit::page(a.f.peers.base[r], a.f.lay, par)->slot[ticket],
                            ((epoch + 1u) << 8) | static_cast<uint32_t>(a.f.rank));
      ptx::st_release_sys(heap_at<uint32_t>(a.f.peers.base[r], a.f.lay.flags_off) + FLAG_TRAINED + a.f.rank,
                          epoch + 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) atomicMax(&plan->t_stamp[STAMP_UPLOAD_END], globaltimer_ns());
  }

  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

Mx8MlpLayout mx8_mlp_layout(int in_dim, int hidden) {
  Mx8MlpLayout l;
  l.kb1 = (in_dim + 127) / 128;
  l.kb2 = (hidden + 127) / 128;
  const int rb1 = (hidden + 127) / 128;
  int cur = 0;
  auto take = [&](int bytes) { const int o = cur; cur += (bytes + 127) / 128 * 128; return o; };
  l.w1q = take(hidden * in_dim);
  l.w1sf = take(rb1 * l.kb1 * kSfChunk);
  l.w2q = take(64 * hidden);
  l.w2sf = take(l.kb2 * kSfChunk);
  l.b1 = take(hidden * 4);
  l.b2 = take(64 * 4);
  l.total = cur;
  return l;
}

cudaError_t mlp_round_sm100(const MlpRoundArgs& r, cudaStream_t stream) {
  bind_context_once();
  if (r.hidden % 8 || r.in_dim % 8 || r.n_params % 4 || r.batch % 8 || r.ncp % 8 || r.n_classes > 64)
    return cudaErrorInvalidValue;
  const int mt_b = (r.batch + kBM - 1) / kBM, nt_h = (r.hidden + kBN - 1) / kBN;
  const int nt_d = (r.in_dim + kBN - 1) / kBN;
  // phase plan: r.plan / r.epiopt when >= 0, else BFLC_MLP_CHAIN = 0 | 3 and BFLC_MLP_EPIOPT = 0 | 1
  // (see the kernel), else the defaults
  static const int chain_env0 = [] { const char* e = std::getenv("BFLC_MLP_CHAIN"); return e ? std::atoi(e) : kDefaultPlan; }();
  static const bool epiopt_env0 = [] { const char* e = std::getenv("BFLC_MLP_EPIOPT"); return !(e && e[0] == '0'); }();
  const int chain_env = r.plan >= 0 ? r.plan : chain_env0;
  const bool epiopt = r.epiopt >= 0 ? r.epiopt != 0 : epiopt_env0;
  const bool chain_ok = r.hidden == kChainH && r.ncp == 64 && r.n_classes <= 64;
  const int chain = (!chain_ok || chain_env == 0) ? 0 : 3;
  const bool fp8 = r.fp8;
  if (fp8 && (chain != 3 || !epiopt || r.batch % 128 || r.in_dim % 16 || !r.x_q || !r.x_sf || !r.work_q ||
              !r.h_q || !r.h_sf))
    return cudaErrorNotSupported;
  if (r.fed != nullptr && !epiopt) return cudaErrorNotSupported;
  // FedProx needs its anchor; it is not combined with the fused upload (one client per GPU)
  if (!(r.prox_mu >= 0.f) || (r.prox_mu > 0.f && (r.prox_anchor == nullptr || r.fed != nullptr)))
    return cudaErrorInvalidValue;
  const bool prox = r.prox_mu > 0.f;
  // weight-gradient tiles: 64 rows (UMMA M = 64) spread the optimizer epilogue over twice the CTAs;
  // BFLC_MLP_BMW=128 keeps the 128-row tiles
  static const int bmw_env = [] { const char* e = std::getenv("BFLC_MLP_BMW"); return e && std::atoi(e) == 128 ? 128 : 64; }();
  int bm_w = bmw_env;
  int mt_hw = (r.hidden + bm_w - 1) / bm_w;
  if (mt_hw * nt_d + nt_h + 1 > 148) { bm_w = 128; mt_hw = (r.hidden + 127) / 128; }
  const int need = std::max(std::max(mt_b * nt_h, mt_hw * nt_d + nt_h + 1), chain == 3 ? mt_b * 4 : 0);
  const int grid = need > kGrid ? need : kGrid;
  if (grid > 148) return cudaErrorInvalidValue;

  Maps m;
  std::memset(&m, 0, sizeof(m));
  const long long rows_x = static_cast<long long>(r.steps) * r.batch;
  auto mk = [&](CUtensorMap* out, const void* ptr, long long ld, bool mn, int rows_extent, int K,
                int rows_tile, DType dt = DType::BF16) {
    GemmOperand op{ptr, ld, 0, mn};
    return gemm_make_operand_map(out, op, dt, rows_extent, K, 1, rows_tile);
  };
  cudaError_t e;
  // K-major: (rows_extent = M|N, K);  MN-major: memory [K][M|N]
  if ((e = mk(&m.x_k, r.x, r.in_dim, false, (int)rows_x, r.in_dim, kBM)) != cudaSuccess) return e;
  if ((e = mk(&m.w1_k, r.w1_shadow, r.in_dim, false, r.hidden, r.in_dim, kBN)) != cudaSuccess) return e;
  if ((e = mk(&m.h_k, r.h, r.hidden, false, r.batch, r.hidden, kBM)) != cudaSuccess) return e;
  if ((e = mk(&m.w2_k, r.w2_shadow, r.hidden, false, r.n_classes, r.hidden, kBN)) != cudaSuccess) return e;
  if ((e = mk(&m.dl_mn, r.dlogits, r.ncp, true, r.n_classes, r.batch, kBM)) != cudaSuccess) return e;
  if ((e = mk(&m.h_mn, r.h, r.hidden, true, r.hidden, r.batch, kBN)) != cudaSuccess) return e;
  if ((e = mk(&m.dl_k, r.dlogits, r.ncp, false, r.batch, r.n_classes, kBM)) != cudaSuccess) return e;
  if ((e = mk(&m.w2_mn, r.w2_shadow, r.hidden, true, r.hidden, r.n_classes, kBN)) != cudaSuccess) return e;
  if ((e = mk(&m.dh_mn, r.dh, r.hidden, true, r.hidden, r.batch, kBM)) != cudaSuccess) return e;
  if ((e = mk(&m.x_mn, r.x, r.in_dim, true, r.in_dim, (int)rows_x, kBN)) != cudaSuccess) return e;
  const Mx8MlpLayout ql = mx8_mlp_layout(r.in_dim, r.hidden);
  if (fp8) {
    const DType q = DType::FP8_E4M3;
    if ((e = mk(&m.xq_k, r.x_q, r.in_dim, false, (int)rows_x, r.in_dim, kBM, q)) != cudaSuccess) return e;
    if ((e = mk(&m.w1q_k, r.work_q + ql.w1q, r.in_dim, false, r.hidden, r.in_dim, kBN, q)) != cudaSuccess) return e;
    if ((e = mk(&m.hq_k, r.h_q, r.hidden, false, r.batch, r.hidden, kBM, q)) != cudaSuccess) return e;
    if ((e = mk(&m.w2q_k, r.work_q + ql.w2q, r.hidden, false, 64, r.hidden, 64, q)) != cudaSuccess) return e;
  }

  Args a{};
  a.B = r.batch; a.steps = r.steps; a.in_dim = r.in_dim; a.hidden = r.hidden;
  a.n_classes = r.n_classes; a.ncp = r.ncp; a.n_params = r.n_params;
  a.chain = chain; a.epiopt = epiopt ? 1 : 0; a.dbg = r.dbg;
  a.x_ready = r.x_ready; a.round_seq = r.round_seq;
  a.pred = r.pred ? r.pred : current_predicate();
  a.barrier = r.barrier;
  a.master = r.master; a.b1 = r.b1; a.b2 = r.b2;
  a.grad = r.grad; a.gw1 = r.gw1; a.gb1 = r.gb1; a.gw2 = r.gw2; a.gb2 = r.gb2;
  a.shadow = reinterpret_cast<__nv_bfloat16*>(r.shadow);
  a.adam_m = r.adam_m; a.adam_v = r.adam_v; a.adam = r.adam ? 1 : 0;
  a.lr = r.lr; a.beta1 = r.beta1; a.beta2 = r.beta2; a.eps = r.eps; a.step_base = r.step_base;
  a.h = reinterpret_cast<__nv_bfloat16*>(r.h);
  a.dlogits = reinterpret_cast<__nv_bfloat16*>(r.dlogits);
  a.dh = reinterpret_cast<__nv_bfloat16*>(r.dh);
  a.labels = r.labels; a.loss_sum = r.loss_sum; a.correct = r.correct;
  a.x_sf = r.x_sf; a.work_q = r.work_q; a.h_q = r.h_q; a.h_sf = r.h_sf; a.ql = ql; a.bm_w = bm_w;
  a.has_fed = r.fed != nullptr ? 1 : 0;
  if (r.fed != nullptr) a.f = *r.fed;
  a.upq_off[0] = r.upq_off[0]; a.upq_off[1] = r.upq_off[1];
  a.n_samples = r.n_samples; a.n_loss_terms = r.n_loss_terms; a.byz_mode = r.byz_mode; a.byz_scale = r.byz_scale;
  a.straggle_us = r.straggle_us;
  a.prox_anchor = prox ? r.prox_anchor : nullptr; a.prox_mu = prox ? r.prox_mu : 0.f;

  auto kern = fp8 ? (prox ? mlp_round_kernel<true, true> : mlp_round_kernel<true, false>)
                  : (prox ? mlp_round_kernel<false, true> : mlp_round_kernel<false, false>);
  static bool configured[4] = {false, false, false, false};
  const int ki = (fp8 ? 1 : 0) + (prox ? 2 : 0);
  if (!configured[ki]) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal);
    if (e != cudaSuccess) return e;
    configured[ki] = true;
  }
  note_launch();
  return launch_pdl(kern, dim3(grid), dim3(kThreads), kSmemTotal, stream, m, a);
}

}  // namespace bflc
