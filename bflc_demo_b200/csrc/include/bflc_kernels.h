// Host-callable C++ API of the sm_100a kernel library (no torch dependency).
// All launchers are asynchronous on `stream`.
//
// Parity map (reference = iammcy/BFLC-demo, CPU-only TensorFlow + C++ contract):
//   gemm / linear       <- K1  x@W+b                 python-sdk/main.py:120,180,293
//   xent epilogue       <- K2  softmax-xent mean     python-sdk/main.py:123
//   backward + SGD/Adam <- K3  autodiff + optimizer  python-sdk/main.py:126-130
//   accuracy epilogue   <- K6  argmax==argmax mean   python-sdk/main.py:182-183
//   consensus kernel    <- K7-K10 median/top-K/FedAvg/apply
//                              CommitteePrecompiled.cpp:349-456
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace bflc {

enum class DType : int { F32 = 0, BF16 = 1, FP8_E4M3 = 2, U8 = 3 };
enum class Act : int { NONE = 0, RELU = 1, GELU = 2 };
enum class EpiKind : int { GENERIC = 0, XENT = 1, ARGMAX_ACC = 2 };

// D[b] (M x N) = alpha * A[b] (M x K) * B[b]^T (N x K)
//   K-major operand : memory is [rows = M|N][K], K contiguous
//   MN-major operand: memory is [K][M|N], M|N contiguous
struct GemmOperand {
  const void* ptr = nullptr;
  int64_t ld = 0;            // row stride in elements
  int64_t batch_stride = 0;  // in elements; 0 = shared across the batch
  bool mn_major = false;
};

struct GemmEpilogue {
  EpiKind kind = EpiKind::GENERIC;
  // ---- generic ----
  void* d = nullptr;  // output [batch][M][ldd]
  DType d_dtype = DType::BF16;
  int64_t ldd = 0;
  int64_t d_batch_stride = 0;
  float alpha = 1.f;
  const float* bias = nullptr;              // [N] fp32, per output column
  const float* const* bias_ptrs = nullptr;  // optional per-batch bias pointers (device array)
  Act act = Act::NONE;
  void* aux_out = nullptr;       // bf16 pre-activation copy (GELU backward needs it)
  const void* aux_in = nullptr;  // bf16 [M][ldd]: act-backward mask source
  int act_bwd = 0;               // 1: out *= (aux_in > 0)  2: out *= gelu'(aux_in)
  float* colsum = nullptr;       // [N] fp32 += column sums of the stored values (bias grad)
  int split_k = 1;               // >1: fp32 atomic accumulate into a zeroed d
  int accumulate = 0;            // 1: d += result (fp32 d only, non-atomic)
  // ---- xent / accuracy (row-wise over the N <= BN logits of a row) ----
  const int32_t* labels = nullptr;  // [batch][M]
  int64_t labels_batch_stride = 0;
  float grad_scale = 1.f;         // dlogits = (softmax - onehot) * grad_scale
  float* loss_sum = nullptr;      // += sum_rows (lse - z_label)
  unsigned int* correct = nullptr;  // [batch] += #(argmax == label)
};

// Implicit-GEMM convolution: one operand is an NHWC bf16 activation read through a 4-D tensor
// map, so the im2col matrix is never written.  Each K block (mode 1) or N tile (mode 2) is one
// filter tap (r, s) x 64 channels, fetched as a TMA box shifted by the tap offset; boxes that
// hang over the image border are zero-filled by the TMA unit (= the padding).
//   mode 1, flip 0  forward        : A = x  [N,H,W,C]    rows = output pixels, B = w [Cout][KH*KW*C]
//   mode 1, flip 1  input gradient : A = dy [N,OH,OW,C]  rows = input pixels (stride 1 only),
//                                    B = w read MN-major, tap-mirrored
//   mode 2          weight gradient: B = x shifted per tap, reduction over output pixels,
//                                    A = dy [pixels][Cout] MN-major, D = dW [Cout][KH*KW*C]
struct ConvView {
  int mode = 0;
  int flip = 0;
  const void* x = nullptr;  // the NHWC activation
  int N = 0, H = 0, W = 0, C = 0;   // its dims
  int OH = 0, OW = 0;               // pixel grid the GEMM rows / reduction enumerate
  int KH = 1, KW = 1, stride = 1, pad = 0;
};

struct GemmDynamic;  // device-resident per-launch arguments, defined below

struct GemmProblem {
  int M = 0, N = 0, K = 0, batch = 1;
  DType ab_dtype = DType::BF16;
  GemmOperand a, b;
  // optional: per-batch B tensor maps living in device memory (grouped GEMM whose
  // B operands are in *different allocations*, e.g. peer GPUs' weights)
  const CUtensorMap* b_maps_dev = nullptr;
  // optional: batch count / map selection / bias / readiness flags read from device memory
  const GemmDynamic* dyn = nullptr;
  GemmEpilogue epi;
  // debug overrides for descriptor bring-up (0 = use built-in)
  uint32_t dbg_lbo_a = 0, dbg_sbo_a = 0, dbg_lbo_b = 0, dbg_sbo_b = 0;
  int force_bn = 0;  // 0 = heuristic; 64/128/256 pins the N-tile (must match pre-built b maps)
  ConvView conv;     // mode != 0: the A (mode 1) or B (mode 2) operand is an implicit im2col view
};

// cuTensorMapEncodeTiled is a driver call and needs a context current on the calling thread;
// worker threads (e.g. PyTorch's autograd thread) may never have bound the primary context
// (observed: CUDA_ERROR_INVALID_CONTEXT).  Bind it once per thread with cudaSetDevice (legal while
// a stream capture is active -- cudaFree(nullptr), the usual idiom, invalidates the capture when
// a thread makes its first GEMM call inside one, e.g. autograd's worker during graph capture).
inline void bind_context_once() {
  static thread_local bool bound = false;
  if (!bound) {
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) (void)cudaSetDevice(dev);
    bound = true;
  }
}

// returns cudaSuccess or the failing status; throws nothing
cudaError_t gemm_sm100(const GemmProblem& p, cudaStream_t stream);
// 2-CTA variant (cta_group::2, 256x256 tiles per CTA pair): bf16, K-major operands, generic
// bias/activation epilogue only; returns cudaErrorNotSupported for anything else.
cudaError_t gemm2_sm100(const GemmProblem& p, cudaStream_t stream);
// Block-scaled fp8 (MXFP8: e4m3 + one UE8M0 scale per 32 K-elements), K-major A [M,K] and
// B [N,K]; sfa/sfb are the chunk arrays written by quantize_mx8 (csrc/kernels/gemm_mx8_sm100.cu).
struct Mx8Problem {
  int M = 0, N = 0, K = 0;
  const void* a = nullptr; long long lda = 0; const uint8_t* sfa = nullptr;
  const void* b = nullptr; long long ldb = 0; const uint8_t* sfb = nullptr;
  void* d = nullptr; DType d_dtype = DType::BF16; long long ldd = 0;
  float alpha = 1.f; const float* bias = nullptr; Act act = Act::NONE;
};
cudaError_t gemm_mx8_sm100(const Mx8Problem& p, cudaStream_t stream);
// bytes of the scale-factor chunk array for a [rows, K] operand
long long mx8_sf_bytes(int rows, int K);
// x [R, K] (f32 / bf16 / u8, row pitch ldx elements) * in_scale -> q e4m3 [R, ldq] + scale chunks
cudaError_t quantize_mx8(const void* x, DType x_dtype, long long ldx, int R, int K, float in_scale,
                         void* q, long long ldq, void* sf, cudaStream_t stream);
// Build the B-operand tensor map the kernel would use (for b_maps_dev arrays).
cudaError_t gemm_make_b_map(const GemmProblem& p, CUtensorMap* out_host);
// Encode the TMA descriptor of one GEMM operand (rows_tile = 128 for A, the N-tile for B).
cudaError_t gemm_make_operand_map(CUtensorMap* out, const GemmOperand& op, DType dt,
                                  int rows_extent, int K, int batch, int rows_tile);

struct FedArgs;  // symmetric-heap addressing of the federated kernels, defined below

// Byte layout of a "quantised model blob" of the 2-layer MLP: what a trainer publishes for the
// committee in fp8 mode and what the persistent trainer keeps as its own MXFP8 compute copy.
//   w1q  e4m3 [hidden][in_dim]      w1sf  scale chunks [hidden/128][kb1][512]
//   w2q  e4m3 [64][hidden]          w2sf  scale chunks [1][kb2][512]      (classes padded to 64)
//   b1   fp32 [hidden]              b2    fp32 [64]
struct Mx8MlpLayout {
  int w1q = 0, w1sf = 0, w2q = 0, w2sf = 0, b1 = 0, b2 = 0, total = 0;
  int kb1 = 0, kb2 = 0;   // K-blocks (128 elements) along in_dim / hidden
};
Mx8MlpLayout mx8_mlp_layout(int in_dim, int hidden);

// Whole local-training pass of the 2-layer MLP in ONE persistent kernel (mlp_round_sm100.cu).
struct MlpRoundArgs {
  int batch = 0, steps = 0, in_dim = 0, hidden = 0, n_classes = 0, ncp = 0;
  long long n_params = 0;
  const void* x = nullptr;            // bf16 [steps*batch][in_dim]
  const int32_t* labels = nullptr;    // [steps*batch]
  float* master = nullptr;            // flat fp32 parameters (w1 | b1 | w2 | b2, 8-aligned)
  void* shadow = nullptr;             // flat bf16 copy
  float* grad = nullptr;              // flat fp32 gradients (zeroed; left zeroed)
  const void* w1_shadow = nullptr; const void* w2_shadow = nullptr;
  const float* b1 = nullptr; const float* b2 = nullptr;
  float* gw1 = nullptr; float* gb1 = nullptr; float* gw2 = nullptr; float* gb2 = nullptr;
  void* h = nullptr; void* dlogits = nullptr; void* dh = nullptr;   // bf16 scratch
  float* loss_sum = nullptr; unsigned int* correct = nullptr;
  unsigned int* barrier = nullptr;    // zero before launch
  const int* pred = nullptr;          // null -> thread-local predicate
  bool adam = false; float* adam_m = nullptr; float* adam_v = nullptr;
  float lr = 1e-3f, beta1 = 0.9f, beta2 = 0.999f, eps = 1e-8f;
  const int* step_base = nullptr;
  unsigned long long* dbg = nullptr;  // optional [steps][32] %globaltimer stamps (CTA 0)
  // optional input pipeline: producer of step s waits until x_ready[s] >= *round_seq
  const unsigned int* x_ready = nullptr; const unsigned int* round_seq = nullptr;
  int plan = -1;     // phase plan override: 0 | 1 | 3 (see mlp_round_sm100.cu); -1 = env / default
  int epiopt = -1;   // optimizer in the weight-gradient epilogues: 0 | 1; -1 = env / default
  // ---- block-scaled fp8 forward (fwd1 and fwd2 as tcgen05.mma.kind::mxf8f6f4.block_scale;
  //      the weight/hidden gradients stay bf16).  Needs plan 3 + epiopt, hidden == 256.
  bool fp8 = false;
  const void* x_q = nullptr;          // e4m3 [steps*batch][in_dim]  (quantize_inputs_mx8)
  const uint8_t* x_sf = nullptr;      // its scale chunks
  uint8_t* work_q = nullptr;          // Mx8MlpLayout blob: this trainer's quantised weights,
                                      // refreshed by the optimizer epilogue every step
  uint8_t* h_q = nullptr; uint8_t* h_sf = nullptr;   // scratch: e4m3 [batch][hidden] + chunks
  // ---- fused UploadLocalUpdate (needs epiopt): the optimizer epilogue of the LAST step also
  //      writes the peer-readable upload buffers (fp32 master + bf16 shadow, or the fp8 blob at
  //      heap offset upq_off[parity]); CTA 0 then pushes {n_samples, avg_cost} into every
  //      replica and releases FLAG_TRAINED on every peer.  Replaces fed_upload.
  const FedArgs* fed = nullptr;
  long long upq_off[2] = {0, 0};
  int n_samples = 0, n_loss_terms = 0, byz_mode = 0;
  float byz_scale = 0.f;
  int straggle_us = 0;   // fault injection: publish this late (first-K-wins admission test)
  // ---- FedProx: every optimizer update uses g' = fmaf(prox_mu, w - anchor, g), w = the master
  //      before that update.  The anchor is the fp32 global model at round start (the layout of
  //      `master`).  prox_mu > 0 needs an anchor and no fused upload (else cudaErrorInvalidValue);
  //      the reported loss stays the cross-entropy alone.
  const float* prox_anchor = nullptr;
  float prox_mu = 0.f;
};
cudaError_t mlp_round_sm100(const MlpRoundArgs& r, cudaStream_t stream);

// Committee validation of up to max_cand candidates in one launch (hidden == 256, classes <= 64):
// per (128 rows, candidate) CTA  relu(x W1_z^T + b1_z) W2_z^T + b2_z -> argmax == label -> correct[z].
// `maps` is the device tensor-map table the round plan indexes (layer-1 maps encoded with a
// 256-row box, layer-2 maps with a 64-row box); dyn1/dyn2 are the plan's per-layer GemmDynamic.
struct GemmDynamic;
struct MlpValArgs {
  int n_val = 0, in_dim = 0, hidden = 0, n_classes = 0, max_cand = 0;
  const void* x = nullptr; long long ldx = 0;     // bf16 [n_val][in_dim]  (fp8: e4m3, ldx = in_dim)
  const CUtensorMap* maps = nullptr;
  const GemmDynamic* dyn1 = nullptr; const GemmDynamic* dyn2 = nullptr;
  const int32_t* labels = nullptr; unsigned int* correct = nullptr;
  const int* pred = nullptr;
  // fp8: candidates are Mx8MlpLayout blobs (their addresses come from the round plan's
  // cand_blob[]); x_sf = scale chunks of x
  bool fp8 = false;
  const uint8_t* x_sf = nullptr;
  const uint8_t* const* cand_blob = nullptr;   // device array [max_cand]
  // fused gather ("QueryAllUpdates" inside the validation kernel): when cand_src is set, the
  // CTAs of candidate z first copy z's blob out of the trainer's HBM (cand_src[z], P2P loads,
  // 1/gridDim.x each) into the local slot cand_blob[z], meet on pull_cnt[z], then validate from
  // the local copy -- no separate pull kernel.  Needs gridDim.x <= 128 (co-residency).
  const uint8_t* const* cand_src = nullptr;    // device array [max_cand] (RoundPlan::cand_src)
  unsigned int* pull_cnt = nullptr;            // device array [max_cand], zeroed by the plan kernel
  long long blob_bytes = 0;
  unsigned long long* stamps = nullptr;        // optional RoundPlan::t_stamp (pull begin / end)
};
cudaError_t mlp_val_sm100(const MlpValArgs& r, cudaStream_t stream);

// x u8 [R][K] (pixels) -> bf16 [R][K] (x * scale), e4m3 [R][K] and MXFP8 scale chunks in one pass
// (K % 16 == 0).  Any of dst_bf16 / dst_q may be null.
cudaError_t prep_inputs_u8(const uint8_t* src, void* dst_bf16, void* dst_q, uint8_t* dst_sf, int R,
                           int K, float scale, cudaStream_t s);
// chunked, tag-driven variant for the host->device input pipeline (see k_prep_chunks)
cudaError_t prep_inputs_u8_chunks(const uint8_t* src, void* dst_bf16, void* dst_q, uint8_t* dst_sf,
                                  int rows_per_chunk, int K, int n_chunks, float scale,
                                  const int* in_flags, const int* in_seq, unsigned int* cnt,
                                  unsigned int* ready, unsigned int* err, cudaStream_t s);
// fp32 master weights of the MLP -> Mx8MlpLayout blob (start of a round: the consensus kernel
// has just written the new global model into the training buffers)
cudaError_t quantize_mlp_blob(const float* master, long long off_w1, long long off_b1,
                              long long off_w2, long long off_b2, int in_dim, int hidden,
                              int n_classes, uint8_t* blob, cudaStream_t s);

// N-tile width the launcher would choose for a problem (z = batch * split_k)
int gemm_pick_bn(int N, EpiKind kind, int M, int z);
// number of kernels launched by this library since process start (bench bookkeeping)
unsigned long long launch_count();
void note_launch();

// ---------------------------------------------------------------- elementwise
cudaError_t cast_f32_to_bf16(const float* src, void* dst, int64_t n, cudaStream_t s);
cudaError_t cast_bf16_to_f32(const void* src, float* dst, int64_t n, cudaStream_t s);
cudaError_t cast_u8_to_bf16(const uint8_t* src, void* dst, int64_t n, float scale, cudaStream_t s);
cudaError_t quantize_fp8(const void* src_bf16, uint8_t* dst, int64_t n, float inv_scale,
                         cudaStream_t s);
cudaError_t amax_bf16(const void* src, int64_t n, float* amax_out, cudaStream_t s);
cudaError_t fill_f32(float* dst, int64_t n, float v, cudaStream_t s);

// ------------------------------------------------------------------ optimizers
// Flat multi-tensor update. master fp32 is updated in place; shadow (bf16,
// optional fp8 second shadow) is the compute copy the GEMMs read.  `active` (device
// flag, may be null) lets a captured graph skip the update on non-trainer ranks.
struct OptimArgs {
  float* master = nullptr;
  const float* grad = nullptr;
  void* shadow_bf16 = nullptr;
  int64_t n = 0;
  float lr = 1e-3f, weight_decay = 0.f;
  // adam
  float* m = nullptr;
  float* v = nullptr;
  float beta1 = 0.9f, beta2 = 0.999f, eps = 1e-8f;
  const int* step_dev = nullptr;  // device base step (steps before this round), may be null
  int step = 1;                   // Adam t = (step_dev ? *step_dev : 0) + step
  const int* active = nullptr;
  int zero_grad = 1;  // clear grad after use (it is an accumulation target)
};
cudaError_t sgd_step(const OptimArgs& a, cudaStream_t s);
cudaError_t adam_step(const OptimArgs& a, cudaStream_t s);

// ------------------------------------------------------- NN support kernels
cudaError_t im2col_bf16(const void* x, void* col, int N, int C, int H, int W, int KH, int KW,
                        int stride, int pad, int OH, int OW, int64_t ld_col, cudaStream_t s);
// up[n, s*oh, s*ow, :] = dy[n, oh, ow, :], zeros elsewhere (strided-convolution input gradient)
cudaError_t upsample_zero_bf16(const void* dy, void* up, int N, int H, int W, int OH, int OW, int C,
                               int stride, cudaStream_t s);
cudaError_t col2im_bf16(const void* col, void* dx, int N, int C, int H, int W, int KH, int KW,
                        int stride, int pad, int OH, int OW, int64_t ld_col, cudaStream_t s);
cudaError_t maxpool2d_fwd(const void* x, void* y, int32_t* idx, int N, int C, int H, int W, int k,
                          int stride, int pad, int OH, int OW, cudaStream_t s);
cudaError_t maxpool2d_bwd(const void* dy, const int32_t* idx, float* dx_f32, int64_t n_out,
                          int64_t per_out, int64_t per_in, cudaStream_t s);
cudaError_t avgpool_global_fwd(const void* x, void* y, int N, int HW, int C, cudaStream_t s);
cudaError_t avgpool_global_bwd(const void* dy, void* dx, int N, int HW, int C, cudaStream_t s);
// channels-last batch norm over [rows][C]; train mode computes batch statistics
cudaError_t batchnorm_fwd(const void* x, void* y, const float* gamma, const float* beta,
                          float* mean, float* rstd, float* run_mean, float* run_var,
                          int64_t rows, int C, float eps, float momentum, int training, int relu,
                          const void* residual, cudaStream_t s);
cudaError_t batchnorm_bwd(const void* dy, const void* x, const void* y, const float* gamma,
                          const float* mean, const float* rstd, void* dx, float* dgamma,
                          float* dbeta, void* dresidual, int64_t rows, int C, int relu,
                          cudaStream_t s);
cudaError_t layernorm_fwd(const void* x, const void* residual, void* y, const float* gamma,
                          const float* beta, float* mean, float* rstd, int64_t rows, int C,
                          float eps, cudaStream_t s);
cudaError_t layernorm_bwd(const void* dy, const void* xin, const float* gamma, const float* mean,
                          const float* rstd, void* dx, float* dgamma, float* dbeta, int64_t rows,
                          int C, cudaStream_t s);
cudaError_t softmax_rows_fwd(const void* x, void* y, int64_t rows, int cols, float scale,
                             cudaStream_t s);
cudaError_t softmax_rows_bwd(const void* dy, const void* y, void* dx, int64_t rows, int cols,
                             float scale, cudaStream_t s);
cudaError_t embedding_fwd(const int32_t* ids, const void* table_bf16, const void* pos_bf16,
                          void* out, int64_t rows, int seq, int C, cudaStream_t s);
cudaError_t embedding_bwd(const int32_t* ids, const void* dy, float* dtable, float* dpos,
                          int64_t rows, int seq, int C, cudaStream_t s);
cudaError_t add_bf16(const void* a, const void* b, void* out, int64_t n, cudaStream_t s);
// dz = dy * act'(aux), colsum += column sums of dz (bias gradient); mode 0 none, 1 ReLU, 2 GELU
cudaError_t act_bwd_colsum(const void* dy, const void* aux, void* dz, float* colsum, int64_t rows,
                           int C, int mode, cudaStream_t s);
// Fused multi-head self-attention, seq_len 128 / head_dim 64 (attn_sm100.cu): q, k, v, o and the
// gradients are [B*S, ld] bf16 matrices with head h in columns [h*64, h*64+64); lse is fp32
// [B*H*S] (row log-sum-exp, saved by the forward for the backward).
cudaError_t attention_fwd_sm100(const void* q, const void* k, const void* v, void* o, float* lse, int B,
                                int S, int H, int D, long long ld, float scale, cudaStream_t stream);
cudaError_t attention_bwd_sm100(const void* q, const void* k, const void* v, const void* o,
                                const void* dout, const float* lse, void* dq, void* dk, void* dv, int B,
                                int S, int H, int D, long long ld, float scale, cudaStream_t stream);
cudaError_t transpose_0213_bf16(const void* x, void* y, int d0, int d1, int d2, int d3,
                                cudaStream_t s);

// -------------------------------------------------- federated hot-path kernels
constexpr int kMaxRanks = 8;
constexpr int kMaxPlanLayers = 4;

// Per-launch dynamic GEMM arguments that live in device memory so one captured CUDA graph
// serves every round even though committee membership changes ("roles as data").
struct GemmDynamic {
  int active_batches;                     // CTAs with batch index >= this exit immediately
  int map_index[kMaxRanks];               // b_maps_dev[map_index[b]] is batch b's B operand
  const float* bias[kMaxRanks];           // per-batch bias (may point into a peer's HBM)
  const uint32_t* wait_flag[kMaxRanks];   // producer waits *wait_flag[b] >= wait_value first
  uint32_t wait_value;
};

// Device-resident round state ("the ledger page"): one replica per rank inside its symmetric
// heap, kept identical on all ranks by the consensus kernel.
struct RoundState {
  uint32_t epoch;                 // current federated round
  uint32_t n_ranks, n_comm, n_aggregate;
  uint32_t role[kMaxRanks];       // RoleBits (consensus_math.hpp)
  float last_median[kMaxRanks];
  uint32_t selected_mask;
  float global_loss;
  unsigned long long model_digest;
  uint32_t blocks_appended;
  uint32_t n_needed;              // NEEDED_UPDATE_COUNT: updates admitted per round.  == #trainers:
                                  // every trainer is awaited; < #trainers: first-K-wins (C:239-244)
};

struct UploadMeta {
  uint32_t n_samples;
  float avg_cost;
};

// Scratch written by the plan kernel at the start of every round (local, not replicated).
struct RoundPlan {
  int is_trainer;                 // predicate flags consumed by captured kernels
  int is_comm;
  int n_cand;
  int cand_rank[kMaxRanks];       // trainer rank of candidate slot z
  uint32_t parity;
  GemmDynamic dyn[kMaxPlanLayers];
  const uint8_t* cand_blob[kMaxRanks];  // fp8 MLP: candidate z's Mx8MlpLayout blob (staging slot or peer)
  const uint8_t* cand_src[kMaxRanks];   // fused gather: the trainer's upload blob the slot is filled from
  unsigned int pull_cnt[kMaxRanks];     // fused gather: CTAs of candidate z that finished their share
  unsigned int correct[kMaxRanks];  // validation hits per candidate slot (accuracy epilogue)
  float loss_sum;                   // local-training loss accumulator (xent epilogue)
  unsigned int train_correct;
  int opt_step;                     // optimizer steps completed before this round (Adam t base)
  int opt_total;                    // running total, advanced by the plan kernel on trainer ranks
  unsigned int upload_blocks_done;
  unsigned int consensus_blocks_done;
  unsigned long long digest_acc;
  unsigned int step_barrier;         // phase barrier of the persistent training kernel (zeroed per round)
  unsigned int round_seq;            // rounds planned so far on this rank (k_plan increments; never reset)
  // %globaltimer (ns) phase stamps of the current round, see StampSlot
  unsigned long long t_stamp[8];
};

enum StampSlot : int {
  STAMP_PLAN = 0,          // k_plan start
  STAMP_UPLOAD_BEGIN = 1,  // local training finished, k_upload running
  STAMP_UPLOAD_END = 2,    // flags released on every peer
  STAMP_PULL_BEGIN = 3,    // committee: k_pull running (waits on trainers' flags)
  STAMP_PULL_END = 4,      // last pull block done -> validation GEMMs may start
  STAMP_CONS_BEGIN = 5,    // validation finished, k_consensus running
  STAMP_CONS_SCORED = 6,   // all committee score rows + uploads visible
  STAMP_CONS_END = 7,      // new global model published, FLAG_DONE released
};

struct PeerTable {
  char* base[kMaxRanks];  // peer-mapped base pointer of each rank's symmetric heap
  char* mc_base;          // NVLS multicast VA of the same heap (null if unavailable)
};

// Byte offsets of the regions inside every rank's symmetric heap (identical on all ranks).
struct HeapLayout {
  long long flags_off;         // uint32 [FLAG_COUNT]
  long long state_off;         // RoundState
  long long plan_off;          // RoundPlan
  long long scores_off;        // float [2 parity][kMaxRanks committee][kMaxRanks trainer]
  long long meta_off;          // UploadMeta [2 parity][kMaxRanks]
  long long work_master_off;   // fp32 training weights (torch parameters alias this)
  long long work_shadow_off;   // bf16 copy the GEMMs read
  long long upload_master_off[2];  // fp32 uploaded local model, by epoch parity
  long long upload_shadow_off[2];  // bf16 of the same (what the committee validates)
  long long global_off;        // fp32 global model replica
  long long global_shadow_off; // bf16
  long long ring_off;          // BlockRecord [ring_slots]
  long long n_params;          // elements (multiple of 8)
  long long admit_off;         // AdmitPage [2 parity]: first-K-wins admission (ticket + slots)
  int ring_slots;
  int pad;
};

// First-K-wins admission (reference: UploadLocalUpdate drops an update once update_count reached
// NEEDED_UPDATE_COUNT, C:239-244 -- there the order is the chain's transaction order; here it is
// the order of an atomic ticket counter on rank 0's page).  A trainer that finished its local
// pass takes a ticket; tickets 0..K-1 are admitted: the trainer writes (epoch+1)<<8 | rank into
// slot[ticket] of EVERY replica with a release store issued after its upload is visible, so a
// reader that acquires a slot may read that trainer's upload.  Later tickets are rejected: the
// trainer publishes nothing and its update is ignored, exactly like a dropped transaction.
struct AdmitPage {
  uint32_t ticket;                 // (epoch+1)<<8 | tickets handed out; only rank 0's copy is used
  uint32_t slot[kMaxRanks];        // candidate slot z -> (epoch+1)<<8 | trainer rank
  uint32_t pad[7];
};

// One record per finished round, written by the consensus kernel and drained by the host
// C++ ledger, which re-executes the election from the raw score rows (state-machine
// replication check) and chains the block hash.
struct BlockRecord {
  uint32_t epoch;
  uint32_t n_ranks, n_comm, n_aggregate;
  uint32_t role_before[kMaxRanks];
  uint32_t role_after[kMaxRanks];
  float score_rows[kMaxRanks][kMaxRanks];  // [committee][trainer]
  uint32_t scored_mask[kMaxRanks];         // bit t of row c: score_rows[c][t] is valid
  float median[kMaxRanks];
  uint32_t n_samples[kMaxRanks];
  float avg_cost[kMaxRanks];
  float weight[kMaxRanks];
  uint32_t admitted_mask;
  uint32_t selected_mask;
  float global_loss;
  uint32_t weight_by_score;
  unsigned long long model_digest;
  uint32_t seq;  // epoch + 1, release-stored last: the record is complete when seq matches
  uint32_t pad;
};

enum FlagSlot : int {
  FLAG_TRAINED = 0,   // [kMaxRanks] trainer r's upload for epoch e is readable   -> e + 1
  FLAG_SCORED = 8,    // [kMaxRanks] committee r's score row for epoch e landed   -> e + 1
  FLAG_DONE = 16,     // [kMaxRanks] rank r finished aggregating epoch e           -> e + 1
  FLAG_SLICE = 24,    // [kMaxRanks] two-shot: slice owner r published epoch e     -> e + 1
  FLAG_COUNT = 64
};

struct FedArgs {
  PeerTable peers;
  HeapLayout lay;
  int rank;
  int n_ranks;
};

struct PlanLayer {
  long long bias_off;   // element offset of this layer's bias in the flat parameter buffer
  int use_bias;
};

// start of round: predicates, candidate list, per-layer GemmDynamic, accumulator reset,
// and (safety) wait until every rank finished consuming the buffers about to be reused.
// fp8 MLP: where candidate blobs live (local staging [slot][bytes], or directly each trainer's
// upload blob at heap offset upq_off[parity])
struct PlanBlobs {
  uint8_t* stage = nullptr; long long bytes = 0; long long upq_off[2] = {0, 0};
  int fused_pull = 0;   // staged slots are filled by the validation kernel itself (MlpValArgs::cand_src)
};
cudaError_t fed_plan_round(const FedArgs& f, const PlanLayer* layers, int n_layers,
                           int steps_per_round, int staged, cudaStream_t s,
                           const PlanBlobs* blobs = nullptr);
// trainer ("UploadLocalUpdate", CommitteePrecompiled.cpp:215-258): copy the trained weights
// into the peer-readable upload buffers, push {n_samples, avg_cost} to every replica and
// release FLAG_TRAINED on every peer.  byz_mode 1 = sign-flipped, scaled delta (fault
// injection, SURVEY.md 5.3).  straggle_us > 0: sleep that long before publishing (a slow
// client; fault injection for first-K-wins admission).
cudaError_t fed_upload(const FedArgs& f, int n_samples, int n_loss_terms, int byz_mode,
                       float byz_scale, cudaStream_t s, int straggle_us = 0);
// everyone ("UploadScores" + "Aggregate", CommitteePrecompiled.cpp:259-298, 349-456):
// committee ranks push their score row to every replica; all ranks wait for the rows, run
// the consensus math, reduce the selected uploads over P2P loads in a fixed order, write
// the new global model (+bf16, + next round's training buffers), append the BlockRecord,
// re-elect, epoch++ and release FLAG_DONE.
// host_mirror (optional, pinned host memory, >= (kMirrorSeqWord + 1) words): the kernel's last
// block copies the committed RoundState there and then release-stores the new epoch into word
// kMirrorSeqWord -- the host reads the round's result by polling that word.
// bump_seq (optional, device): round counter of the host->device input pipeline, incremented
// once at the very end of the round (prep_inputs_u8_chunks / mlp_round wait for tag *seq + 1).
constexpr int kMirrorSeqWord = 64;
cudaError_t fed_consensus_aggregate(const FedArgs& f, int n_val, int weight_by_score,
                                    int two_shot, int use_multicast, cudaStream_t s,
                                    uint32_t* host_mirror = nullptr, uint32_t* bump_seq = nullptr);

// committee ranks: pull every candidate's uploaded weights (bf16 shadow, optionally the fp32
// master) out of the trainers' HBM into local staging [slot z][n_params], each as soon as its
// trainer's flag is up.  stage_master may be null.
// `ranges` (optional, device, [n_ranges][2] = {first float4, float4 count}): pull only these
// parts of the fp32 master -- the 1-D parameters a forward pass reads in fp32.
cudaError_t fed_pull_candidates(const FedArgs& f, void* stage_shadow, float* stage_master,
                                cudaStream_t s, const long long* ranges = nullptr, int n_ranges = 0);
// committee ranks, fp8 MLP: pull each candidate's blob (nbytes at heap offset off0/off1 by
// epoch parity) into stage + slot * nbytes as soon as its trainer's flag is up
cudaError_t fed_pull_blobs(const FedArgs& f, long long off0, long long off1, long long nbytes,
                           void* stage, cudaStream_t s);
// stream-blocking wait until every trainer of the current epoch released FLAG_TRAINED
cudaError_t fed_wait_trained(const FedArgs& f, cudaStream_t s);

// thread-local predicate: kernels launched while it is set start with
// `if (*pred == 0) return;` (role predication inside a captured graph)
void set_predicate(const int* pred);
void set_pdl(bool on);   // programmatic dependent launch for all library kernels (default on)
bool pdl_enabled();
unsigned long long pdl_fallbacks();  // launches retried without the PDL attribute
void set_debug_times(long long* dev_buf8);  // GEMM phase clock stamps of CTA (0,0,0)
const int* current_predicate();

// stand-alone P2P / multicast bandwidth probes (profiles/, substrate smoke test)
cudaError_t p2p_read_probe(const float4* peer_src, float4* local_dst, int64_t n_vec,
                           cudaStream_t s);
cudaError_t mc_store_probe(float4* mc_dst, const float4* local_src, int64_t n_vec,
                           cudaStream_t s);

}  // namespace bflc
