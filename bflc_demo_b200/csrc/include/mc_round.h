// Device structs and launchers of the multi-client engine (engine/multiclient.py): C <= 32
// virtual clients share one GPU, every buffer lives in local HBM.  Separate from RoundState /
// RoundPlan / BlockRecord (one client per GPU, <= 8 ranks), whose layouts stay fixed.
//
//   k_mc_plan         QueryState for every client: trainer predicates, barrier words, Adam step
//                     bases, committee list, simulated arrival order + first-K admission
//                     (per-client shard sizes, step counts and validation rows: McClients)
//   mlp_round x C     local training, one persistent launch per client (predicated)
//   k_mc_byzantine    fault injection: update := global - s * (trained - global)
//   mc_val            committee validation: every member x every admitted candidate, one launch
//   k_mc_consensus    scores, run_consensus<32>, ledger page, block record
//   k_mc_fedavg       FedAvg of the selected masters into the global model and every client
//                     (optionally followed by a server optimizer step: McServerOpt)
#pragma once
#include <cstdint>

#include "bflc_kernels.h"

namespace bflc {

constexpr int kMcMaxClients = 32;

// The ledger page of the multi-client engine.
struct McState {
  uint32_t epoch;
  uint32_t n_clients, n_comm, n_aggregate;
  uint32_t n_needed;                 // NEEDED_UPDATE_COUNT; < #trainers: first-K admission
  uint32_t seed;                     // arrival order of epoch e = permutation of (seed, e)
  uint32_t straggler_mask;           // these clients always arrive last
  uint32_t blocks_appended;
  uint32_t role[kMcMaxClients];      // RoleBits (consensus_math.hpp)
  float last_median[kMcMaxClients];
  uint32_t admitted_mask;
  uint32_t selected_mask;
  float global_loss;
  uint32_t pad;
  unsigned long long model_digest;
};

// Per-round scratch, rewritten by k_mc_plan.
struct McPlan {
  int is_trainer[kMcMaxClients];          // predicate of client c's training launch
  unsigned int barrier[kMcMaxClients];    // grid-barrier word of client c's persistent trainer
  int opt_step[kMcMaxClients];            // Adam t base of client c (steps before this round)
  int opt_total[kMcMaxClients];           // running step count (never reset)
  float loss_sum[kMcMaxClients];          // client c's training loss accumulator
  unsigned int train_correct[kMcMaxClients];
  int n_cand;
  int cand[kMcMaxClients];                // admitted clients in arrival order (candidate slots)
  int n_comm;
  int comm[kMcMaxClients];                // committee members, ascending id (committee slots)
  uint32_t admitted_mask;
  uint32_t epoch;                         // the epoch being run (consensus -> FedAvg)
  unsigned int correct[kMcMaxClients][kMcMaxClients];   // [member][candidate] validation hits
  int n_sel;
  int sel[kMcMaxClients];                 // selected clients, ascending id = FedAvg order
  float sel_w[kMcMaxClients];
  unsigned int fedavg_blocks_done;
  uint32_t pad;
  unsigned long long digest_acc;
};

// One record per round, drained by the host ledger (Ledger.AppendDeviceRound with n = C).
struct McBlockRecord {
  uint32_t epoch;
  uint32_t n_clients, n_comm, n_aggregate;
  uint32_t role_before[kMcMaxClients];
  uint32_t role_after[kMcMaxClients];
  float score_rows[kMcMaxClients][kMcMaxClients];   // [committee][trainer]
  uint32_t scored_mask[kMcMaxClients];
  float median[kMcMaxClients];
  uint32_t n_samples[kMcMaxClients];
  float avg_cost[kMcMaxClients];
  float weight[kMcMaxClients];
  uint32_t admitted_mask;
  uint32_t selected_mask;
  float global_loss;
  uint32_t weight_by_score;
  unsigned long long model_digest;
  uint32_t seq;   // epoch + 1, written last
  uint32_t pad;
};

// Per-client addresses and shard constants, kept in device memory (one entry per client),
// written once at construction.  Clients may hold shards of different sizes: client c trains
// steps[c] mini-batches of `batch` rows, reports n_samples[c] and validates as a committee member on
// the first n_val[c] rows of its own shard.
struct McClients {
  float* master[kMcMaxClients];            // fp32 work master (training weights, FedAvg operand)
  uint16_t* shadow[kMcMaxClients];         // bf16 work shadow
  uint8_t* blob[kMcMaxClients];            // fp8: Mx8MlpLayout blob (training copy + candidate)
  const int32_t* labels[kMcMaxClients];    // the client's labels (validation reads [0, n_val))
  const uint8_t* x_sf[kMcMaxClients];      // fp8: scale chunks of the client's inputs
  uint32_t n_samples[kMcMaxClients];       // S_c = (rows_c / batch) * batch, the FedAvg weight
  int steps[kMcMaxClients];                // training steps per round (loss terms = steps * batch)
  int n_val[kMcMaxClients];                // validation rows of the client as a committee member
  int batch;
  int pad;
};

struct McArgs {
  McState* st;
  McPlan* plan;
  McBlockRecord* ring;
  int ring_slots;
  const McClients* clients;   // device
  float* global_master;
  uint16_t* global_shadow;
  long long n_params;
};

// Adam step bases advance by each trainer's own McClients::steps
cudaError_t mc_plan_round(const McArgs& a, cudaStream_t s);
// byzantine clients (host list, ascending): if they trained, master/shadow := g - s * (w - g)
cudaError_t mc_byzantine(const McArgs& a, const int* ids, int n_ids, float scale, cudaStream_t s);
// scores, sample counts and average costs come from the per-client constants in McClients
cudaError_t mc_consensus(const McArgs& a, int weight_by_score, cudaStream_t s);
// Server-side optimizer of the FedOpt family (Reddi et al., 2021) applied per element to the
// pseudo-gradient d = avg - g, g the current global model, after the FedAvg sum:
//   momentum  m = fmaf(b1, m, d);                           g = fmaf(lr, m, g)
//   adam      m = fmaf(b1, m, c1 * d); v = fmaf(b2, v, c2 * (d * d));      g = g + lr * m / (sqrtf(v) + tau)
//   yogi      m as adam; d2 = d * d; v = v - c2 * d2 * sign(v - d2);       g as adam
// c1 = 1 - b1, c2 = 1 - b2 of the fp32 b1, b2 (rounded to fp32 on the host), no bias correction; m starts at 0 and v
// at tau^2 (the caller's buffers).  A round with nothing selected leaves g, m and v unchanged.
enum McServerMode : int { MC_SERVER_NONE = 0, MC_SERVER_MOMENTUM = 1, MC_SERVER_ADAM = 2, MC_SERVER_YOGI = 3 };
struct McServerOpt {
  int mode = MC_SERVER_NONE;
  float lr = 1.f, beta1 = 0.9f, beta2 = 0.99f, tau = 1e-3f;
  float* m = nullptr;   // [n_params] fp32 server state: first moment (every mode but none)
  float* v = nullptr;   // second moment (adam, yogi)
};
cudaError_t mc_fedavg(const McArgs& a, int n_clients, cudaStream_t s, const McServerOpt& so = McServerOpt{});
// copy one blob to every client's blob slot (fp8: the quantised new global model)
cudaError_t mc_broadcast_blob(const McArgs& a, const uint8_t* src, long long bytes, int n_clients,
                              cudaStream_t s);

// Committee validation of the multi-client round (mlp_val_sm100.cu, same chain body as
// mlp_val_sm100): CTA (m-tile, candidate slot z, committee slot k) scores candidate plan->cand[z]
// on the first clients->n_val[member] rows of member plan->comm[k] (its own labels and, in fp8,
// scale chunks) and adds the hits to plan->correct[member][candidate].  The grid spans the largest
// client's tiles; a CTA past its member's n_val exits.
struct McValArgs {
  int max_n_val = 0;                       // max over clients of n_val: grid x = its 128-row tiles
  int in_dim = 0, hidden = 0, n_classes = 0;
  int max_cand = 0, max_comm = 0;          // grid extent (slots beyond the plan's counts exit)
  const McPlan* plan = nullptr;
  unsigned int* correct = nullptr;         // &plan->correct[0][0]
  const CUtensorMap* x_maps = nullptr;     // [client]: rows [0, n_val[client]) of the client's inputs
  const CUtensorMap* w_maps = nullptr;     // [layer][client] (bf16 shadows or fp8 blobs)
  const McClients* clients = nullptr;      // candidate weights; the member's n_val, labels, x_sf
  long long b1_off = 0, b2_off = 0;        // bf16: element offsets of b1 / b2 in the master
  bool fp8 = false;
};
cudaError_t mc_val_sm100(const McValArgs& r, cudaStream_t stream);

}  // namespace bflc
