// Device structs and launchers of the multi-client engine (engine/multiclient.py): C <= 32
// virtual clients share one GPU, every buffer lives in local HBM.  Separate from RoundState /
// RoundPlan / BlockRecord (one client per GPU, <= 8 ranks), whose layouts stay fixed.
//
//   k_mc_plan         QueryState for every client: trainer predicates, barrier words, Adam step
//                     bases, committee list, simulated arrival order + first-K admission
//   mlp_round x C     local training, one persistent launch per client (predicated)
//   k_mc_byzantine    fault injection: update := global - s * (trained - global)
//   mc_val            committee validation: every member x every admitted candidate, one launch
//   k_mc_consensus    scores, run_consensus<32>, ledger page, block record
//   k_mc_fedavg       FedAvg of the selected masters into the global model and every client
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

// Per-client addresses, kept in device memory (one entry per client).
struct McClients {
  float* master[kMcMaxClients];            // fp32 work master (training weights, FedAvg operand)
  uint16_t* shadow[kMcMaxClients];         // bf16 work shadow
  uint8_t* blob[kMcMaxClients];            // fp8: Mx8MlpLayout blob (training copy + candidate)
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

cudaError_t mc_plan_round(const McArgs& a, int steps_per_round, cudaStream_t s);
// byzantine clients (host list, ascending): if they trained, master/shadow := g - s * (w - g)
cudaError_t mc_byzantine(const McArgs& a, const int* ids, int n_ids, float scale, cudaStream_t s);
cudaError_t mc_consensus(const McArgs& a, int n_val, int n_samples, int n_loss_terms,
                         int weight_by_score, cudaStream_t s);
cudaError_t mc_fedavg(const McArgs& a, int n_clients, cudaStream_t s);
// copy one blob to every client's blob slot (fp8: the quantised new global model)
cudaError_t mc_broadcast_blob(const McArgs& a, const uint8_t* src, long long bytes, int n_clients,
                              cudaStream_t s);

// Committee validation of the multi-client round (mlp_val_sm100.cu, same chain body as
// mlp_val_sm100): CTA (m-tile, candidate slot z, committee slot k) scores candidate plan->cand[z]
// on the first n_val rows of member plan->comm[k] and adds the hits to
// plan->correct[member][candidate].
struct McValArgs {
  int n_val = 0, in_dim = 0, hidden = 0, n_classes = 0;
  int max_cand = 0, max_comm = 0;          // grid extent (slots beyond the plan's counts exit)
  const McPlan* plan = nullptr;
  unsigned int* correct = nullptr;         // &plan->correct[0][0]
  const CUtensorMap* x_maps = nullptr;     // [client]: rows [0, n_val) of the client's inputs
  const CUtensorMap* w_maps = nullptr;     // [layer][client] (bf16 shadows or fp8 blobs)
  const McClients* clients = nullptr;      // bf16: biases from master; fp8: the blob
  long long b1_off = 0, b2_off = 0;        // bf16: element offsets of b1 / b2 in the master
  const int32_t* labels = nullptr; long long labels_stride = 0;   // [client][rows]
  bool fp8 = false;
  const uint8_t* x_sf = nullptr; long long x_sf_stride = 0;       // fp8: [client] scale chunks
};
cudaError_t mc_val_sm100(const McValArgs& r, cudaStream_t stream);

}  // namespace bflc
