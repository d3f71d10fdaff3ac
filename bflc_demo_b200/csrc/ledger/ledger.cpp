// See ledger.hpp for the reference parity map.
#include "ledger.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <stdexcept>

#include "consensus_math.hpp"

namespace bflc {

// ------------------------------------------------------------------ sha256
namespace {
constexpr uint32_t kK[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4,
    0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be, 0x550c7dc3, 0x72be5d74, 0x80deb1fe,
    0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f,
    0x4a7484aa, 0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7,
    0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85, 0x2e1b2138, 0x4d2c6dfc,
    0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b,
    0xc24b8b70, 0xc76c51a3, 0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116,
    0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f, 0x682e6ff3,
    0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7,
    0xc67178f2};
inline uint32_t rotr(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }

void sha_block(uint32_t h[8], const uint8_t* p) {
  uint32_t w[64];
  for (int i = 0; i < 16; ++i)
    w[i] = (uint32_t(p[4 * i]) << 24) | (uint32_t(p[4 * i + 1]) << 16) |
           (uint32_t(p[4 * i + 2]) << 8) | uint32_t(p[4 * i + 3]);
  for (int i = 16; i < 64; ++i) {
    const uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3);
    const uint32_t s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
    w[i] = w[i - 16] + s0 + w[i - 7] + s1;
  }
  uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
  for (int i = 0; i < 64; ++i) {
    const uint32_t S1 = rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25);
    const uint32_t ch = (e & f) ^ (~e & g);
    const uint32_t t1 = hh + S1 + ch + kK[i] + w[i];
    const uint32_t S0 = rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22);
    const uint32_t mj = (a & b) ^ (a & c) ^ (b & c);
    const uint32_t t2 = S0 + mj;
    hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
  }
  h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
}

// little-endian binary writer / reader used for block hashing and snapshots
struct Writer {
  std::string buf;
  template <typename T>
  void pod(const T& v) { buf.append(reinterpret_cast<const char*>(&v), sizeof(T)); }
  template <typename T>
  void vec(const std::vector<T>& v) {
    pod<uint64_t>(v.size());
    if (!v.empty()) buf.append(reinterpret_cast<const char*>(v.data()), sizeof(T) * v.size());
  }
  void hash(const Hash256& h) { buf.append(reinterpret_cast<const char*>(h.data()), 32); }
};
struct Reader {
  const std::string& buf;
  size_t pos = 0;
  explicit Reader(const std::string& b) : buf(b) {}
  void need(size_t n) const {   // overflow-safe: pos <= buf.size() always holds
    if (n > buf.size() - pos) throw std::runtime_error("ledger snapshot truncated");
  }
  template <typename T>
  T pod() {
    need(sizeof(T));
    T v;
    std::memcpy(&v, buf.data() + pos, sizeof(T));
    pos += sizeof(T);
    return v;
  }
  template <typename T>
  std::vector<T> vec() {
    const uint64_t n = pod<uint64_t>();
    if (n > (buf.size() - pos) / sizeof(T)) throw std::runtime_error("ledger snapshot truncated");
    std::vector<T> v(n);
    if (n) std::memcpy(v.data(), buf.data() + pos, n * sizeof(T));
    pos += n * sizeof(T);
    return v;
  }
  Hash256 hash() {
    need(32);
    Hash256 h;
    std::memcpy(h.data(), buf.data() + pos, 32);
    pos += 32;
    return h;
  }
};

void write_block(Writer& w, const Block& b, bool with_hash) {
  w.pod(b.index); w.pod<int32_t>(b.epoch); w.hash(b.prev_hash);
  w.vec(b.role_before); w.vec(b.role_after); w.vec(b.admitted); w.vec(b.committee);
  w.pod<uint64_t>(b.scores.size());
  for (const auto& row : b.scores) w.vec(row);
  w.vec(b.median); w.vec(b.selected); w.vec(b.weight);
  w.pod(b.global_loss); w.hash(b.model_hash); w.pod(b.device_digest); w.pod(b.from_device);
  if (with_hash) w.hash(b.hash);
}
Block read_block(Reader& r) {
  Block b;
  b.index = r.pod<uint64_t>(); b.epoch = r.pod<int32_t>(); b.prev_hash = r.hash();
  b.role_before = r.vec<uint32_t>(); b.role_after = r.vec<uint32_t>();
  b.admitted = r.vec<int>(); b.committee = r.vec<int>();
  const uint64_t nrows = r.pod<uint64_t>();
  for (uint64_t i = 0; i < nrows; ++i) b.scores.push_back(r.vec<float>());
  b.median = r.vec<float>(); b.selected = r.vec<int>(); b.weight = r.vec<float>();
  b.global_loss = r.pod<float>(); b.model_hash = r.hash();
  b.device_digest = r.pod<uint64_t>(); b.from_device = r.pod<uint8_t>();
  b.hash = r.hash();
  return b;
}

uint64_t splitmix64(uint64_t& s) {
  uint64_t z = (s += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

using CIn = ConsensusIn<kCMaxRanks>;
using COut = ConsensusOut<kCMaxRanks>;
}  // namespace

Hash256 sha256(const void* data, size_t n) {
  uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a,
                   0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
  const uint8_t* p = static_cast<const uint8_t*>(data);
  size_t full = n / 64;
  for (size_t i = 0; i < full; ++i) sha_block(h, p + 64 * i);
  uint8_t tail[128] = {0};
  const size_t rem = n - full * 64;
  std::memcpy(tail, p + full * 64, rem);
  tail[rem] = 0x80;
  const size_t tl = rem + 9 <= 64 ? 64 : 128;
  const uint64_t bits = static_cast<uint64_t>(n) * 8;
  for (int i = 0; i < 8; ++i) tail[tl - 1 - i] = static_cast<uint8_t>(bits >> (8 * i));
  sha_block(h, tail);
  if (tl == 128) sha_block(h, tail + 64);
  Hash256 out;
  for (int i = 0; i < 8; ++i) {
    out[4 * i] = h[i] >> 24; out[4 * i + 1] = h[i] >> 16; out[4 * i + 2] = h[i] >> 8;
    out[4 * i + 3] = h[i];
  }
  return out;
}

std::string hex(const Hash256& h) {
  static const char* d = "0123456789abcdef";
  std::string s(64, '0');
  for (int i = 0; i < 32; ++i) { s[2 * i] = d[h[i] >> 4]; s[2 * i + 1] = d[h[i] & 15]; }
  return s;
}

const char* status_name(Status s) {
  switch (s) {
    case Status::OK: return "OK";
    case Status::NOT_STARTED: return "NOT_STARTED";
    case Status::STALE_EPOCH: return "STALE_EPOCH";
    case Status::DUPLICATE: return "DUPLICATE";
    case Status::QUOTA_FULL: return "QUOTA_FULL";
    case Status::NOT_COMMITTEE: return "NOT_COMMITTEE";
    case Status::UNKNOWN_CLIENT: return "UNKNOWN_CLIENT";
    case Status::BAD_PAYLOAD: return "BAD_PAYLOAD";
    case Status::AGGREGATED: return "AGGREGATED";
    case Status::NOT_TRAINER: return "NOT_TRAINER";
    case Status::NOT_READY: return "NOT_READY";
  }
  return "?";
}

std::string LedgerConfig::validate() const {
  if (client_num < 1 || client_num > kCMaxRanks) return "client_num must be in [1, 64]";
  if (comm_count < 1) return "comm_count must be >= 1";
  if (aggregate_count < 1) return "aggregate_count must be >= 1";
  if (aggregate_count > needed_update_count) return "aggregate_count > needed_update_count";
  if (model_size < 1) return "model_size must be >= 1";
  if (!(learning_rate > 0.f)) return "learning_rate must be > 0";
  if (solo) {
    if (comm_count > client_num) return "comm_count > client_num";
    if (needed_update_count > client_num) return "needed_update_count > client_num";
    return "";
  }
  // comm_count > needed_update_count is allowed (BASELINE config #4: committee 5 of 8): the
  // election takes every scored trainer and refills from the outgoing committee.
  if (needed_update_count > client_num - comm_count)
    return "needed_update_count > client_num - comm_count (not enough trainers)";
  return "";
}

Ledger::Ledger(const LedgerConfig& cfg) : cfg_(cfg) {
  const std::string err = cfg.validate();
  if (!err.empty()) throw std::invalid_argument("LedgerConfig: " + err);
  global_.assign(static_cast<size_t>(cfg.model_size), 0.f);  // InitGlobalModel, C:321-346
}

void Ledger::log(std::string s) {
  if (log_.size() < 4096) log_.push_back(std::move(s));
}

const MethodInfo* method_table(int* n) {
  static const MethodInfo kTable[] = {
      {Method::RegisterNode, "RegisterNode()", false},
      {Method::QueryState, "QueryState()", true},
      {Method::QueryGlobalModel, "QueryGlobalModel()", true},
      {Method::UploadLocalUpdate, "UploadLocalUpdate(string,int256)", false},
      {Method::UploadScores, "UploadScores(int256,string)", false},
      {Method::QueryAllUpdates, "QueryAllUpdates()", true},
  };
  if (n) *n = 6;
  return kTable;
}

Method method_from_signature(const std::string& s) {
  int n = 0;
  const MethodInfo* t = method_table(&n);
  for (int i = 0; i < n; ++i) {
    const std::string sig = t[i].signature;
    if (s == sig || s == sig.substr(0, sig.find('('))) return t[i].id;
  }
  return Method::Unknown;
}

Status Ledger::RegisterNode(int client) {
  std::lock_guard<std::mutex> g(mu_);
  ++ctr_.calls;
  if (client < 0 || client >= cfg_.client_num) return Status::UNKNOWN_CLIENT;
  if (role_.count(client)) return Status::OK;  // idempotent, C:171
  role_[client] = ROLE_TRAINER;
  registered_.push_back(client);
  ++ctr_.register_ok;
  if (static_cast<int>(role_.size()) == cfg_.client_num && epoch_ == kEpochNotStarted) {
    // C:175-186: once everybody registered pick the first committee and start epoch 0.
    std::vector<int> ids;
    for (auto& kv : role_) ids.push_back(kv.first);
    if (cfg_.seed != 0) {
      uint64_t s = cfg_.seed;
      for (size_t i = ids.size(); i > 1; --i) std::swap(ids[i - 1], ids[splitmix64(s) % i]);
    }
    if (cfg_.solo) {
      for (auto& kv : role_) kv.second = ROLE_TRAINER | ROLE_COMM;
    } else {
      for (int i = 0; i < cfg_.comm_count; ++i) role_[ids[static_cast<size_t>(i)]] = ROLE_COMM;
    }
    epoch_ = 0;
    log("all " + std::to_string(cfg_.client_num) + " nodes registered, epoch 0 starts");
  }
  return Status::OK;
}

std::pair<uint32_t, int> Ledger::QueryState(int client) {
  std::lock_guard<std::mutex> g(mu_);
  ++ctr_.calls; ++ctr_.queries;
  auto it = role_.find(client);
  return {it == role_.end() ? static_cast<uint32_t>(ROLE_TRAINER) : it->second, epoch_};
}

std::pair<std::vector<float>, int> Ledger::QueryGlobalModel() {
  std::lock_guard<std::mutex> g(mu_);
  ++ctr_.calls; ++ctr_.queries;
  return {global_, epoch_};
}

Status Ledger::UploadLocalUpdate(int client, const std::vector<float>& delta, UpdateMeta meta,
                                 int ep) {
  std::lock_guard<std::mutex> g(mu_);
  ++ctr_.calls;
  auto reject = [&](Status s) {
    ++ctr_.uploads_rejected;
    log("the update of local model is not collected (" + std::string(status_name(s)) + ")");
    return s;
  };
  if (epoch_ == kEpochNotStarted) return reject(Status::NOT_STARTED);
  if (ep != epoch_) return reject(Status::STALE_EPOCH);
  auto it = role_.find(client);
  if (it == role_.end()) return reject(Status::UNKNOWN_CLIENT);
  if (!(it->second & ROLE_TRAINER)) return reject(Status::NOT_TRAINER);
  if (updates_.count(client)) return reject(Status::DUPLICATE);
  if (static_cast<int>(updates_.size()) >= cfg_.needed_update_count)
    return reject(Status::QUOTA_FULL);
  if (static_cast<int64_t>(delta.size()) != cfg_.model_size) return reject(Status::BAD_PAYLOAD);
  LocalUpdate u;
  u.sender = client; u.delta = delta; u.meta = meta; u.arrival = arrivals_++;
  updates_.emplace(client, std::move(u));
  ++ctr_.uploads_ok;
  log("the update of local model is collected");
  return Status::OK;
}

std::vector<LocalUpdate> Ledger::QueryAllUpdates() {
  std::lock_guard<std::mutex> g(mu_);
  ++ctr_.calls; ++ctr_.queries;
  std::vector<LocalUpdate> out;
  if (static_cast<int>(updates_.size()) < cfg_.needed_update_count) return out;  // C:304-307
  for (auto& kv : updates_) out.push_back(kv.second);
  std::sort(out.begin(), out.end(),
            [](const LocalUpdate& a, const LocalUpdate& b) { return a.arrival < b.arrival; });
  return out;
}

Status Ledger::UploadScores(int client, int ep, const std::map<int, float>& scores) {
  std::lock_guard<std::mutex> g(mu_);
  ++ctr_.calls;
  auto reject = [&](Status s) { ++ctr_.scores_rejected; return s; };
  if (epoch_ == kEpochNotStarted) return reject(Status::NOT_STARTED);
  if (ep != epoch_) return reject(Status::STALE_EPOCH);
  auto it = role_.find(client);
  if (it == role_.end() || !(it->second & ROLE_COMM)) return reject(Status::NOT_COMMITTEE);
  if (static_cast<int>(updates_.size()) < cfg_.needed_update_count)
    return reject(Status::NOT_READY);
  std::map<int, float> row;
  for (auto& kv : scores) {
    if (!updates_.count(kv.first)) continue;  // only admitted trainers can be scored
    if (!std::isfinite(kv.second)) return reject(Status::BAD_PAYLOAD);
    row[kv.first] = kv.second;
  }
  // A repeated upload replaces the row and is NOT counted twice (the reference increments
  // score_count on duplicates, C:279-289 -- a latent bug that is deliberately not emulated).
  scores_[client] = std::move(row);
  ++ctr_.scores_ok;
  log(std::to_string(scores_.size()) + " scores has been uploaded");
  if (static_cast<int>(scores_.size()) == cfg_.comm_count) {
    aggregate_locked();
    return Status::AGGREGATED;
  }
  return Status::OK;
}

void Ledger::aggregate_locked() {
  // Aggregate, C:349-456
  CIn in;
  std::memset(&in, 0, sizeof(in));
  COut out;
  std::memset(&out, 0, sizeof(out));
  const int n = cfg_.client_num;
  in.n_ranks = n;
  in.n_comm = cfg_.comm_count;
  in.n_aggregate = cfg_.aggregate_count;
  in.weight_by_score = cfg_.weight_by_score;
  for (auto& kv : role_) in.role[kv.first] = kv.second;
  for (auto& kv : updates_) {
    in.admitted[kv.first] = 1;
    in.n_samples[kv.first] = kv.second.meta.n_samples;
    in.avg_cost[kv.first] = kv.second.meta.avg_cost;
  }
  for (auto& row : scores_)
    for (auto& kv : row.second) {
      in.scored[row.first][kv.first] = 1;
      in.score[row.first][kv.first] = kv.second;
    }
  run_consensus<kCMaxRanks>(in, out);

  // steps 2-4: global -= lr * sum_k w_k * delta_k, fixed (ascending id) order
  std::vector<float> total(global_.size(), 0.f);
  for (int t = 0; t < n; ++t) {
    if (!out.selected[t]) continue;
    const float w = out.weight[t];
    const std::vector<float>& d = updates_.at(t).delta;
    for (size_t i = 0; i < total.size(); ++i) total[i] = std::fmaf(w, d[i], total[i]);
  }
  for (size_t i = 0; i < global_.size(); ++i) global_[i] -= cfg_.learning_rate * total[i];

  Block b;
  b.epoch = epoch_;
  b.role_before.assign(static_cast<size_t>(n), 0);
  b.role_after.assign(static_cast<size_t>(n), 0);
  for (int r = 0; r < n; ++r) {
    b.role_before[static_cast<size_t>(r)] = in.role[r];
    b.role_after[static_cast<size_t>(r)] = out.role_after[r];
  }
  std::vector<const LocalUpdate*> adm;
  for (auto& kv : updates_) adm.push_back(&kv.second);
  std::sort(adm.begin(), adm.end(),
            [](const LocalUpdate* a, const LocalUpdate* c) { return a->arrival < c->arrival; });
  for (auto* u : adm) { b.admitted.push_back(u->sender); b.median.push_back(out.median[u->sender]); }
  for (auto& row : scores_) {
    b.committee.push_back(row.first);
    std::vector<float> r;
    for (int t : b.admitted) {
      auto f = row.second.find(t);
      r.push_back(f == row.second.end() ? std::nanf("") : f->second);
    }
    b.scores.push_back(std::move(r));
  }
  for (int t = 0; t < n; ++t)
    if (out.selected[t]) { b.selected.push_back(t); b.weight.push_back(out.weight[t]); }
  b.global_loss = out.global_loss;
  b.model_hash = sha256(global_.data(), global_.size() * sizeof(float));
  last_loss_ = out.global_loss;
  log("the " + std::to_string(epoch_) + " epoch , global loss : " + std::to_string(out.global_loss));

  for (int r = 0; r < n; ++r)
    if (role_.count(r)) role_[r] = out.role_after[r];
  updates_.clear();
  scores_.clear();
  epoch_ += 1;
  ++ctr_.aggregations;
  append_block_locked(std::move(b));
}

Hash256 Ledger::hash_block(const Block& b) const {
  Writer w;
  write_block(w, b, /*with_hash=*/false);
  return sha256(w.buf.data(), w.buf.size());
}

void Ledger::append_block_locked(Block&& b) {
  b.index = chain_.size();
  if (!chain_.empty()) b.prev_hash = chain_.back().hash;
  b.hash = hash_block(b);
  chain_.push_back(std::move(b));
}

void Ledger::Bootstrap(const std::vector<uint32_t>& roles) {
  std::lock_guard<std::mutex> g(mu_);
  if (static_cast<int>(roles.size()) != cfg_.client_num)
    throw std::invalid_argument("Bootstrap: one role per client required");
  role_.clear(); registered_.clear();
  for (int r = 0; r < cfg_.client_num; ++r) {
    role_[r] = roles[static_cast<size_t>(r)];
    registered_.push_back(r);
  }
  epoch_ = 0;
}

std::string Ledger::AppendDeviceRound(const DeviceRound& r) {
  std::lock_guard<std::mutex> g(mu_);
  const int n = cfg_.client_num;
  if (r.epoch != epoch_)
    return "epoch mismatch: device " + std::to_string(r.epoch) + " host " + std::to_string(epoch_);
  // the device path keeps its masks in 32-bit words (kMaxRanks = 8 today)
  if (n > 32) return "device rounds support at most 32 clients";
  const size_t un = static_cast<size_t>(n);
  if (r.role_before.size() < un || r.role_after.size() < un || r.score_rows.size() < un ||
      r.scored_mask.size() < un || r.n_samples.size() < un || r.avg_cost.size() < un)
    return "short device record";
  for (size_t c = 0; c < un; ++c)
    if (r.score_rows[c].size() < un) return "short score row in device record";
  CIn in;
  std::memset(&in, 0, sizeof(in));
  COut out;
  std::memset(&out, 0, sizeof(out));
  in.n_ranks = n; in.n_comm = cfg_.comm_count; in.n_aggregate = cfg_.aggregate_count;
  in.weight_by_score = r.weight_by_score;
  for (int c = 0; c < n; ++c) {
    if (role_.at(c) != r.role_before[static_cast<size_t>(c)])
      return "role_before mismatch at rank " + std::to_string(c);
    in.role[c] = r.role_before[static_cast<size_t>(c)];
    in.admitted[c] = (r.admitted_mask >> c) & 1u;
    in.n_samples[c] = r.n_samples[static_cast<size_t>(c)];
    in.avg_cost[c] = r.avg_cost[static_cast<size_t>(c)];
    for (int t = 0; t < n; ++t) {
      in.scored[c][t] = (r.scored_mask[static_cast<size_t>(c)] >> t) & 1u;
      in.score[c][t] = r.score_rows[static_cast<size_t>(c)][static_cast<size_t>(t)];
    }
  }
  run_consensus<kCMaxRanks>(in, out);  // re-execute the election on the host
  uint32_t sel = 0;
  for (int t = 0; t < n; ++t)
    if (out.selected[t]) sel |= 1u << t;
  if (sel != r.selected_mask) return "selected set mismatch";
  for (int c = 0; c < n; ++c)
    if (out.role_after[c] != r.role_after[static_cast<size_t>(c)])
      return "re-election mismatch at rank " + std::to_string(c);
  if (std::fabs(out.global_loss - r.global_loss) > 1e-5f * (1.f + std::fabs(out.global_loss)))
    return "global_loss mismatch";

  Block b;
  b.epoch = epoch_;
  b.from_device = 1;
  b.device_digest = r.model_digest;
  b.role_before.assign(r.role_before.begin(), r.role_before.begin() + n);
  b.role_after.assign(r.role_after.begin(), r.role_after.begin() + n);
  for (int t = 0; t < n; ++t)
    if (in.admitted[t]) { b.admitted.push_back(t); b.median.push_back(out.median[t]); }
  for (int c = 0; c < n; ++c) {
    if (!(in.role[c] & ROLE_COMM)) continue;
    b.committee.push_back(c);
    std::vector<float> row;
    for (int t : b.admitted) row.push_back(in.scored[c][t] ? in.score[c][t] : std::nanf(""));
    b.scores.push_back(std::move(row));
  }
  for (int t = 0; t < n; ++t)
    if (out.selected[t]) { b.selected.push_back(t); b.weight.push_back(out.weight[t]); }
  b.global_loss = out.global_loss;
  last_loss_ = out.global_loss;
  for (int c = 0; c < n; ++c) role_[c] = out.role_after[c];
  epoch_ += 1;
  ++ctr_.aggregations;
  log("the " + std::to_string(b.epoch) + " epoch , global loss : " + std::to_string(b.global_loss));
  append_block_locked(std::move(b));
  return "";
}

int Ledger::epoch() const { std::lock_guard<std::mutex> g(mu_); return epoch_; }
int Ledger::update_count() const { std::lock_guard<std::mutex> g(mu_); return (int)updates_.size(); }
int Ledger::score_count() const { std::lock_guard<std::mutex> g(mu_); return (int)scores_.size(); }
size_t Ledger::n_blocks() const { std::lock_guard<std::mutex> g(mu_); return chain_.size(); }
float Ledger::last_global_loss() const { std::lock_guard<std::mutex> g(mu_); return last_loss_; }
OpCounters Ledger::counters() const { std::lock_guard<std::mutex> g(mu_); return ctr_; }
std::vector<Block> Ledger::blocks() const { std::lock_guard<std::mutex> g(mu_); return chain_; }
std::vector<std::string> Ledger::drain_log() {
  std::lock_guard<std::mutex> g(mu_);
  std::vector<std::string> out;
  out.swap(log_);
  return out;
}
std::vector<uint32_t> Ledger::roles() const {
  std::lock_guard<std::mutex> g(mu_);
  std::vector<uint32_t> out(static_cast<size_t>(cfg_.client_num), 0);
  for (auto& kv : role_) out[static_cast<size_t>(kv.first)] = kv.second;
  return out;
}

Hash256 Ledger::state_hash() const {
  std::lock_guard<std::mutex> g(mu_);
  Writer w;
  w.pod<int32_t>(epoch_);
  for (auto& kv : role_) { w.pod<int32_t>(kv.first); w.pod(kv.second); }
  w.vec(global_);
  for (auto& kv : updates_) { w.pod<int32_t>(kv.first); w.vec(kv.second.delta); }
  for (auto& row : scores_)
    for (auto& kv : row.second) { w.pod<int32_t>(row.first); w.pod<int32_t>(kv.first); w.pod(kv.second); }
  if (!chain_.empty()) w.hash(chain_.back().hash);
  return sha256(w.buf.data(), w.buf.size());
}

bool Ledger::verify_chain() const {
  std::lock_guard<std::mutex> g(mu_);
  Hash256 prev{};
  for (size_t i = 0; i < chain_.size(); ++i) {
    const Block& b = chain_[i];
    if (b.index != i || b.prev_hash != prev || hash_block(b) != b.hash) return false;
    prev = b.hash;
  }
  return true;
}

std::string Ledger::snapshot() const {
  std::lock_guard<std::mutex> g(mu_);
  Writer w;
  w.pod<uint32_t>(0xB1F1C0DEu);  // magic
  w.pod<uint32_t>(1);            // version
  w.pod<int32_t>(cfg_.client_num); w.pod<int32_t>(cfg_.comm_count);
  w.pod<int32_t>(cfg_.aggregate_count); w.pod<int32_t>(cfg_.needed_update_count);
  w.pod(cfg_.learning_rate); w.pod<int64_t>(cfg_.model_size);
  w.pod<int32_t>(cfg_.weight_by_score); w.pod<int32_t>(cfg_.solo); w.pod<uint64_t>(cfg_.seed);
  w.pod<int32_t>(epoch_);
  w.vec(global_); w.vec(registered_);
  w.pod<uint64_t>(role_.size());
  for (auto& kv : role_) { w.pod<int32_t>(kv.first); w.pod(kv.second); }
  w.pod<uint64_t>(updates_.size());
  for (auto& kv : updates_) {
    w.pod<int32_t>(kv.first); w.vec(kv.second.delta); w.pod(kv.second.meta.n_samples);
    w.pod(kv.second.meta.avg_cost); w.pod(kv.second.arrival);
  }
  w.pod<uint64_t>(scores_.size());
  for (auto& row : scores_) {
    w.pod<int32_t>(row.first); w.pod<uint64_t>(row.second.size());
    for (auto& kv : row.second) { w.pod<int32_t>(kv.first); w.pod(kv.second); }
  }
  w.pod(arrivals_); w.pod(last_loss_);
  w.pod<uint64_t>(chain_.size());
  for (auto& b : chain_) write_block(w, b, true);
  return w.buf;
}

std::unique_ptr<Ledger> Ledger::restore(const std::string& blob) {
  Reader r(blob);
  if (r.pod<uint32_t>() != 0xB1F1C0DEu) throw std::runtime_error("not a ledger snapshot");
  if (r.pod<uint32_t>() != 1) throw std::runtime_error("unsupported snapshot version");
  LedgerConfig c;
  c.client_num = r.pod<int32_t>(); c.comm_count = r.pod<int32_t>();
  c.aggregate_count = r.pod<int32_t>(); c.needed_update_count = r.pod<int32_t>();
  c.learning_rate = r.pod<float>(); c.model_size = r.pod<int64_t>();
  c.weight_by_score = r.pod<int32_t>(); c.solo = r.pod<int32_t>(); c.seed = r.pod<uint64_t>();
  // the constructor zero-fills a model of model_size floats: refuse a size the blob cannot hold
  // before allocating it (a corrupted size field would otherwise cost gigabytes of host memory)
  if (c.model_size > static_cast<int64_t>((blob.size() - r.pos) / sizeof(float)))
    throw std::runtime_error("ledger snapshot: model size mismatch");
  auto LP = std::make_unique<Ledger>(c);
  Ledger& L = *LP;
  L.epoch_ = r.pod<int32_t>();
  L.global_ = r.vec<float>(); L.registered_ = r.vec<int>();
  // every client id in the blob indexes fixed [kCMaxRanks] arrays later (aggregate_locked): a
  // crafted snapshot must not be able to name an id outside [0, client_num)
  auto id = [&](int k) {
    if (k < 0 || k >= c.client_num) throw std::runtime_error("ledger snapshot: client id out of range");
    return k;
  };
  if (static_cast<int64_t>(L.global_.size()) != c.model_size)
    throw std::runtime_error("ledger snapshot: model size mismatch");
  for (int k : L.registered_) id(k);
  for (uint64_t n = r.pod<uint64_t>(), i = 0; i < n; ++i) {
    const int k = id(r.pod<int32_t>());
    L.role_[k] = r.pod<uint32_t>();
  }
  for (uint64_t n = r.pod<uint64_t>(), i = 0; i < n; ++i) {
    LocalUpdate u;
    u.sender = id(r.pod<int32_t>()); u.delta = r.vec<float>(); u.meta.n_samples = r.pod<uint32_t>();
    u.meta.avg_cost = r.pod<float>(); u.arrival = r.pod<uint64_t>();
    if (static_cast<int64_t>(u.delta.size()) != c.model_size)
      throw std::runtime_error("ledger snapshot: update size mismatch");
    L.updates_.emplace(u.sender, std::move(u));
  }
  for (uint64_t n = r.pod<uint64_t>(), i = 0; i < n; ++i) {
    const int c2 = id(r.pod<int32_t>());
    std::map<int, float> row;
    for (uint64_t m = r.pod<uint64_t>(), j = 0; j < m; ++j) {
      const int t = id(r.pod<int32_t>());
      row[t] = r.pod<float>();
    }
    L.scores_[c2] = std::move(row);
  }
  L.arrivals_ = r.pod<uint64_t>(); L.last_loss_ = r.pod<float>();
  for (uint64_t n = r.pod<uint64_t>(), i = 0; i < n; ++i) L.chain_.push_back(read_block(r));
  if (!L.verify_chain()) throw std::runtime_error("snapshot chain fails verification");
  return LP;
}

}  // namespace bflc
