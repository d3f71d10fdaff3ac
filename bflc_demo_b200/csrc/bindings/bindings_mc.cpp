// Bindings of the multi-client engine's kernels (csrc/include/mc_round.h).
#include <ATen/cuda/CUDAContext.h>
#include <torch/extension.h>

#include <cstdint>
#include <cstring>
#include <string>

#include "bflc_kernels.h"
#include "mc_round.h"

namespace py = pybind11;

namespace {

void check(cudaError_t e, const char* what) {
  TORCH_CHECK(e == cudaSuccess, "bflc::", what, " failed: ", cudaGetErrorString(e));
}
cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

template <typename T>
T* P(int64_t addr) { return reinterpret_cast<T*>(static_cast<uintptr_t>(addr)); }

// {st, plan, ring, ring_slots, clients, global_master, global_shadow, n_params}
bflc::McArgs make_mc(const py::dict& d) {
  bflc::McArgs a;
  std::memset(&a, 0, sizeof(a));
  a.st = P<bflc::McState>(d["st"].cast<int64_t>());
  a.plan = P<bflc::McPlan>(d["plan"].cast<int64_t>());
  a.ring = P<bflc::McBlockRecord>(d["ring"].cast<int64_t>());
  a.ring_slots = d["ring_slots"].cast<int>();
  a.clients = P<const bflc::McClients>(d["clients"].cast<int64_t>());
  a.global_master = P<float>(d["global_master"].cast<int64_t>());
  a.global_shadow = P<uint16_t>(d["global_shadow"].cast<int64_t>());
  a.n_params = d["n_params"].cast<int64_t>();
  TORCH_CHECK(a.st && a.plan && a.ring && a.clients && a.ring_slots > 0, "incomplete multi-client args");
  return a;
}

}  // namespace

void bind_mc(py::module_& m) {
  m.def("mc_state_init_bytes", [](int n_clients, int n_comm, int n_aggregate, int n_needed, int seed,
                                  uint32_t straggler_mask, std::vector<int> roles) {
    TORCH_CHECK(n_clients >= 1 && n_clients <= bflc::kMcMaxClients && (int)roles.size() == n_clients,
                "1 <= clients <= 32, one role per client");
    bflc::McState st;
    std::memset(&st, 0, sizeof(st));
    st.n_clients = n_clients; st.n_comm = n_comm; st.n_aggregate = n_aggregate; st.n_needed = n_needed;
    st.seed = static_cast<uint32_t>(seed); st.straggler_mask = straggler_mask;
    for (int r = 0; r < n_clients; ++r) st.role[r] = static_cast<uint32_t>(roles[r]);
    return py::bytes(reinterpret_cast<const char*>(&st), sizeof(st));
  });
  // per-client lists, one entry per client (blob / x_sf: empty in bf16)
  m.def("mc_clients_bytes", [](std::vector<int64_t> master, std::vector<int64_t> shadow, std::vector<int64_t> blob,
                               std::vector<int64_t> labels, std::vector<int64_t> x_sf,
                               std::vector<int64_t> n_samples, std::vector<int> steps, std::vector<int> n_val,
                               int batch) {
    const size_t n = master.size();
    TORCH_CHECK(n >= 1 && n <= (size_t)bflc::kMcMaxClients, "1 <= clients <= ", bflc::kMcMaxClients);
    TORCH_CHECK(shadow.size() == n && labels.size() == n && n_samples.size() == n && steps.size() == n &&
                n_val.size() == n && (blob.empty() || blob.size() == n) && (x_sf.empty() || x_sf.size() == n),
                "per-client lists: one entry per client");
    TORCH_CHECK(blob.empty() == x_sf.empty(), "fp8 needs both the blobs and the scale chunks");
    TORCH_CHECK(batch > 0, "batch must be positive");
    bflc::McClients c;
    std::memset(&c, 0, sizeof(c));
    for (size_t i = 0; i < n; ++i) {
      TORCH_CHECK(steps[i] > 0 && n_val[i] > 0 && n_samples[i] > 0 && n_samples[i] <= 0xffffffffll &&
                  (int64_t)steps[i] * batch <= (int64_t)INT32_MAX,
                  "client ", i, ": steps, n_val and n_samples must be positive");
      TORCH_CHECK(master[i] && shadow[i] && labels[i], "client ", i, ": null pointer");
      c.master[i] = P<float>(master[i]);
      c.shadow[i] = P<uint16_t>(shadow[i]);
      c.blob[i] = blob.empty() ? nullptr : P<uint8_t>(blob[i]);
      c.labels[i] = P<const int32_t>(labels[i]);
      c.x_sf[i] = x_sf.empty() ? nullptr : P<const uint8_t>(x_sf[i]);
      c.n_samples[i] = static_cast<uint32_t>(n_samples[i]);
      c.steps[i] = steps[i];
      c.n_val[i] = n_val[i];
    }
    c.batch = batch;
    return py::bytes(reinterpret_cast<const char*>(&c), sizeof(c));
  });
  m.def("mc_plan_round", [](const py::dict& d) {
    check(bflc::mc_plan_round(make_mc(d), cur_stream()), "mc_plan_round");
  });
  m.def("mc_byzantine", [](const py::dict& d, std::vector<int> ids, double scale) {
    check(bflc::mc_byzantine(make_mc(d), ids.data(), (int)ids.size(), (float)scale, cur_stream()), "mc_byzantine");
  });
  m.def("mc_consensus", [](const py::dict& d, bool weight_by_score) {
    check(bflc::mc_consensus(make_mc(d), weight_by_score ? 1 : 0, cur_stream()), "mc_consensus");
  });
  // server optimizer: "none" (plain FedAvg) | "momentum" | "adam" | "yogi"; m / v: device
  // addresses of the fp32 [n_params] server state (v: adam and yogi only)
  m.def("mc_fedavg", [](const py::dict& d, int n_clients, const std::string& server_optimizer, double lr,
                        double beta1, double beta2, double tau, int64_t m_ptr, int64_t v_ptr) {
    bflc::McServerOpt so;
    if (server_optimizer == "none") so.mode = bflc::MC_SERVER_NONE;
    else if (server_optimizer == "momentum") so.mode = bflc::MC_SERVER_MOMENTUM;
    else if (server_optimizer == "adam") so.mode = bflc::MC_SERVER_ADAM;
    else if (server_optimizer == "yogi") so.mode = bflc::MC_SERVER_YOGI;
    else TORCH_CHECK(false, "server_optimizer must be none, momentum, adam or yogi, got ", server_optimizer);
    so.lr = (float)lr; so.beta1 = (float)beta1; so.beta2 = (float)beta2; so.tau = (float)tau;
    so.m = P<float>(m_ptr); so.v = P<float>(v_ptr);
    check(bflc::mc_fedavg(make_mc(d), n_clients, cur_stream(), so), "mc_fedavg");
  }, py::arg("args"), py::arg("n_clients"), py::arg("server_optimizer") = "none", py::arg("lr") = 1.0,
     py::arg("beta1") = 0.9, py::arg("beta2") = 0.99, py::arg("tau") = 1e-3, py::arg("m") = 0, py::arg("v") = 0);
  m.def("mc_broadcast_blob", [](const py::dict& d, at::Tensor src, int n_clients) {
    check(bflc::mc_broadcast_blob(make_mc(d), src.data_ptr<uint8_t>(), src.numel(), n_clients, cur_stream()),
          "mc_broadcast_blob");
  });
  // labels, n_val and (fp8) scale chunks of every member come from its McClients entry
  m.def("mc_val", [](int64_t plan_ptr, int64_t correct_ptr, at::Tensor x_maps, at::Tensor w_maps,
                     int64_t clients_ptr, int64_t b1_off, int64_t b2_off, int max_n_val, int in_dim, int hidden,
                     int n_classes, int max_cand, int max_comm, bool fp8) {
    const int64_t ctm = static_cast<int64_t>(sizeof(CUtensorMap));
    TORCH_CHECK(max_cand >= 1 && max_cand <= bflc::kMcMaxClients && max_comm >= 1 &&
                max_comm <= bflc::kMcMaxClients, "1 <= max_cand, max_comm <= ", bflc::kMcMaxClients);
    TORCH_CHECK(max_n_val > 0, "max_n_val must be positive");
    TORCH_CHECK(x_maps.is_cuda() && x_maps.nbytes() >= bflc::kMcMaxClients * ctm && w_maps.is_cuda() &&
                w_maps.nbytes() >= 2 * bflc::kMcMaxClients * ctm,
                "x_maps: one tensor map per client slot, w_maps: [2][", bflc::kMcMaxClients, "] (device)");
    bflc::McValArgs r;
    r.max_n_val = max_n_val; r.in_dim = in_dim; r.hidden = hidden; r.n_classes = n_classes;
    r.max_cand = max_cand; r.max_comm = max_comm;
    r.plan = P<const bflc::McPlan>(plan_ptr);
    r.correct = P<unsigned int>(correct_ptr);
    r.x_maps = reinterpret_cast<const CUtensorMap*>(x_maps.data_ptr());
    r.w_maps = reinterpret_cast<const CUtensorMap*>(w_maps.data_ptr());
    r.clients = P<const bflc::McClients>(clients_ptr);
    r.b1_off = b1_off; r.b2_off = b2_off;
    r.fp8 = fp8;
    check(bflc::mc_val_sm100(r, cur_stream()), "mc_val_sm100");
  }, py::arg("plan_ptr"), py::arg("correct_ptr"), py::arg("x_maps"), py::arg("w_maps"), py::arg("clients_ptr"),
     py::arg("b1_off"), py::arg("b2_off"), py::arg("max_n_val"), py::arg("in_dim"), py::arg("hidden"),
     py::arg("n_classes"), py::arg("max_cand"), py::arg("max_comm"), py::arg("fp8") = false);
  // TMA descriptor of a K-major operand [rows][K] (row pitch ld elements), box rows_tile x 128 B
  m.def("operand_map", [](int64_t ptr, int64_t ld, int rows, int K, bool fp8, int rows_tile) {
    CUtensorMap t;
    bflc::GemmOperand op{P<const void>(ptr), ld, 0, false};
    check(bflc::gemm_make_operand_map(&t, op, fp8 ? bflc::DType::FP8_E4M3 : bflc::DType::BF16, rows, K, 1, rows_tile),
          "gemm_make_operand_map");
    return py::bytes(reinterpret_cast<const char*>(&t), sizeof(t));
  });
  // a GemmDynamic record (device-resident per-launch GEMM / mlp_val arguments) built on the host
  m.def("gemm_dynamic_bytes", [](int active, std::vector<int> map_index, std::vector<int64_t> bias) {
    TORCH_CHECK(map_index.size() <= (size_t)bflc::kMaxRanks && bias.size() <= (size_t)bflc::kMaxRanks,
                "at most kMaxRanks batches");
    bflc::GemmDynamic g;
    std::memset(&g, 0, sizeof(g));
    g.active_batches = active;
    for (size_t i = 0; i < map_index.size(); ++i) g.map_index[i] = map_index[i];
    for (size_t i = 0; i < bias.size(); ++i) g.bias[i] = P<const float>(bias[i]);
    return py::bytes(reinterpret_cast<const char*>(&g), sizeof(g));
  });
}
