// Bindings for the symmetric heap, the federated hot-path kernels, optimizers and
// elementwise helpers.  (GEMM bindings: torch_bindings.cpp.)
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <cstring>
#include <memory>
#include <cuda.h>

#include <optional>

#include "bflc_kernels.h"
#include "mc_round.h"
#include "symm_heap.hpp"

namespace py = pybind11;
using OptT = std::optional<at::Tensor>;

namespace {

void check(cudaError_t e, const char* what) {
  TORCH_CHECK(e == cudaSuccess, "bflc::", what, " failed: ", cudaGetErrorString(e));
}
cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

template <typename T>
T* P(int64_t addr) { return reinterpret_cast<T*>(static_cast<uintptr_t>(addr)); }

bflc::FedArgs make_fed(const py::dict& d) {
  bflc::FedArgs f;
  std::memset(&f, 0, sizeof(f));
  f.rank = d["rank"].cast<int>();
  f.n_ranks = d["n_ranks"].cast<int>();
  auto bases = d["peer_bases"].cast<std::vector<int64_t>>();
  TORCH_CHECK((int)bases.size() == f.n_ranks && f.n_ranks <= bflc::kMaxRanks, "bad peer table");
  for (int r = 0; r < f.n_ranks; ++r) f.peers.base[r] = P<char>(bases[r]);
  f.peers.mc_base = P<char>(d["mc_base"].cast<int64_t>());
  auto& l = f.lay;
  l.flags_off = d["flags_off"].cast<int64_t>();
  l.state_off = d["state_off"].cast<int64_t>();
  l.plan_off = d["plan_off"].cast<int64_t>();
  l.scores_off = d["scores_off"].cast<int64_t>();
  l.meta_off = d["meta_off"].cast<int64_t>();
  l.work_master_off = d["work_master_off"].cast<int64_t>();
  l.work_shadow_off = d["work_shadow_off"].cast<int64_t>();
  auto um = d["upload_master_off"].cast<std::vector<int64_t>>();
  auto us = d["upload_shadow_off"].cast<std::vector<int64_t>>();
  l.upload_master_off[0] = um.at(0); l.upload_master_off[1] = um.at(1);
  l.upload_shadow_off[0] = us.at(0); l.upload_shadow_off[1] = us.at(1);
  l.global_off = d["global_off"].cast<int64_t>();
  l.global_shadow_off = d["global_shadow_off"].cast<int64_t>();
  l.ring_off = d["ring_off"].cast<int64_t>();
  l.n_params = d["n_params"].cast<int64_t>();
  l.admit_off = d["admit_off"].cast<int64_t>();
  l.ring_slots = d["ring_slots"].cast<int>();
  return f;
}

struct PyHeap {
  std::unique_ptr<bflc::SymmHeap> h;
};

}  // namespace

void bind_extra(py::module_& m) {
  // ------------------------------------------------------------ symmetric heap
  py::class_<PyHeap>(m, "SymmHeap")
      .def(py::init([](int64_t bytes, int rank, int world, int device, const std::string& mode) {
        bflc::SymmHeap::Mode md = mode == "vmm"   ? bflc::SymmHeap::Mode::VMM
                                  : mode == "ipc" ? bflc::SymmHeap::Mode::IPC
                                                  : bflc::SymmHeap::Mode::LOCAL;
        auto p = std::make_unique<PyHeap>();
        p->h = std::make_unique<bflc::SymmHeap>((size_t)bytes, rank, world, device, md);
        return p;
      }))
      .def("export_handle", [](PyHeap& s) { return py::bytes(s.h->export_handle()); })
      .def("import_handles",
           [](PyHeap& s, const std::vector<py::bytes>& blobs) {
             std::vector<std::string> v;
             for (auto& b : blobs) v.emplace_back(static_cast<std::string>(b));
             s.h->import_handles(v);
           })
      .def("fd_listen", [](PyHeap& s, const std::string& tag) { return s.h->fd_listen(tag); })
      .def("import_via_sockets",
           [](PyHeap& s, const std::vector<std::string>& names) { s.h->import_via_sockets(names); })
      .def("mc_import_via_sockets",
           [](PyHeap& s, const std::vector<std::string>& names) { return s.h->mc_import_via_sockets(names); })
      .def("mc_create_and_export", [](PyHeap& s) { return py::bytes(s.h->mc_create_and_export()); })
      .def("mc_import_and_add",
           [](PyHeap& s, const py::bytes& b) { return s.h->mc_import_and_add(std::string(b)); })
      .def("mc_bind_and_map", [](PyHeap& s) { return s.h->mc_bind_and_map(); })
      .def("local_ptr", [](PyHeap& s) { return reinterpret_cast<int64_t>(s.h->local_ptr()); })
      .def("peer_ptr", [](PyHeap& s, int r) { return reinterpret_cast<int64_t>(s.h->peer_ptr(r)); })
      .def("mc_ptr", [](PyHeap& s) { return reinterpret_cast<int64_t>(s.h->mc_ptr()); })
      .def("bytes", [](PyHeap& s) { return (int64_t)s.h->bytes(); })
      .def("last_error", [](PyHeap& s) { return s.h->last_error(); })
      .def_static("multicast_supported", [](int dev) { return bflc::SymmHeap::multicast_supported(dev); });

  // A torch tensor aliasing raw device memory (heap regions, peer-mapped regions).
  m.def("tensor_from_ptr", [](int64_t ptr, std::vector<int64_t> shape, py::object dtype, int device) {
    auto st = torch::python::detail::py_object_to_dtype(dtype);
    auto opts = at::TensorOptions().dtype(st).device(at::kCUDA, device);
    // target_device: a peer-mapped (VMM / IPC) pointer reports the OWNING GPU as its device;
    // the view must still be a tensor of the local device so local kernels accept it.
    return at::for_blob(P<void>(ptr), shape)
        .deleter([](void*) {})
        .options(opts)
        .target_device(at::Device(at::kCUDA, static_cast<c10::DeviceIndex>(device)))
        .make_tensor();
  });

  m.def("struct_sizes", [] {
    py::dict d;
    d["RoundState"] = sizeof(bflc::RoundState);
    d["RoundPlan"] = sizeof(bflc::RoundPlan);
    d["BlockRecord"] = sizeof(bflc::BlockRecord);
    d["UploadMeta"] = sizeof(bflc::UploadMeta);
    d["AdmitPage"] = sizeof(bflc::AdmitPage);
    d["GemmDynamic"] = sizeof(bflc::GemmDynamic);
    d["FLAG_COUNT"] = (int)bflc::FLAG_COUNT;
    d["kMaxRanks"] = bflc::kMaxRanks;
    d["kMirrorSeqWord"] = bflc::kMirrorSeqWord;
    d["plan_dyn_off"] = offsetof(bflc::RoundPlan, dyn);
    d["plan_correct_off"] = offsetof(bflc::RoundPlan, correct);
    d["plan_loss_sum_off"] = offsetof(bflc::RoundPlan, loss_sum);
    d["plan_train_correct_off"] = offsetof(bflc::RoundPlan, train_correct);
    d["plan_opt_step_off"] = offsetof(bflc::RoundPlan, opt_step);
    d["plan_is_trainer_off"] = offsetof(bflc::RoundPlan, is_trainer);
    d["plan_is_comm_off"] = offsetof(bflc::RoundPlan, is_comm);
    d["plan_step_barrier_off"] = offsetof(bflc::RoundPlan, step_barrier);
    d["plan_stamps_off"] = offsetof(bflc::RoundPlan, t_stamp);
    d["plan_round_seq_off"] = offsetof(bflc::RoundPlan, round_seq);
    d["plan_opt_total_off"] = offsetof(bflc::RoundPlan, opt_total);
    d["plan_cand_blob_off"] = offsetof(bflc::RoundPlan, cand_blob);
    d["plan_cand_src_off"] = offsetof(bflc::RoundPlan, cand_src);
    d["plan_pull_cnt_off"] = offsetof(bflc::RoundPlan, pull_cnt);
    d["state_epoch_off"] = offsetof(bflc::RoundState, epoch);
    d["state_role_off"] = offsetof(bflc::RoundState, role);
    d["state_global_loss_off"] = offsetof(bflc::RoundState, global_loss);
    d["state_digest_off"] = offsetof(bflc::RoundState, model_digest);
    d["CUtensorMap"] = sizeof(CUtensorMap);
    // multi-client engine (mc_round.h)
    d["McState"] = sizeof(bflc::McState);
    d["McPlan"] = sizeof(bflc::McPlan);
    d["McBlockRecord"] = sizeof(bflc::McBlockRecord);
    d["McClients"] = sizeof(bflc::McClients);
    d["kMcMaxClients"] = bflc::kMcMaxClients;
    d["mc_plan_is_trainer_off"] = offsetof(bflc::McPlan, is_trainer);
    d["mc_plan_barrier_off"] = offsetof(bflc::McPlan, barrier);
    d["mc_plan_opt_step_off"] = offsetof(bflc::McPlan, opt_step);
    d["mc_plan_loss_sum_off"] = offsetof(bflc::McPlan, loss_sum);
    d["mc_plan_train_correct_off"] = offsetof(bflc::McPlan, train_correct);
    d["mc_plan_n_cand_off"] = offsetof(bflc::McPlan, n_cand);
    d["mc_plan_cand_off"] = offsetof(bflc::McPlan, cand);
    d["mc_plan_n_comm_off"] = offsetof(bflc::McPlan, n_comm);
    d["mc_plan_comm_off"] = offsetof(bflc::McPlan, comm);
    d["mc_plan_correct_off"] = offsetof(bflc::McPlan, correct);
    return d;
  });

  // host-side init of the replicated ledger page
  m.def("state_init_bytes", [](int n_ranks, int n_comm, int n_aggregate, std::vector<int> roles, int n_needed) {
    bflc::RoundState st;
    std::memset(&st, 0, sizeof(st));
    st.epoch = 0; st.n_ranks = n_ranks; st.n_comm = n_comm; st.n_aggregate = n_aggregate;
    st.n_needed = (uint32_t)n_needed;
    for (int r = 0; r < n_ranks && r < bflc::kMaxRanks; ++r) st.role[r] = (uint32_t)roles.at(r);
    return py::bytes(reinterpret_cast<const char*>(&st), sizeof(st));
  }, py::arg("n_ranks"), py::arg("n_comm"), py::arg("n_aggregate"), py::arg("roles"), py::arg("n_needed") = 0);

  // ------------------------------------------------------------ fed kernels
  m.def("fed_plan_round", [](const py::dict& fd, std::vector<std::pair<int64_t, bool>> layers,
                             int steps_per_round, bool staged, int64_t blob_stage_ptr, int64_t blob_bytes,
                             std::vector<int64_t> upq_off, bool fused_pull) {
    bflc::FedArgs f = make_fed(fd);
    bflc::PlanLayer pl[bflc::kMaxPlanLayers];
    TORCH_CHECK((int)layers.size() <= bflc::kMaxPlanLayers, "too many plan layers");
    for (size_t i = 0; i < layers.size(); ++i) {
      pl[i].bias_off = layers[i].first;
      pl[i].use_bias = layers[i].second ? 1 : 0;
    }
    bflc::PlanBlobs pb;
    const bool blobs = blob_bytes > 0;
    if (blobs) {
      TORCH_CHECK(upq_off.size() == 2, "upq_off: heap offsets of the two parity upload blobs");
      pb.stage = P<uint8_t>(blob_stage_ptr); pb.bytes = blob_bytes;
      pb.upq_off[0] = upq_off[0]; pb.upq_off[1] = upq_off[1];
      pb.fused_pull = fused_pull ? 1 : 0;
    }
    check(bflc::fed_plan_round(f, pl, (int)layers.size(), steps_per_round, staged ? 1 : 0, cur_stream(),
                               blobs ? &pb : nullptr),
          "fed_plan_round");
  }, py::arg("fed"), py::arg("layers"), py::arg("steps_per_round"), py::arg("staged"),
     py::arg("blob_stage_ptr") = 0, py::arg("blob_bytes") = 0, py::arg("upq_off") = std::vector<int64_t>{},
     py::arg("fused_pull") = false);
  m.def("fed_pull_blobs", [](const py::dict& fd, int64_t off0, int64_t off1, int64_t nbytes, at::Tensor stage) {
    check(bflc::fed_pull_blobs(make_fed(fd), off0, off1, nbytes, stage.data_ptr(), cur_stream()), "fed_pull_blobs");
  });
  m.def("fed_upload", [](const py::dict& fd, int n_samples, int n_loss_terms, int byz_mode,
                         double byz_scale, int straggle_us) {
    check(bflc::fed_upload(make_fed(fd), n_samples, n_loss_terms, byz_mode, (float)byz_scale, cur_stream(),
                           straggle_us),
          "fed_upload");
  }, py::arg("fed"), py::arg("n_samples"), py::arg("n_loss_terms"), py::arg("byz_mode"), py::arg("byz_scale"),
     py::arg("straggle_us") = 0);
  m.def("fed_consensus_aggregate", [](const py::dict& fd, int n_val, bool weight_by_score,
                                      bool two_shot, bool use_mc, int64_t host_mirror,
                                      int64_t bump_seq) {
    check(bflc::fed_consensus_aggregate(make_fed(fd), n_val, weight_by_score ? 1 : 0,
                                        two_shot ? 1 : 0, use_mc ? 1 : 0, cur_stream(),
                                        P<uint32_t>(host_mirror), P<uint32_t>(bump_seq)),
          "fed_consensus_aggregate");
  }, py::arg("fed"), py::arg("n_val"), py::arg("weight_by_score"), py::arg("two_shot"),
     py::arg("use_mc"), py::arg("host_mirror") = 0, py::arg("bump_seq") = 0);
  m.def("fed_pull_candidates", [](const py::dict& fd, at::Tensor stage_shadow, const OptT& stage_master,
                                  const OptT& ranges) {
    // ranges: int64 [n][2] device tensor {first float4, float4 count} -- the fp32 parts to pull
    const long long* rp = ranges.has_value() ? reinterpret_cast<const long long*>(ranges->data_ptr<int64_t>())
                                             : nullptr;
    check(bflc::fed_pull_candidates(make_fed(fd), stage_shadow.data_ptr(),
                                    stage_master.has_value() ? stage_master->data_ptr<float>() : nullptr,
                                    cur_stream(), rp, ranges.has_value() ? (int)ranges->size(0) : 0),
          "fed_pull_candidates");
  }, py::arg("fed"), py::arg("stage_shadow"), py::arg("stage_master"), py::arg("ranges") = py::none());
  m.def("fed_wait_trained", [](const py::dict& fd) {
    check(bflc::fed_wait_trained(make_fed(fd), cur_stream()), "fed_wait_trained");
  });
  m.def("set_predicate", [](int64_t ptr) { bflc::set_predicate(P<const int>(ptr)); });
  m.def("current_predicate_is_null", [] { return bflc::current_predicate() == nullptr; });
  m.def("set_pdl", [](bool on) { bflc::set_pdl(on); });
  m.def("pdl_fallbacks", [] { return bflc::pdl_fallbacks(); });
  m.def("set_debug_times", [](int64_t ptr) { bflc::set_debug_times(P<long long>(ptr)); });
  m.def("p2p_read_probe", [](int64_t src, int64_t dst, int64_t n_vec) {
    check(bflc::p2p_read_probe(P<const float4>(src), P<float4>(dst), n_vec, cur_stream()),
          "p2p_read_probe");
  });
  m.def("mc_store_probe", [](int64_t mc_dst, int64_t src, int64_t n_vec) {
    check(bflc::mc_store_probe(P<float4>(mc_dst), P<const float4>(src), n_vec, cur_stream()),
          "mc_store_probe");
  });

  // ------------------------------------------------------------ optimizers
  // whole local-training pass of the 2-layer MLP in one persistent kernel
  m.def("mx8_mlp_layout", [](int in_dim, int hidden) {
    const bflc::Mx8MlpLayout l = bflc::mx8_mlp_layout(in_dim, hidden);
    py::dict d;
    d["w1q"] = l.w1q; d["w1sf"] = l.w1sf; d["w2q"] = l.w2q; d["w2sf"] = l.w2sf;
    d["b1"] = l.b1; d["b2"] = l.b2; d["total"] = l.total; d["kb1"] = l.kb1; d["kb2"] = l.kb2;
    return d;
  });
  m.def("mlp_round", [](at::Tensor x, at::Tensor labels, at::Tensor master, at::Tensor shadow,
                        at::Tensor grad, std::vector<int64_t> offs, at::Tensor h, at::Tensor dlogits,
                        at::Tensor dh, at::Tensor loss_sum, at::Tensor correct, int64_t barrier_ptr,
                        int batch, int steps, int in_dim, int hidden, int n_classes, double lr,
                        bool adam, const OptT& mm, const OptT& vv, int64_t step_base_ptr,
                        const OptT& dbg, int plan, int epiopt, int64_t x_ready_ptr,
                        int64_t round_seq_ptr, const OptT& x_q, const OptT& x_sf, const OptT& work_q,
                        const OptT& h_q, const OptT& h_sf, const std::optional<py::dict>& fed,
                        std::vector<int64_t> upq_off, int n_samples, int n_loss_terms, int byz_mode,
                        double byz_scale, int straggle_us, double prox_mu, const OptT& prox_anchor) {
    TORCH_CHECK(offs.size() == 4, "offs = element offsets of w1, b1, w2, b2 in the flat buffer");
    bflc::MlpRoundArgs r;
    r.batch = batch; r.steps = steps; r.in_dim = in_dim; r.hidden = hidden; r.n_classes = n_classes;
    r.ncp = (int)dlogits.stride(0);
    r.n_params = master.numel();
    r.x = x.data_ptr(); r.labels = labels.data_ptr<int32_t>();
    float* mp = master.data_ptr<float>(); float* gp = grad.data_ptr<float>();
    auto* sp = reinterpret_cast<uint16_t*>(shadow.data_ptr());
    r.master = mp; r.shadow = sp; r.grad = gp;
    r.w1_shadow = sp + offs[0]; r.w2_shadow = sp + offs[2];
    r.b1 = mp + offs[1]; r.b2 = mp + offs[3];
    r.gw1 = gp + offs[0]; r.gb1 = gp + offs[1]; r.gw2 = gp + offs[2]; r.gb2 = gp + offs[3];
    r.h = h.data_ptr(); r.dlogits = dlogits.data_ptr(); r.dh = dh.data_ptr();
    r.loss_sum = loss_sum.data_ptr<float>();
    r.correct = reinterpret_cast<unsigned int*>(correct.data_ptr());
    r.barrier = P<unsigned int>(barrier_ptr);
    r.adam = adam;
    r.adam_m = mm.has_value() ? mm->data_ptr<float>() : nullptr;
    r.adam_v = vv.has_value() ? vv->data_ptr<float>() : nullptr;
    r.lr = (float)lr;
    r.step_base = P<const int>(step_base_ptr);
    r.plan = plan; r.epiopt = epiopt;
    r.x_ready = P<const unsigned int>(x_ready_ptr); r.round_seq = P<const unsigned int>(round_seq_ptr);
    if (dbg.has_value()) {
      TORCH_CHECK(dbg->numel() >= (int64_t)steps * 32 && dbg->element_size() == 8, "dbg: int64 [steps, 32]");
      r.dbg = reinterpret_cast<unsigned long long*>(dbg->data_ptr());
    }
    if (x_q.has_value()) {
      TORCH_CHECK(x_sf.has_value() && work_q.has_value() && h_q.has_value() && h_sf.has_value(),
                  "fp8 mode needs x_q, x_sf, work_q, h_q, h_sf");
      r.fp8 = true;
      r.x_q = x_q->data_ptr(); r.x_sf = x_sf->data_ptr<uint8_t>();
      r.work_q = work_q->data_ptr<uint8_t>();
      r.h_q = h_q->data_ptr<uint8_t>(); r.h_sf = h_sf->data_ptr<uint8_t>();
    }
    bflc::FedArgs f;
    if (fed.has_value()) {
      f = make_fed(*fed);
      r.fed = &f;
      if (upq_off.size() == 2) { r.upq_off[0] = upq_off[0]; r.upq_off[1] = upq_off[1]; }
      r.n_samples = n_samples; r.n_loss_terms = n_loss_terms; r.byz_mode = byz_mode; r.byz_scale = (float)byz_scale;
      r.straggle_us = straggle_us;
    }
    if (prox_anchor.has_value()) {
      TORCH_CHECK(prox_anchor->scalar_type() == at::kFloat && prox_anchor->numel() == master.numel() &&
                  prox_anchor->is_contiguous() && prox_anchor->device() == master.device(),
                  "prox_anchor: contiguous fp32 with the master's layout, on the master's device");
      r.prox_anchor = prox_anchor->data_ptr<float>();
    }
    r.prox_mu = (float)prox_mu;
    check(bflc::mlp_round_sm100(r, cur_stream()), "mlp_round_sm100");
  }, py::arg("x"), py::arg("labels"), py::arg("master"), py::arg("shadow"), py::arg("grad"), py::arg("offs"),
     py::arg("h"), py::arg("dlogits"), py::arg("dh"), py::arg("loss_sum"), py::arg("correct"),
     py::arg("barrier_ptr"), py::arg("batch"), py::arg("steps"), py::arg("in_dim"), py::arg("hidden"),
     py::arg("n_classes"), py::arg("lr"), py::arg("adam"), py::arg("m"), py::arg("v"),
     py::arg("step_base_ptr"), py::arg("dbg"), py::arg("plan"), py::arg("epiopt"), py::arg("x_ready_ptr") = 0,
     py::arg("round_seq_ptr") = 0, py::arg("x_q") = py::none(), py::arg("x_sf") = py::none(),
     py::arg("work_q") = py::none(), py::arg("h_q") = py::none(), py::arg("h_sf") = py::none(),
     py::arg("fed") = py::none(), py::arg("upq_off") = std::vector<int64_t>{}, py::arg("n_samples") = 0,
     py::arg("n_loss_terms") = 0, py::arg("byz_mode") = 0, py::arg("byz_scale") = 0.0,
     py::arg("straggle_us") = 0, py::arg("prox_mu") = 0.0, py::arg("prox_anchor") = py::none());
  // committee validation of every candidate in one launch (fwd1 -> relu -> fwd2 -> argmax)
  m.def("mlp_val", [](at::Tensor x, at::Tensor labels, at::Tensor correct, at::Tensor maps,
                      int64_t dyn1_ptr, int64_t dyn2_ptr, int n_val, int in_dim, int hidden,
                      int n_classes, int max_cand, const OptT& x_sf, int64_t cand_blob_ptr,
                      int64_t cand_src_ptr, int64_t pull_cnt_ptr, int64_t blob_bytes, int64_t stamps_ptr) {
    bflc::MlpValArgs r;
    r.n_val = n_val; r.in_dim = in_dim; r.hidden = hidden; r.n_classes = n_classes;
    r.max_cand = max_cand;
    r.x = x.data_ptr(); r.ldx = x.stride(0);
    r.maps = reinterpret_cast<const CUtensorMap*>(maps.data_ptr());
    r.dyn1 = P<const bflc::GemmDynamic>(dyn1_ptr);
    r.dyn2 = P<const bflc::GemmDynamic>(dyn2_ptr);
    r.labels = labels.data_ptr<int32_t>();
    r.correct = reinterpret_cast<unsigned int*>(correct.data_ptr());
    if (x_sf.has_value()) {
      r.fp8 = true;
      r.x_sf = x_sf->data_ptr<uint8_t>();
      r.cand_blob = P<const uint8_t* const>(cand_blob_ptr);
      if (cand_src_ptr != 0) {   // fused gather of the candidate blobs inside the kernel
        r.cand_src = P<const uint8_t* const>(cand_src_ptr);
        r.pull_cnt = P<unsigned int>(pull_cnt_ptr);
        r.blob_bytes = blob_bytes;
        r.stamps = P<unsigned long long>(stamps_ptr);
      }
    }
    check(bflc::mlp_val_sm100(r, cur_stream()), "mlp_val_sm100");
  }, py::arg("x"), py::arg("labels"), py::arg("correct"), py::arg("maps"), py::arg("dyn1_ptr"),
     py::arg("dyn2_ptr"), py::arg("n_val"), py::arg("in_dim"), py::arg("hidden"), py::arg("n_classes"),
     py::arg("max_cand"), py::arg("x_sf") = py::none(), py::arg("cand_blob_ptr") = 0,
     py::arg("cand_src_ptr") = 0, py::arg("pull_cnt_ptr") = 0, py::arg("blob_bytes") = 0,
     py::arg("stamps_ptr") = 0);
  m.def("quantize_mlp_blob", [](at::Tensor master, std::vector<int64_t> offs, int in_dim, int hidden,
                                int n_classes, at::Tensor blob) {
    TORCH_CHECK(offs.size() == 4, "offs = element offsets of w1, b1, w2, b2");
    check(bflc::quantize_mlp_blob(master.data_ptr<float>(), offs[0], offs[1], offs[2], offs[3], in_dim, hidden,
                                  n_classes, blob.data_ptr<uint8_t>(), cur_stream()),
          "quantize_mlp_blob");
  });
  m.def("optim_step",
        [](bool adam, at::Tensor master, at::Tensor grad, const OptT& shadow, const OptT& mm,
           const OptT& vv, double lr, double wd, double b1, double b2, double eps, int step,
           int64_t step_dev_ptr, int64_t active_ptr, bool zero_grad) {
          bflc::OptimArgs a;
          a.master = master.data_ptr<float>();
          a.grad = grad.data_ptr<float>();
          a.shadow_bf16 = shadow.has_value() ? shadow->data_ptr() : nullptr;
          a.n = master.numel();
          a.lr = (float)lr; a.weight_decay = (float)wd;
          a.m = mm.has_value() ? mm->data_ptr<float>() : nullptr;
          a.v = vv.has_value() ? vv->data_ptr<float>() : nullptr;
          a.beta1 = (float)b1; a.beta2 = (float)b2; a.eps = (float)eps;
          a.step = step;
          a.step_dev = P<const int>(step_dev_ptr);
          a.active = active_ptr ? P<const int>(active_ptr) : bflc::current_predicate();
          a.zero_grad = zero_grad ? 1 : 0;
          check(adam ? bflc::adam_step(a, cur_stream()) : bflc::sgd_step(a, cur_stream()),
                "optim_step");
        });

  // ------------------------------------------------------------ elementwise
  m.def("cast_f32_to_bf16", [](at::Tensor src, at::Tensor dst) {
    check(bflc::cast_f32_to_bf16(src.data_ptr<float>(), dst.data_ptr(), src.numel(), cur_stream()),
          "cast_f32_to_bf16");
  });
  m.def("cast_bf16_to_f32", [](at::Tensor src, at::Tensor dst) {
    check(bflc::cast_bf16_to_f32(src.data_ptr(), dst.data_ptr<float>(), src.numel(), cur_stream()),
          "cast_bf16_to_f32");
  });
  // input preparation: u8 pixels -> bf16 (+ e4m3 and MXFP8 scale chunks); the chunked variant is
  // the flag-driven side-branch kernel of the host->device input pipeline (see k_prep_chunks)
  m.def("prep_inputs", [](at::Tensor src, const OptT& dst_bf16, const OptT& dst_q, const OptT& dst_sf,
                          double scale) {
    TORCH_CHECK(src.dim() == 2 && src.is_contiguous(), "src: contiguous u8 [R, K]");
    check(bflc::prep_inputs_u8(src.data_ptr<uint8_t>(), dst_bf16.has_value() ? dst_bf16->data_ptr() : nullptr,
                               dst_q.has_value() ? dst_q->data_ptr() : nullptr,
                               dst_sf.has_value() ? dst_sf->data_ptr<uint8_t>() : nullptr, (int)src.size(0),
                               (int)src.size(1), (float)scale, cur_stream()),
          "prep_inputs_u8");
  });
  m.def("prep_inputs_chunks", [](at::Tensor src, const OptT& dst_bf16, const OptT& dst_q, const OptT& dst_sf,
                                 int rows_per_chunk, int n_chunks, double scale, at::Tensor in_flags,
                                 at::Tensor in_seq, at::Tensor cnt, at::Tensor ready, at::Tensor err) {
    TORCH_CHECK(src.dim() == 2 && src.is_contiguous(), "src: contiguous u8 [R, K]");
    check(bflc::prep_inputs_u8_chunks(src.data_ptr<uint8_t>(), dst_bf16.has_value() ? dst_bf16->data_ptr() : nullptr,
                                      dst_q.has_value() ? dst_q->data_ptr() : nullptr,
                                      dst_sf.has_value() ? dst_sf->data_ptr<uint8_t>() : nullptr, rows_per_chunk,
                                      (int)src.size(1), n_chunks, (float)scale, in_flags.data_ptr<int32_t>(),
                                      in_seq.data_ptr<int32_t>(), reinterpret_cast<unsigned int*>(cnt.data_ptr()),
                                      reinterpret_cast<unsigned int*>(ready.data_ptr()),
                                      reinterpret_cast<unsigned int*>(err.data_ptr()), cur_stream()),
          "prep_inputs_u8_chunks");
  });
  // cudaGraphLaunch of an instantiated graph (torch.cuda.CUDAGraph.raw_cuda_graph_exec()) on a
  // given stream: the per-round launch without the stream-guard / generator bookkeeping of
  // CUDAGraph.replay() on the Python path.
  m.def("graph_launch", [](int64_t exec_ptr, int64_t stream_ptr) {
    check(cudaGraphLaunch(reinterpret_cast<cudaGraphExec_t>(static_cast<uintptr_t>(exec_ptr)),
                          reinterpret_cast<cudaStream_t>(static_cast<uintptr_t>(stream_ptr))),
          "cudaGraphLaunch");
  });
  m.def("h2d_pipeline", [](int64_t host_x, int64_t dev_x, int64_t chunk_bytes, int c_begin, int c_end,
                           int64_t host_y, int64_t dev_y, int64_t y_bytes, int64_t dev_flags,
                           int64_t host_seq, int64_t stream_ptr, bool write_value) {
    // chunks [c_begin, c_end); the labels travel with chunk 0 (y_bytes > 0).  A chunk's tag is a
    // stream-ordered 32-bit write behind its copy: cuStreamWriteValue32 (a stream memory
    // operation, no copy-engine descriptor) or, as a fallback, a 4-byte copy of *host_seq.
    using WriteFn = CUresult (*)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
    static WriteFn wv = [] {
      void* sym = nullptr;
      cudaDriverEntryPointQueryResult q;
      if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &sym, cudaEnableDefault, &q) != cudaSuccess ||
          q != cudaDriverEntryPointSuccess)
        sym = nullptr;
      return reinterpret_cast<WriteFn>(sym);
    }();
    cudaStream_t s = reinterpret_cast<cudaStream_t>(static_cast<uintptr_t>(stream_ptr));
    const uint32_t tag = static_cast<uint32_t>(*P<const int32_t>(host_seq));
    if (y_bytes > 0)
      check(cudaMemcpyAsync(P<void>(dev_y), P<const void>(host_y), (size_t)y_bytes, cudaMemcpyHostToDevice, s),
            "h2d labels");
    for (int c = c_begin; c < c_end; ++c) {
      check(cudaMemcpyAsync(P<char>(dev_x) + c * chunk_bytes, P<const char>(host_x) + c * chunk_bytes,
                            (size_t)chunk_bytes, cudaMemcpyHostToDevice, s), "h2d chunk");
      bool done = false;
      if (write_value && wv != nullptr)
        done = wv(reinterpret_cast<CUstream>(s), static_cast<CUdeviceptr>(dev_flags + 4 * c), tag, 0u) == CUDA_SUCCESS;
      if (!done)
        check(cudaMemcpyAsync(P<int32_t>(dev_flags) + c, P<const void>(host_seq), 4, cudaMemcpyHostToDevice, s),
              "h2d tag");
    }
  }, py::arg("host_x"), py::arg("dev_x"), py::arg("chunk_bytes"), py::arg("c_begin"), py::arg("c_end"),
     py::arg("host_y"), py::arg("dev_y"), py::arg("y_bytes"), py::arg("dev_flags"), py::arg("host_seq"),
     py::arg("stream_ptr"), py::arg("write_value") = true);
  m.def("cast_u8_to_bf16", [](at::Tensor src, at::Tensor dst, double scale) {
    check(bflc::cast_u8_to_bf16(src.data_ptr<uint8_t>(), dst.data_ptr(), src.numel(), (float)scale,
                                cur_stream()),
          "cast_u8_to_bf16");
  });
  m.def("quantize_fp8", [](at::Tensor src, at::Tensor dst, double inv_scale) {
    check(bflc::quantize_fp8(src.data_ptr(), reinterpret_cast<uint8_t*>(dst.data_ptr()),
                             src.numel(), (float)inv_scale, cur_stream()),
          "quantize_fp8");
  });
  m.def("amax_bf16", [](at::Tensor src, at::Tensor out) {
    check(bflc::amax_bf16(src.data_ptr(), src.numel(), out.data_ptr<float>(), cur_stream()),
          "amax_bf16");
  });
  m.def("fill_f32", [](at::Tensor dst, double v) {
    check(bflc::fill_f32(dst.data_ptr<float>(), dst.numel(), (float)v, cur_stream()), "fill_f32");
  });
  m.def("add_bf16", [](at::Tensor a, at::Tensor b, at::Tensor out) {
    check(bflc::add_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.numel(), cur_stream()),
          "add_bf16");
  });
}
