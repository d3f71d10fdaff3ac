// pybind11 / torch bindings of the sm_100a kernel library and the symmetric-heap runtime.
// Tensors are only used as typed pointers + the current CUDA stream; all math is in
// csrc/kernels/*.cu.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <optional>

#include "bflc_kernels.h"
#include "symm_heap.hpp"

namespace py = pybind11;
using OptT = std::optional<at::Tensor>;

namespace {

void check(cudaError_t e, const char* what) {
  TORCH_CHECK(e == cudaSuccess, "bflc::", what, " failed: ", cudaGetErrorString(e));
}
cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

template <typename T>
T* opt_ptr(const OptT& t) {
  return t.has_value() ? reinterpret_cast<T*>(t->data_ptr()) : nullptr;
}
const void* raw(const at::Tensor& t) { return t.data_ptr(); }

void gemm(const at::Tensor& a, const at::Tensor& b, const OptT& d, int64_t M, int64_t N,
          int64_t K, int64_t batch, int64_t lda, int64_t ldb, int64_t a_bs, int64_t b_bs,
          bool a_mn, bool b_mn, bool is_fp8, int64_t epi_kind, int64_t d_dtype, int64_t ldd,
          int64_t d_bs, double alpha, const OptT& bias, int64_t act, const OptT& aux_out,
          const OptT& aux_in, int64_t act_bwd, const OptT& colsum, int64_t split_k,
          bool accumulate, const OptT& labels, int64_t labels_bs, double grad_scale,
          const OptT& loss_sum, const OptT& correct, const OptT& b_maps, const OptT& bias_ptrs,
          int64_t dbg_lbo_a, int64_t dbg_sbo_a, int64_t dbg_lbo_b, int64_t dbg_sbo_b,
          int64_t dyn_ptr, int64_t force_bn) {
  TORCH_CHECK(a.is_cuda() && b.is_cuda(), "gemm operands must be CUDA tensors");
  c10::cuda::CUDAGuard guard(a.device());
  bflc::GemmProblem p;
  p.M = (int)M; p.N = (int)N; p.K = (int)K; p.batch = (int)batch;
  p.ab_dtype = is_fp8 ? bflc::DType::FP8_E4M3 : bflc::DType::BF16;
  p.a = {raw(a), lda, a_bs, a_mn};
  p.b = {raw(b), ldb, b_bs, b_mn};
  p.b_maps_dev = b_maps.has_value()
                     ? reinterpret_cast<const CUtensorMap*>(b_maps->data_ptr())
                     : nullptr;
  p.dyn = reinterpret_cast<const bflc::GemmDynamic*>(static_cast<uintptr_t>(dyn_ptr));
  p.force_bn = (int)force_bn;
  auto& e = p.epi;
  e.kind = static_cast<bflc::EpiKind>(epi_kind);
  e.d = d.has_value() ? d->data_ptr() : nullptr;
  e.d_dtype = static_cast<bflc::DType>(d_dtype);
  e.ldd = ldd;
  e.d_batch_stride = d_bs;
  e.alpha = (float)alpha;
  e.bias = opt_ptr<const float>(bias);
  e.bias_ptrs = bias_ptrs.has_value()
                    ? reinterpret_cast<const float* const*>(bias_ptrs->data_ptr())
                    : nullptr;
  e.act = static_cast<bflc::Act>(act);
  e.aux_out = aux_out.has_value() ? aux_out->data_ptr() : nullptr;
  e.aux_in = aux_in.has_value() ? aux_in->data_ptr() : nullptr;
  e.act_bwd = (int)act_bwd;
  e.colsum = opt_ptr<float>(colsum);
  e.split_k = (int)split_k;
  e.accumulate = accumulate ? 1 : 0;
  e.labels = opt_ptr<const int32_t>(labels);
  e.labels_batch_stride = labels_bs;
  e.grad_scale = (float)grad_scale;
  e.loss_sum = opt_ptr<float>(loss_sum);
  e.correct = opt_ptr<unsigned int>(correct);
  p.dbg_lbo_a = (uint32_t)dbg_lbo_a; p.dbg_sbo_a = (uint32_t)dbg_sbo_a;
  p.dbg_lbo_b = (uint32_t)dbg_lbo_b; p.dbg_sbo_b = (uint32_t)dbg_sbo_b;
  const cudaError_t err = bflc::gemm_sm100(p, cur_stream());
  TORCH_CHECK(err == cudaSuccess, "bflc::gemm_sm100 failed: ", cudaGetErrorString(err), " [M=", M,
              " N=", N, " K=", K, " batch=", batch, " lda=", lda, " ldb=", ldb, " a_bs=", a_bs,
              " b_bs=", b_bs, " a_mn=", a_mn, " b_mn=", b_mn, " fp8=", is_fp8, " epi=", epi_kind,
              " d_dtype=", d_dtype, " ldd=", ldd, " split_k=", split_k, " a%16=",
              reinterpret_cast<uintptr_t>(raw(a)) % 16, " b%16=",
              reinterpret_cast<uintptr_t>(raw(b)) % 16, "]");
}

// Encode the B-operand tensor map for (ptr, N, K, ld, ...) and return its 128 raw bytes.
py::bytes gemm_b_map(int64_t ptr, int64_t N, int64_t K, int64_t ldb, bool b_mn, bool is_fp8,
                     int64_t epi_kind, int64_t force_bn) {
  bflc::GemmProblem p;
  p.M = 128; p.N = (int)N; p.K = (int)K; p.batch = 1;
  p.ab_dtype = is_fp8 ? bflc::DType::FP8_E4M3 : bflc::DType::BF16;
  p.b = {reinterpret_cast<const void*>(ptr), ldb, 0, b_mn};
  p.epi.kind = static_cast<bflc::EpiKind>(epi_kind);
  p.force_bn = (int)force_bn;
  CUtensorMap m;
  check(bflc::gemm_make_b_map(p, &m), "gemm_make_b_map");
  return py::bytes(reinterpret_cast<const char*>(&m), sizeof(m));
}

}  // namespace

void bind_extra(py::module_& m);  // defined in bindings_extra.cpp
void bind_nn(py::module_& m);     // defined in bindings_nn.cpp
void bind_mc(py::module_& m);     // defined in bindings_mc.cpp

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "bflc_demo_b200 native kernels (sm_100a)";
  m.def("gemm", &gemm, py::arg("a"), py::arg("b"), py::arg("d"), py::arg("M"), py::arg("N"),
        py::arg("K"), py::arg("batch") = 1, py::arg("lda"), py::arg("ldb"), py::arg("a_bs") = 0,
        py::arg("b_bs") = 0, py::arg("a_mn") = false, py::arg("b_mn") = false,
        py::arg("is_fp8") = false, py::arg("epi_kind") = 0, py::arg("d_dtype") = 1,
        py::arg("ldd") = 0, py::arg("d_bs") = 0, py::arg("alpha") = 1.0,
        py::arg("bias") = py::none(), py::arg("act") = 0, py::arg("aux_out") = py::none(),
        py::arg("aux_in") = py::none(), py::arg("act_bwd") = 0, py::arg("colsum") = py::none(),
        py::arg("split_k") = 1, py::arg("accumulate") = false, py::arg("labels") = py::none(),
        py::arg("labels_bs") = 0, py::arg("grad_scale") = 1.0, py::arg("loss_sum") = py::none(),
        py::arg("correct") = py::none(), py::arg("b_maps") = py::none(),
        py::arg("bias_ptrs") = py::none(), py::arg("dbg_lbo_a") = 0, py::arg("dbg_sbo_a") = 0,
        py::arg("dbg_lbo_b") = 0, py::arg("dbg_sbo_b") = 0, py::arg("dyn_ptr") = 0,
        py::arg("force_bn") = 0);
  m.def("gemm2", [](const at::Tensor& a, const at::Tensor& b, at::Tensor d, int64_t M, int64_t N,
                    int64_t K, int64_t lda, int64_t ldb, double alpha, const OptT& bias, int64_t act) {
    bflc::GemmProblem p;
    p.M = (int)M; p.N = (int)N; p.K = (int)K;
    p.a = {raw(a), lda, 0, false};
    p.b = {raw(b), ldb, 0, false};
    p.epi.d = d.data_ptr();
    p.epi.d_dtype = d.scalar_type() == at::kFloat ? bflc::DType::F32 : bflc::DType::BF16;
    p.epi.ldd = d.stride(0);
    p.epi.alpha = (float)alpha;
    p.epi.bias = opt_ptr<const float>(bias);
    p.epi.act = static_cast<bflc::Act>(act);
    check(bflc::gemm2_sm100(p, cur_stream()), "gemm2_sm100");
  });
  m.def("gemm_b_map", &gemm_b_map);
  m.def("gemm_pick_bn", [](int64_t N, int64_t kind, int64_t M, int64_t z) {
    return bflc::gemm_pick_bn((int)N, static_cast<bflc::EpiKind>(kind), (int)M, (int)z);
  });
  m.def("launch_count", [] { return bflc::launch_count(); });
  bind_extra(m);
  bind_nn(m);
  bind_mc(m);
}
