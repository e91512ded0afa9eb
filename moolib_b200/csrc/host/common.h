// Host layer (C++/pybind11 over torch tensors) of moolib_b200: mirrors the Python API of the reference's `moolib._C`
// for the two hot paths and calls the sm_100a kernels through the C-ABI in include/moolib_b200.h.
// torch here is the owner of device memory, streams and dtypes -- plumbing, not the product.
#pragma once

#include <pybind11/pybind11.h>
#include <pybind11/stl.h>
#include <torch/extension.h>

#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>

#include <stdexcept>
#include <string>
#include <vector>

#include "moolib_b200.h"

namespace py = pybind11;

namespace mbh {

// Throws std::runtime_error (-> Python RuntimeError, as the reference does for its own errors) on a negative code.
inline int check(int rc, const char* what) {
  if (rc < 0) {
    throw std::runtime_error(std::string(what) + ": moolib_b200 error " + std::to_string(rc) + ": " + mb_last_error());
  }
  return rc;
}

// MB_DT_* of a gradient dtype the NVLink allreduce reduces (float32, bfloat16, float16), -1 for any other
inline int32_t dtypeCode(c10::ScalarType t) {
  switch (t) {
    case c10::ScalarType::Float: return MB_DT_F32;
    case c10::ScalarType::BFloat16: return MB_DT_BF16;
    case c10::ScalarType::Half: return MB_DT_F16;
    default: return -1;
  }
}

inline mb_stream_t current_stream(int device) {
  return static_cast<mb_stream_t>(c10::cuda::getCurrentCUDAStream(device).stream());
}

// torch.Tensor <-> Python (src/tensorpython.cc:18-30 in the reference)
inline bool is_tensor(const py::handle& h) { return THPVariable_Check(h.ptr()); }
inline torch::Tensor to_tensor(const py::handle& h) { return THPVariable_Unpack(h.ptr()); }
inline py::object to_python(const torch::Tensor& t) { return py::reinterpret_steal<py::object>(THPVariable_Wrap(t)); }

// Debug aid (MOOLIB_B200_TRACE=1): the host layer records the phase it is in; a watchdog thread prints it whenever it
// has not changed for 3 s.  Costs one relaxed store per phase when disabled.
void trace_phase(const char* phase);
#define MBH_PHASE(name) ::mbh::trace_phase(name)

// Number of kernels this process launched through the host layer (bench.py's gpu_launches claim).
uint64_t& launch_counter();

// CPU tensor <-> bytes (dtype, shape, raw storage): control-plane payloads (late-joiner model sync, CPU-model sums)
std::string packTensor(const torch::Tensor& t);
torch::Tensor unpackTensor(const std::string& b);
std::string pickleDumps(const py::handle& o);
py::object pickleLoads(const std::string& b);

// Unregister control-plane handlers from a destructor that may run with the GIL held: a handler that is executing on
// the IO thread may itself be waiting for the GIL (Python reduce ops, Rpc::call), and unhandle() waits for it.
template <typename Rpc>
void unhandleAll(Rpc& rpc, std::initializer_list<std::string> names) {
  if (PyGILState_Check()) {
    py::gil_scoped_release nogil;
    for (auto& n : names) rpc.unhandle(n);
  } else {
    for (auto& n : names) rpc.unhandle(n);
  }
}

// utils::stackFields / unstackFields (reference: src/batch_utils.cc:259-325), implemented in batcher.cc
py::object stackFields(const py::tuple& input, int64_t dim);
py::tuple unstackFields(const py::handle& input, int64_t batchSize, int64_t dim);
// every tensor of a nest on `device`; pinned host tensors are read by one launch of the copy kernel (batcher.cc)
py::object nestToDevice(const py::handle& nest, const std::string& device);

void bind_batcher(py::module_& m);
void bind_accumulator(py::module_& m);
void bind_envpool(py::module_& m);
void bind_rpc(py::module_& m);
void bind_learner_ops(py::module_& m);

}  // namespace mbh
