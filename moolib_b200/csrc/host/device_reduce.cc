#include "device_reduce.h"

#include <c10/cuda/CUDAGuard.h>
#include <cuda_runtime_api.h>

namespace mbh {

// ---- PyFuture ------------------------------------------------------------------------------------------------------
bool PyFuture::done() {
  if (progress) progress();
  return state->done();
}
void PyFuture::wait(double timeout) {
  auto deadline = Clock::now() + std::chrono::duration<double>(timeout < 0 ? 1e9 : timeout);
  while (true) {
    if (progress) progress();
    if (state->done()) return;
    if (Clock::now() >= deadline) return;
    {
      py::gil_scoped_release nogil;
      state->wait(progress ? 0.0002 : 0.05);
    }
    if (PyErr_CheckSignals() != 0) throw py::error_already_set();
  }
}
py::object PyFuture::get() {
  int f;
  std::string err;
  Bytes v;
  {
    std::lock_guard<std::mutex> l(state->mu);
    f = state->flags;
    err = state->error;
    if ((f & 1) && !ready) v = state->value;
  }
  if (f & 1) return ready ? *ready : decode(v);
  if (f & 2) throw std::runtime_error(err);
  if (f & 4) throw std::runtime_error("Future was cancelled");
  throw std::runtime_error("Future::get() called in invalid state");
}
py::object PyFuture::result(std::optional<double> timeout) {
  if (!done()) wait(timeout ? *timeout : -1.0);
  if (!state->done()) throw std::runtime_error("Future timed out");
  return get();
}
py::object PyFuture::exception() {
  if (progress) progress();
  std::lock_guard<std::mutex> l(state->mu);
  if (state->flags & 2) return py::module_::import("builtins").attr("RuntimeError")(state->error);
  return py::none();
}
void PyFuture::cancel() {
  keep.reset();
  state->cancel();
}

// ---- DeviceReducer -------------------------------------------------------------------------------------------------
DeviceReducer::DeviceReducer(std::shared_ptr<GroupService> service, std::shared_ptr<GroupInfo> info, std::string tag,
                             int device, uint64_t maxBytes, int nslots)
    : service_(std::move(service)), info_(std::move(info)), tag_(std::move(tag)), device_(device), maxBytes_(maxBytes),
      nslots_(nslots) {}

DeviceReducer::~DeviceReducer() {
  if (ctx_) mb_ar_ctx_destroy(ctx_);
  if (stream_) cudaStreamDestroy(stream_);
}

cudaStream_t DeviceReducer::stream() {
  if (!stream_) {
    c10::cuda::CUDAGuard g(device_);
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (cudaStreamCreateWithPriority(&stream_, cudaStreamNonBlocking, hi) != cudaSuccess) {
      cudaGetLastError();
      stream_ = nullptr;
      throw std::runtime_error("moolib_b200: cannot create the reducer stream");
    }
  }
  return stream_;
}

bool DeviceReducer::poll() {
  uint32_t cur;
  std::vector<std::string> members;
  {
    std::lock_guard<std::mutex> l(info_->mutex);
    cur = info_->syncId;
    members = info_->members;
  }
  if (cur == 0 || members.empty()) return false;
  if (cur != syncId_) {
    // new epoch: (re)create / reset the context and start the handle exchange
    connected_ = false;
    failed_ = false;
    exchange_.reset();
    auto me = std::find(members.begin(), members.end(), service_->rpc()->getName());
    if (me == members.end()) return false;
    if (members.size() > MB_AR_MAX_WORLD) {
      failed_ = true;
      error_ = "moolib_b200: the NVLink allreduce supports at most " + std::to_string(MB_AR_MAX_WORLD) +
               " members per group (one box); this group has " + std::to_string(members.size());
      syncId_ = cur;
      return false;
    }
    rank_ = (int)(me - members.begin());
    world_ = (int)members.size();
    syncId_ = cur;
    if (!ctx_) check(mb_ar_ctx_create(rank_, world_, device_, maxBytes_, nslots_, &ctx_), "mb_ar_ctx_create");
    else check(mb_ar_ctx_reset(ctx_, rank_, world_), "mb_ar_ctx_reset");
    if (world_ == 1) {
      connected_ = true;
      return true;
    }
    mb_ar_handle h;
    check(mb_ar_ctx_export(ctx_, &h), "mb_ar_ctx_export");
    Writer w;
    w.u64((uint64_t)rank_);
    w.str(std::string(reinterpret_cast<const char*>(h.bytes), sizeof(h.bytes)));
    // allgather = allreduce with concatenation (records carry their own rank)
    try {
      exchange_ = service_->allReduce(info_, "mbctx/" + tag_, w.b, [](const Bytes& a, const Bytes& b) { return a + b; });
    } catch (const std::exception& e) {
      syncId_ = 0;  // group is changing underneath us; retry on the next poll
      return false;
    }
  }
  if (connected_) return true;
  if (failed_ || !exchange_) return false;
  auto& st = *exchange_->future;
  if (!st.done()) return false;
  Bytes gathered;
  if (!(st.snapshot(&gathered, nullptr) & 1)) {
    // cancelled by a group change or timed out: a new epoch will follow
    exchange_.reset();
    syncId_ = 0;
    return false;
  }
  Reader r(gathered);
  int imported = 0;
  while (!r.done()) {
    int peer = (int)r.u64();
    std::string hb = r.str();
    if (hb.size() != sizeof(mb_ar_handle) || peer < 0 || peer >= world_) continue;
    if (peer == rank_) continue;
    mb_ar_handle h;
    std::memcpy(h.bytes, hb.data(), sizeof(h.bytes));
    int rc = mb_ar_ctx_import(ctx_, peer, &h);
    if (rc < 0) {
      failed_ = true;
      error_ = std::string("mb_ar_ctx_import: ") + mb_last_error();
      return false;
    }
    ++imported;
  }
  exchange_.reset();
  if (imported != world_ - 1) {
    failed_ = true;
    error_ = "moolib_b200: handle exchange returned " + std::to_string(imported) + " of " + std::to_string(world_ - 1) +
             " peers";
    return false;
  }
  connected_ = true;
  return true;
}

// ---- DeviceReducerSet ----------------------------------------------------------------------------------------------
std::shared_ptr<DeviceReducer> DeviceReducerSet::get(const std::string& tag, int device, uint64_t maxBytes, int nslots) {
  std::lock_guard<std::mutex> l(mu_);
  // the exchange name must be identical on every rank, so it must NOT contain the local device index
  std::string name = tag + "/" + std::to_string(maxBytes) + "/" + std::to_string(nslots);
  std::string key = name + "@" + std::to_string(device);
  auto& r = reducers_[key];
  if (!r) r = std::make_shared<DeviceReducer>(service_, info_, name, device, maxBytes, nslots);
  return r;
}

namespace {
uint64_t sizeClass(uint64_t bytes) {
  uint64_t c = 1ull << 20;
  while (c < bytes) c <<= 1;
  return c;
}

// group.all_reduce on a CUDA tensor: [connect once per (name, size class)] -> [control-plane gate: everyone has called and
// has this name's peers mapped] -> stage + K-A0 + K-A2 on the context's own stream -> event.
// Every operation NAME owns its context (its own epochs, flags, result block and stream): two differently named
// operations in flight can be started in different orders on different ranks without pairing the wrong tensors or
// queueing one gate kernel behind the other.  The control-plane gate stays (one round trip, like the reference's own
// RPC-based all_reduce): a kernel that waits for its peers is only launched once every peer is past context creation and
// cudaIpcOpenMemHandle for that name -- those calls synchronise the device, and a rank blocked in one of them behind its
// own spinning gate could never launch the kernel the other rank's gate is waiting for.
struct TensorReduceOp {
  std::shared_ptr<GroupService> service;
  std::shared_ptr<GroupInfo> info;
  std::shared_ptr<DeviceReducer> reducer;
  std::shared_ptr<FutureState> state;
  std::shared_ptr<SmallReduce> gate;
  std::string name;
  torch::Tensor tensor, flat;
  c10::cuda::CUDAStream stream;  // the caller's stream: the tensor is produced / consumed there
  cudaEvent_t ready = nullptr;   // caller's stream at call time: the tensor's contents are final
  cudaEvent_t event = nullptr;   // the kernels on the reducer's own stream have finished
  uint32_t syncId = 0;
  int phase = 0;  // 0 connecting, 1 gating, 2 kernels in flight, 3 finished
  Clock::time_point start = Clock::now();

  TensorReduceOp(c10::cuda::CUDAStream s) : stream(s) {}
  ~TensorReduceOp() {
    if (event) cudaEventDestroy(event);
    if (ready) cudaEventDestroy(ready);
  }

  void fail(const std::string& e) {
    phase = 3;
    state->setError(e);
  }

  void step() {
    if (phase == 3) return;
    try {
      if (info->syncId.load() != syncId) return fail("AllReduce operation cancelled due to a group change");
      if (phase == 0) {
        if (reducer->failed()) return fail(reducer->error());
        if (!reducer->poll()) {
          if (Clock::now() - start > std::chrono::duration<double>(service->rpc()->getTimeout()))
            return fail("AllReduce operation timed out");
          return;
        }
        Writer w;
        w.u64(1);
        gate = service->allReduce(info, "gate/" + name, w.b, [](const Bytes& a, const Bytes& b) {
          Reader ra(a), rb(b);
          Writer o;
          o.u64(ra.u64() + rb.u64());
          return o.b;
        });
        phase = 1;
      }
      if (phase == 1) {
        auto& g = *gate->future;
        if (!g.done()) return;
        {
          std::string err;
          if (!(g.snapshot(nullptr, &err) & 1)) return fail(err.empty() ? "AllReduce operation cancelled" : err);
        }
        c10::cuda::CUDAGuard dg(reducer->device());
        flat = tensor.is_contiguous() ? tensor : tensor.contiguous();
        uint64_t numel = (uint64_t)flat.numel();
        // Own stream per operation name: a gate that waits for the peers must not block the caller's stream, nor sit
        // in front of another operation's gate (two names started in opposite orders on two ranks would deadlock).
        cudaStream_t side = reducer->stream();
        if (ready) cudaStreamWaitEvent(side, ready, 0);
        mb_stream_t s = static_cast<mb_stream_t>(side);
        mb_ar_hdr hdr{1, 0, 1, 1};
        const uint32_t timeoutMs = (uint32_t)(service->rpc()->getTimeout() * 1000);
        if (flat.scalar_type() == torch::kFloat32) {
          const float* src = flat.data_ptr<float>();
          launch_counter() += check(mb_ar_stage(reducer->ctx(), 0, &src, &numel, 1, 0, 0, s), "mb_ar_stage");
          launch_counter() += check(mb_ar_reduce_gated(reducer->ctx(), 0, &hdr, /*min_batch=*/0, nullptr, nullptr, 0,
                                                       flat.data_ptr<float>(), numel, /*scale=*/0, MB_AR_ALGO_AUTO,
                                                       timeoutMs, s),
                                    "mb_ar_reduce_gated");
        } else {
          // bf16 / fp16: widened to fp32, summed in rank order, rounded once (mb_ar_reduce_gated_ex)
          void* ptr = flat.data_ptr();
          const int32_t dt = dtypeCode(flat.scalar_type());
          launch_counter() += check(mb_ar_stage_ex(reducer->ctx(), 0, &ptr, &numel, &dt, 1, 0, 0, s), "mb_ar_stage_ex");
          launch_counter() += check(mb_ar_reduce_gated_ex(reducer->ctx(), 0, &hdr, /*min_batch=*/0, &ptr, &numel, &dt,
                                                          1, nullptr, 0, /*scale=*/0, MB_AR_ALGO_AUTO, timeoutMs, s),
                                    "mb_ar_reduce_gated_ex");
        }
        if (cudaEventCreateWithFlags(&event, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventRecord(event, side) != cudaSuccess)
          return fail("moolib_b200: cudaEventRecord failed");
        phase = 2;
      }
      if (phase == 2) {
        cudaError_t e = cudaEventQuery(event);
        if (e == cudaErrorNotReady) return;
        if (e != cudaSuccess) return fail(std::string("moolib_b200: CUDA error: ") + cudaGetErrorString(e));
        int status = 0;
        mb_ar_result(reducer->ctx(), 0, nullptr, &status);
        if (status == MB_ETIMEOUT) return fail("AllReduce operation timed out");
        if (status != 0) return fail("moolib_b200: allreduce kernel failed with status " + std::to_string(status));
        check(mb_ar_slot_advance(reducer->ctx(), 0), "mb_ar_slot_advance");
        // whatever the caller enqueues next on its stream sees the result
        cudaStreamWaitEvent(stream.stream(), event, 0);
        if (!flat.is_same(tensor)) {
          c10::cuda::CUDAStreamGuard sg(stream);
          tensor.copy_(flat, true);
        }
        phase = 3;
        state->setResult(Bytes());
      }
    } catch (const std::exception& e) {
      fail(e.what());
    }
  }
};
}  // namespace

std::shared_ptr<PyFuture> DeviceReducerSet::allReduceTensor(const std::string& name, torch::Tensor t,
                                                            py::object pyTensor) {
  if (dtypeCode(t.scalar_type()) < 0)
    throw std::runtime_error("moolib_b200: all_reduce on CUDA tensors supports float32, bfloat16 and float16; got " +
                             std::string(c10::toString(t.scalar_type())));
  int device = t.get_device();
  auto op = std::make_shared<TensorReduceOp>(c10::cuda::getCurrentCUDAStream(device));
  op->service = service_;
  op->info = info_;
  op->name = name;
  op->tensor = t;
  op->state = std::make_shared<FutureState>();
  {
    c10::cuda::CUDAGuard dg(device);
    if (cudaEventCreateWithFlags(&op->ready, cudaEventDisableTiming) == cudaSuccess)
      cudaEventRecord(op->ready, op->stream.stream());
  }
  {
    std::lock_guard<std::mutex> l(info_->mutex);
    op->syncId = info_->syncId;
    auto& m = info_->members;
    if (std::find(m.begin(), m.end(), service_->rpc()->getName()) == m.end())
      throw std::runtime_error("AllReduce: local peer is not a member of the specified group!");
  }
  // at most one operation per name is in flight (GroupService rejects "all-reduce twice concurrently"); the name is
  // part of the context key so that differently named operations never share epochs
  op->reducer = get("ar:" + name, device, sizeClass((uint64_t)t.numel() * t.element_size() + 64), 1);
  {
    std::lock_guard<std::mutex> l(mu_);
    auto& slot = inflight_[name];
    if (auto prev = slot.lock())
      if (!prev->done()) throw std::runtime_error("Attempt to all-reduce twice concurrently with the name '" + name + "'");
    slot = op->state;
  }
  auto fut = std::make_shared<PyFuture>();
  fut->state = op->state;
  fut->ready = std::move(pyTensor);  // in place, like the reference (test/test_reduce.py:56)
  fut->keep = op;
  fut->progress = [op] { op->step(); };
  {
    std::lock_guard<std::mutex> l(mu_);
    std::weak_ptr<TensorReduceOp> weak = op;  // the future keeps the operation alive; a dropped future ends it
    pending_.push_back([weak] {
      auto o = weak.lock();
      if (!o) return true;
      o->step();
      return o->phase == 3;
    });
  }
  op->step();
  return fut;
}

void DeviceReducerSet::progressAll() {
  std::vector<std::function<bool()>> work;
  {
    std::lock_guard<std::mutex> l(mu_);
    if (pending_.empty()) return;
    work.swap(pending_);
  }
  std::vector<std::function<bool()>> keep;
  for (auto& f : work)
    if (!f()) keep.push_back(std::move(f));
  std::lock_guard<std::mutex> l(mu_);
  for (auto& f : keep) pending_.push_back(std::move(f));
}

}  // namespace mbh
