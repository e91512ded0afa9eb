// Accumulator (HP-A host side): moolib's gradient accumulation / model-sync state machine with the data plane replaced
// by the sm_100a kernels.
//
// Mirrors AccumulatorImpl (reference: src/accumulator.cc:150-1192; bound at src/moolib.cc:1695-1862): same methods, same
// asynchronous contract (results are applied only inside update(), src/accumulator.cc:508-551), same virtual-batch gate
// (count allreduce, :1035-1078), leader election by max (modelVersion, name) (:581-625), late-joiner model/state sync
// (:464-488, :719-836).  What changes for CUDA parameters:
//   gradients LIVE in the NVLink staging memory: every parameter's .grad is a view into the slot's current ring buffer
//                       (mb_ar_buffer), so backward() writes where the peers read and reduce_gradients() launches NO
//                       stage kernel (reference: 36 D2H copy_ + 36 zero_, :941-980, :410-418, and a stream synchronize
//                       :937).  A foreign .grad (assigned by the user) or a second local contribution before the gate
//                       opens is folded in by ONE K-A1 launch.
//   the virtual-batch gate is evaluated ON THE DEVICE (K-A0, one warp) right behind the backward pass -- no count
//                       allreduce over the control plane (:1035-1078) and no extra update() tick -- and is followed
//                       stream-ordered by ONE K-A2 launch that pulls every peer's staging over NVLink, sums in rank
//                       order, multiplies by 1.0f/numGradients and writes the slot's result buffer, which .grad is
//                       pointed at when update() applies the result (reference: RPC tree src/group.h:570-654, 36 H2D
//                       copy_ + 36 mul_ :441-442, stream synchronize :450).
// MOOLIB_B200_STRICT_COUNTING=0 restores the reference's accumulate-while-counting with the count on the control plane.
// CPU parameters (BASELINE.json config 0, "plumbing, no GPU") reduce over the control plane in member order.
#include "common.h"
#include "control.h"
#include "device_reduce.h"

#include <ATen/ATen.h>

#include <set>
#include <cuda_runtime_api.h>

namespace mbh {

namespace {

struct ReduceSlot {
  size_t index = 0;
  uint32_t syncId = 0;
  mb_ar_hdr data{0, 0, 0, 0};  // numGradients, numSkipped, batchSize, has_grads (something is staged)
  bool isCounting = false, wantsMoreCounting = false, wantsReduce = false, reduceStarted = false, reduceDone = false;
  std::shared_ptr<SmallReduce> countOp;
  std::shared_ptr<SmallReduce> reduceOp;   // CPU-parameter path
  std::vector<torch::Tensor> cpuStaging;   // CPU-parameter path (src/accumulator.cc:847-874)
  cudaEvent_t event = nullptr;             // device path: completion of the K-A2 launch
  cudaEvent_t staged = nullptr;            // device path: this slot's gradients are complete (compute stream)
  bool kernelInFlight = false;
  void* resultBase = nullptr;              // device gate: where K-A2 leaves the averaged gradients (flat layout)
  bool gated = false;                      // the in-flight launch is K-A0 + K-A2 (mb_ar_reduce_gated)
  Clock::time_point reduceStart;
  ~ReduceSlot() {
    for (cudaEvent_t e : {event, staged})
      if (e) cudaEventDestroy(e);
  }
};

Bytes packU64(uint64_t v) {
  Writer w;
  w.u64(v);
  return w.b;
}

// CPU-path payload = AccumulatorReductionType (src/group.h:195-218)
Bytes packReduction(const mb_ar_hdr& h, const std::vector<torch::Tensor>& grads) {
  Writer w;
  w.u64(h.num_gradients);
  w.u64(h.num_skipped);
  w.u64(h.batch_size);
  w.u32((uint32_t)grads.size());
  for (auto& g : grads) w.str(packTensor(g));
  return w.b;
}
struct Reduction {
  mb_ar_hdr h{0, 0, 0, 0};
  std::vector<torch::Tensor> grads;
};
Reduction unpackReduction(const Bytes& b) {
  Reader r(b);
  Reduction x;
  x.h.num_gradients = r.u64();
  x.h.num_skipped = r.u64();
  x.h.batch_size = r.u64();
  uint32_t n = r.u32();
  for (uint32_t i = 0; i < n; ++i) x.grads.push_back(unpackTensor(r.str()));
  return x;
}
// AccumulatorReductionType::add (src/group.h:201-212)
Bytes addReductions(const Bytes& a, const Bytes& b) {
  Reduction x = unpackReduction(a), n = unpackReduction(b);
  if (n.grads.size() == x.grads.size()) {
    for (size_t i = 0; i < x.grads.size(); ++i) x.grads[i] += n.grads[i];
  } else if (n.grads.size() > x.grads.size()) {
    std::swap(x.grads, n.grads);
  }
  x.h.num_gradients += n.h.num_gradients;
  x.h.num_skipped += n.h.num_skipped;
  x.h.batch_size += n.h.batch_size;
  return packReduction(x.h, x.grads);
}

py::object deepCopyToCpu(const py::handle& v) {
  if (py::isinstance<py::dict>(v)) {
    py::dict d;
    for (auto kv : py::reinterpret_borrow<py::dict>(v)) d[deepCopyToCpu(kv.first)] = deepCopyToCpu(kv.second);
    return std::move(d);
  }
  if (py::isinstance<py::list>(v)) {
    py::list src = py::reinterpret_borrow<py::list>(v), dst(src.size());
    for (size_t i = 0; i < src.size(); ++i) dst[i] = deepCopyToCpu(src[i]);
    return std::move(dst);
  }
  if (is_tensor(v)) return to_python(to_tensor(v).to(torch::kCPU, /*non_blocking=*/false, /*copy=*/true));
  if (py::isinstance<py::tuple>(v)) {
    py::tuple src = py::reinterpret_borrow<py::tuple>(v), dst(src.size());
    for (size_t i = 0; i < src.size(); ++i) dst[i] = deepCopyToCpu(src[i]);
    return std::move(dst);
  }
  return py::reinterpret_borrow<py::object>(v);
}

}  // namespace

class Accumulator {
 public:
  Accumulator(std::string name, py::object parameters, py::object buffers, py::object group) {
    if (group.is_none()) {
      shouldUpdateGroup_ = true;
      ownGroup_ = makeOwnGroup(name);
      parts_ = groupPartsOf(ownGroup_);
      resName_ = name + "::accumulator";
    } else {
      ownGroup_ = group;
      parts_ = groupPartsOf(group);
      resName_ = parts_.info->name + "::" + name;
    }
    myName_ = parts_.rpc->getName();
    slots_.resize(1);
    for (auto v : parameters) {
      if (!is_tensor(v)) throw std::runtime_error("Accumulator parameter is not a Tensor!");
      torch::Tensor t = to_tensor(v);
      gradsOnCuda_ |= t.is_cuda();
      if (t.is_cuda()) device_ = t.get_device();
      params_.push_back(t);
    }
    for (auto v : buffers) {
      if (!is_tensor(v)) throw std::runtime_error("Accumulator buffer is not a Tensor!");
      buffers_.push_back(to_tensor(v));
    }
    if (gradsOnCuda_) {
      for (auto& p : params_) {
        if (!p.requires_grad()) continue;
        if (!p.is_cuda() || p.get_device() != device_ || dtypeCode(p.scalar_type()) < 0)
          throw std::runtime_error(
              "moolib_b200.Accumulator: CUDA parameters must all be on one device and of dtype float32, bfloat16 or "
              "float16 (mixed is fine); got " + std::string(c10::toString(p.scalar_type())) + " on " +
              p.device().str());
      }
    }
    ensureGrads();
    setupHandlers();
  }

  ~Accumulator() {
    try {
      releaseGradViews();
    } catch (...) {
    }
    if (arStream_) cudaStreamDestroy(arStream_);
    unhandleAll(*parts_.rpc, {"Acc::requestModel/" + resName_, "Acc::modelUpdate/" + resName_,
                              "Acc::buffersUpdate/" + resName_, "Acc::modelFetched/" + resName_});
  }

  void connect(const std::string& address) { parts_.rpc->connect(address); }

  // ---- predicates (src/accumulator.cc:372-405) -------------------------------------------------------------------
  bool connectedImpl() {
    bool groupActive;
    {
      std::lock_guard<std::mutex> l(parts_.info->mutex);
      groupActive = !parts_.info->members.empty();
    }
    return groupActive && !members_.empty() && (hasReceivedModel_ || syncLeader_ == myName_);
  }
  bool connected() {
    std::lock_guard<std::mutex> l(mu_);
    return connectedImpl();
  }
  bool wantsState() {
    std::lock_guard<std::mutex> l(mu_);
    return wantsUserState_;
  }
  bool hasNewState() { return hasNewUserState_; }
  bool hasGradients() {
    std::lock_guard<std::mutex> l(mu_);
    return hasGradients_;
  }
  bool wantsGradientsAtIndex(size_t i) {
    auto& v = slots_.at(i);
    if (!v || v->reduceDone) return true;
    if (v->reduceStarted) return false;
    // One contribution (or skip) per count round.  The reference keeps asking for gradients while a count is in flight
    // (src/accumulator.cc:398-404, 984-988 wantsMoreCounting), so a fast loop squeezes extra batches into every
    // reduction and the virtual batch size overshoots (measured: 2.7x at 8 peers).  Holding back until the count returns
    // keeps reductions at the configured size; MOOLIB_B200_STRICT_COUNTING=0 restores the reference behaviour.
    if (strictCounting_ && v->isCounting) return false;
    return true;
  }
  bool anyKernelInFlight() {
    for (auto& v : slots_)
      if (v && v->kernelInFlight) return true;
    return false;
  }
  bool wantsGradientsLocked() {
    // Host-counted CUDA path (MOOLIB_B200_STRICT_COUNTING=0): its K-A2 writes the .grad tensors themselves, so no new
    // backward may start while any slot's kernel is in flight (set_parallel_gradients(n>1) would otherwise race with it).
    if (gradsOnCuda_ && !deviceGate() && anyKernelInFlight()) return false;
    return connectedImpl() && wantsGradientsAtIndex(nextIndex_) && !isWaitingForModel_ && !isFindingLeader_ &&
           !hasGradients_ && (!gradsOnCuda_ || reducerReady_);
  }
  bool deviceGate() const { return gradsOnCuda_ && strictCounting_; }
  bool wantsGradients() {
    std::lock_guard<std::mutex> l(mu_);
    return wantsGradientsLocked();
  }

  // ---- gradients -------------------------------------------------------------------------------------------------
  // .grad of every parameter that requires grad, created (zeros) if missing (src/accumulator.cc:857-866)
  std::vector<torch::Tensor> ensureGrads() {
    torch::NoGradGuard ng;
    std::vector<torch::Tensor> r;
    for (auto& p : params_) {
      if (!p.requires_grad()) continue;
      torch::Tensor g = p.mutable_grad();
      if (!g.defined()) {
        g = torch::zeros_like(p);
        p.mutable_grad() = g;
      }
      if (gradsOnCuda_ && (!g.is_contiguous() || g.scalar_type() != p.scalar_type())) {
        g = g.contiguous().to(p.scalar_type());
        p.mutable_grad() = g;
      }
      r.push_back(g);
    }
    return r;
  }

  void actuallyZeroGradients() {
    torch::NoGradGuard ng;
    std::vector<torch::Tensor> gs;
    for (auto& p : params_) {
      torch::Tensor g = p.mutable_grad();
      if (g.defined()) {
        g.detach_();
        gs.push_back(g);
      }
    }
    if (!gs.empty()) at::_foreach_zero_(gs);
  }

  void zeroGradients() {
    std::lock_guard<std::mutex> l(mu_);
    hasGradients_ = false;
    if (deviceGate() && reducerReady_ && arena_) {
      torch::NoGradGuard ng;
      c10::cuda::CUDAGuard dg(device_);
      GradViews& av = viewsOf(accumBase(nextIndex_));
      if (gradsAre(av) || (appliedBase_ && gradsAre(viewsOf(appliedBase_)))) {
        // .grad shows an applied result (or is already accumulating): (back) to the accumulation buffer, zero-filled by
        // ONE memset of the flat buffer (reference: 36 zero_ launches, src/accumulator.cc:410-418)
        cudaMemsetAsync(av.base, 0, (size_t)arena_->total, c10::cuda::getCurrentCUDAStream(device_).stream());
        pointGradsAt(av);
      } else {
        actuallyZeroGradients();
      }
      appliedBase_ = nullptr;
      return;
    }
    actuallyZeroGradients();
  }

  // ---- gradient arena (device gate path): .grad tensors are views into the symmetric ring / the result buffers ----
  struct GradViews {
    void* base = nullptr;
    std::vector<torch::Tensor> v;  // one per parameter that requires grad, same order as ensureGrads()
  };
  struct GradArena {
    std::vector<uint64_t> numel, off;  // off: bytes, the flat layout of mb_ar_layout (dtype runs, 16 B aligned tensors)
    std::vector<int32_t> dtype;        // MB_DT_*
    std::vector<c10::ScalarType> type;
    std::vector<std::vector<int64_t>> sizes;
    int64_t total = 0;                 // padded bytes
    std::map<void*, GradViews> views;
    std::vector<torch::Tensor> result;  // per slot: where K-A2 writes (local memory, flat layout)
  };

  GradArena& arena() {
    if (!arena_) {
      arena_ = std::make_unique<GradArena>();
      for (auto& p : params_) {
        if (!p.requires_grad()) continue;
        arena_->numel.push_back((uint64_t)p.numel());
        arena_->dtype.push_back(dtypeCode(p.scalar_type()));
        arena_->type.push_back(p.scalar_type());
        arena_->sizes.emplace_back(p.sizes().begin(), p.sizes().end());
      }
      arena_->off.resize(arena_->numel.size());
      uint64_t total = 0;
      if (!arena_->numel.empty())
        check(mb_ar_layout(arena_->numel.data(), arena_->dtype.data(), (int)arena_->numel.size(), arena_->off.data(),
                           &total, nullptr),
              "mb_ar_layout");
      arena_->total = (int64_t)total;
      c10::cuda::CUDAGuard dg(device_);
      for (size_t i = 0; i < slots_.size(); ++i)
        arena_->result.push_back(torch::empty({std::max<int64_t>(arena_->total, 16)}, torch::dtype(torch::kUInt8).device(torch::kCUDA, device_)));
    }
    return *arena_;
  }

  GradViews& viewsOf(void* base) {
    GradArena& a = arena();
    auto it = a.views.find(base);
    if (it != a.views.end()) return it->second;
    GradViews& gv = a.views[base];
    gv.base = base;
    for (size_t i = 0; i < a.numel.size(); ++i)
      gv.v.push_back(torch::from_blob(static_cast<char*>(base) + a.off[i], a.sizes[i],
                                      torch::dtype(a.type[i]).device(torch::kCUDA, device_)));
    return gv;
  }

  bool gradsAre(const GradViews& gv) {
    size_t i = 0;
    for (auto& p : params_) {
      if (!p.requires_grad()) continue;
      const torch::Tensor& g = p.grad();
      if (!g.defined() || g.data_ptr() != gv.v[i].data_ptr() || g.scalar_type() != gv.v[i].scalar_type() ||
          !g.is_contiguous())
        return false;
      ++i;
    }
    return true;
  }

  void pointGradsAt(GradViews& gv) {
    size_t i = 0;
    for (auto& p : params_) {
      if (!p.requires_grad()) continue;
      p.mutable_grad() = gv.v[i++];
    }
  }

  bool slotHoldsData(size_t j) {
    auto& v = slots_[j];
    return v && !v->reduceDone && v->data.has_grads != 0;
  }
  // Where the next contribution for slot j is accumulated: the slot's staging itself while it is empty (zero-copy: the
  // peers will read exactly what backward() wrote), else the next ring buffer (folded in by K-A1).
  void* accumBase(size_t j) { return mb_ar_buffer(reducer()->ctx(), (int)j, slotHoldsData(j) ? 1 : 0); }

  // Point .grad at the accumulation buffer of the slot that the next reduce_gradients() call fills.
  void repointForAccumulation() {
    c10::cuda::CUDAGuard dg(device_);
    GradViews& av = viewsOf(accumBase(nextIndex_));
    if (gradsAre(av)) return;  // already there (and clean: K-A1 zeroes its sources)
    cudaMemsetAsync(av.base, 0, (size_t)arena().total, c10::cuda::getCurrentCUDAStream(device_).stream());
    pointGradsAt(av);
  }

  bool gradsInArena() {
    if (!arena_) return false;
    for (auto& kv : arena_->views)
      if (gradsAre(kv.second)) return true;
    return false;
  }

  // Give every parameter an ordinary .grad tensor again (same values): before the arena's memory goes away.
  void releaseGradViews() {
    if (!arena_) return;
    torch::NoGradGuard ng;
    if (gradsInArena()) {
      for (auto& p : params_) {
        if (!p.requires_grad() || !p.grad().defined()) continue;
        p.mutable_grad() = p.grad().clone();
      }
    }
    arena_.reset();
    appliedBase_ = nullptr;
  }

  uint64_t flatBytes(const std::vector<torch::Tensor>& gs) {
    std::vector<uint64_t> n;
    std::vector<int32_t> d;
    for (auto& g : gs) {
      n.push_back((uint64_t)g.numel());
      d.push_back(dtypeCode(g.scalar_type()));
    }
    uint64_t total = 0;
    if (!n.empty()) check(mb_ar_layout(n.data(), d.data(), (int)n.size(), nullptr, &total, nullptr), "mb_ar_layout");
    return total;
  }
  // (pointers, numel, MB_DT_*) of a gradient list for the _ex entry points
  struct ListEx {
    std::vector<void*> ptrs;
    std::vector<uint64_t> numel;
    std::vector<int32_t> dtype;
  };
  static ListEx listEx(const std::vector<torch::Tensor>& gs) {
    ListEx l;
    for (auto& g : gs) {
      l.ptrs.push_back(g.data_ptr());
      l.numel.push_back((uint64_t)g.numel());
      l.dtype.push_back(dtypeCode(g.scalar_type()));
    }
    return l;
  }

  std::shared_ptr<DeviceReducer> reducer() {
    if (!reducer_) {
      auto gs = ensureGrads();
      // big enough for the gradient set AND for the publish region that carries parameters + buffers to late joiners
      reducer_ = parts_.reducers->get("acc/" + resName_, device_, std::max<uint64_t>({flatBytes(gs), modelFlatBytes(), 16}),
                                      (int)slots_.size());
    }
    return reducer_;
  }

  // reference: reduceImpl, src/accumulator.cc:880-1003
  void reduceImpl(int batchSize) {
    MBH_PHASE("reduceImpl:enter");
    std::lock_guard<std::mutex> l(mu_);
    MBH_PHASE("reduceImpl:locked");
    if (!wantsGradientsLocked())
      throw std::runtime_error("reduceGradients/skipGradients called while wantsGradients() is false");
    size_t index = nextIndex_;
    std::shared_ptr<ReduceSlot> target = slots_[index];
    if (target && target->reduceStarted && !target->reduceDone)
      throw std::runtime_error("reduceImpl internal error, reduce already started!");
    if (!target || target->reduceDone) {
      auto fresh = std::make_shared<ReduceSlot>();
      if (target) {  // keep the CUDA events (creating four per round costs more than the gate kernel)
        std::swap(fresh->event, target->event);
        std::swap(fresh->staged, target->staged);
      }
      target = slots_[index] = fresh;
      target->index = index;
    }
    nextIndex_ = (nextIndex_ == slots_.size() - 1) ? 0 : nextIndex_ + 1;
    target->syncId = hSyncId_;
    torch::NoGradGuard ng;
    if (batchSize) {
      ++target->data.num_gradients;
      target->data.batch_size += (uint64_t)batchSize;
      auto gs = ensureGrads();
      const bool add = target->data.has_grads != 0;
      if (gradsOnCuda_) {
        c10::cuda::CUDAGuard dg(device_);
        const bool zeroCopy = deviceGate() && !add && gradsAre(viewsOf(mb_ar_buffer(reducer()->ctx(), (int)index, 0)));
        if (!zeroCopy) {
          // K-A1: staging (=|+=) grads and grads <- 0 in one launch, ordered after backward() on the current stream
          // (a user-assigned .grad, or another local contribution while the gate is still closed)
          ListEx l = listEx(gs);
          launch_counter() += check(mb_ar_stage_ex(reducer()->ctx(), (int)index, l.ptrs.data(), l.numel.data(),
                                                   l.dtype.data(), (int)gs.size(), add ? 1 : 0, /*zero_src=*/1,
                                                   current_stream(device_)),
                                    "Accumulator.reduce_gradients");
          ++stageLaunches_;
        } else {
          ++zeroCopyRounds_;
        }
      } else {
        if (!add) {
          target->cpuStaging.clear();
          for (auto& g : gs) target->cpuStaging.push_back(g.detach().clone());
        } else {
          for (size_t i = 0; i < gs.size(); ++i) target->cpuStaging[i].add_(gs[i]);
        }
        actuallyZeroGradients();
      }
      target->data.has_grads = 1;
    } else {
      ++target->data.num_skipped;
    }
    if (gradsOnCuda_) {
      c10::cuda::CUDAGuard dg(device_);
      if (deviceGate()) repointForAccumulation();
      if (!target->staged) cudaEventCreateWithFlags(&target->staged, cudaEventDisableTiming);
      cudaEventRecord(target->staged, c10::cuda::getCurrentCUDAStream(device_).stream());
    }
    if (target->syncId == hSyncId_ && target->syncId == parts_.info->syncId.load()) {
      if (deviceGate()) startGatedReduce(target);
      else if (target->isCounting) target->wantsMoreCounting = true;
      else startCount(target);
    }
    MBH_PHASE("idle");
  }
  void reduceGradients(int batchSize) { reduceImpl(batchSize); }
  void skipGradients() { reduceImpl(0); }

  cudaStream_t reduceStream() {
    // K-A0/K-A2 run on their own high-priority stream, ordered only after the slot's gradients are complete: they must
    // not queue behind actor-inference work the loop has enqueued on the compute stream since then (tens of ms at 256
    // envs), because every peer's round waits for the slowest rank to reach its gate.
    if (!arStream_) {
      int lo = 0, hi = 0;
      cudaDeviceGetStreamPriorityRange(&lo, &hi);
      if (cudaStreamCreateWithPriority(&arStream_, cudaStreamNonBlocking, hi) != cudaSuccess) arStream_ = nullptr;
    }
    return arStream_ ? arStream_ : c10::cuda::getCurrentCUDAStream(device_).stream();
  }

  // Device gate (replaces startCount + startReduce, src/accumulator.cc:1005-1078): K-A0 sums every peer's
  // {numGradients, numSkipped, batchSize} over NVLink and opens the gate when sum(batchSize) >= virtualBatchSize; K-A2
  // follows on the same stream and reduces into the slot's result buffer, or returns at once when the gate stayed shut.
  void startGatedReduce(const std::shared_ptr<ReduceSlot>& target) {
    MBH_PHASE("startGatedReduce");
    c10::cuda::CUDAGuard dg(device_);
    GradArena& a = arena();
    cudaStream_t stream = reduceStream();
    if (target->staged) cudaStreamWaitEvent(stream, target->staged, 0);
    if (!target->event) cudaEventCreateWithFlags(&target->event, cudaEventDisableTiming);
    target->isCounting = true;
    target->gated = true;
    target->reduceStart = Clock::now();
    // Two-shot (large gradient sets, N > 2): its all-gather leaves the averaged gradients in every rank's staging
    // buffer, so the result is consumed IN PLACE (.grad will point at this ring position) and the kernel skips its
    // final local copy.  One-shot writes the slot's separate result buffer (peers are still reading the staging).
    const int algo = mb_ar_algo_for(reducer()->ctx(), (uint64_t)a.total);
    target->resultBase = algo == MB_AR_ALGO_TWOSHOT ? mb_ar_buffer(reducer()->ctx(), (int)target->index, 0)
                                                    : a.result[target->index].data_ptr();
    // an all-fp32 model runs exactly mb_ar_reduce_gated (flat destination of a.total / 4 floats)
    launch_counter() += check(
        mb_ar_reduce_gated_ex(reducer()->ctx(), (int)target->index, &target->data, virtualBatchSize_, nullptr,
                              a.numel.data(), a.dtype.data(), (int)a.numel.size(), target->resultBase,
                              (uint64_t)a.total, /*scale=*/1, algo, (uint32_t)(parts_.rpc->getTimeout() * 1000),
                              static_cast<mb_stream_t>(stream)),
        "Accumulator gated allreduce");
    cudaEventRecord(target->event, stream);
    target->kernelInFlight = true;
  }

  // reference: startCount, src/accumulator.cc:1035-1078 (host-counted path: CPU parameters, MOOLIB_B200_STRICT_COUNTING=0)
  void startCount(const std::shared_ptr<ReduceSlot>& target) {
    MBH_PHASE("startCount");
    if (target->syncId != hSyncId_ || target->syncId != parts_.info->syncId.load()) return;
    target->isCounting = true;
    try {
      target->countOp = parts_.service->allReduce(
          parts_.info, "Accumulator reduce size " + std::to_string(target->index) + "/" + resName_,
          packU64(target->data.batch_size), [](const Bytes& a, const Bytes& b) {
            Reader ra(a), rb(b);
            return packU64(ra.u64() + rb.u64());
          });
    } catch (const std::exception&) {
      target->isCounting = false;
      onError();
    }
  }

  // reference: startReduce, src/accumulator.cc:1005-1033
  void startReduce(const std::shared_ptr<ReduceSlot>& target) {
    MBH_PHASE("startReduce");
    if (target->syncId != hSyncId_ || target->syncId != parts_.info->syncId.load()) return;
    target->reduceStarted = true;
    target->reduceStart = Clock::now();
    torch::NoGradGuard ng;
    if (gradsOnCuda_) {
      auto gs = ensureGrads();
      ListEx l = listEx(gs);
      c10::cuda::CUDAGuard dg(device_);
      // Host-counted path: K-A2 (with its in-kernel barrier) writes the .grad tensors themselves.  Safe: every backward
      // pass that contributed was followed by its stage kernel in the same reduce_gradients() call, no new backward is
      // allowed while a kernel is in flight (wantsGradientsLocked), and the compute stream waits for the kernel before
      // has_gradients() turns true.
      cudaStream_t stream = reduceStream();
      if (target->staged) cudaStreamWaitEvent(stream, target->staged, 0);
      // K-A2: barrier + P2P reduce + 1/numGradients scale + scatter into the .grad tensors, one launch
      launch_counter() += check(
          mb_ar_allreduce_ex(reducer()->ctx(), (int)target->index, &target->data, l.ptrs.data(), l.numel.data(),
                             l.dtype.data(), (int)gs.size(), nullptr, 0, /*scale=*/1, MB_AR_ALGO_AUTO,
                             (uint32_t)(parts_.rpc->getTimeout() * 1000), static_cast<mb_stream_t>(stream)),
          "Accumulator allreduce");
      if (!target->event) cudaEventCreateWithFlags(&target->event, cudaEventDisableTiming);
      cudaEventRecord(target->event, stream);
      target->kernelInFlight = true;
      target->gated = false;
    } else {
      try {
        target->reduceOp = parts_.service->allReduce(
            parts_.info, "Accumulator reduce " + std::to_string(target->index) + "/" + resName_,
            packReduction(target->data, target->data.has_grads ? target->cpuStaging : std::vector<torch::Tensor>{}),
            addReductions);
      } catch (const std::exception&) {
        onError();
      }
    }
  }

  // reference: setGradients, src/accumulator.cc:425-462 (CPU path; on the device path the kernel already did it)
  void finishReduce(const std::shared_ptr<ReduceSlot>& target, const mb_ar_hdr& total) {
    target->reduceDone = true;
    ++modelVersion_;
    stats_ = total;
    hasGradients_ = true;
  }

  // Runs the pending "result closure" of the slot whose turn it is; reference: checkGradientResultCallback (:508-517)
  void checkGradientResult() {
    auto& v = slots_[nextResultIndex_];
    if (!v) return;
    bool ran = false;
    if (v->countOp && v->countOp->future->done()) {
      auto op = std::move(v->countOp);
      v->countOp.reset();
      // the slot keeps its turn: the count only opens (or not) the gate, the round ends with the reduction's result
      Bytes value;
      const int flags = op->future->snapshot(&value, nullptr);  // no lock held while we start the next operation
      if (flags & 1) {
        Reader r(value);
        uint64_t size = r.u64();
        if (size >= virtualBatchSize_) {
          if (v->syncId == hSyncId_ && v->syncId == parts_.info->syncId.load()) {
            v->wantsReduce = true;
            startReduce(v);
          }
        } else {
          v->isCounting = false;
          if (v->wantsMoreCounting) startCount(v);
        }
      } else {
        onError();
      }
    } else if (v->kernelInFlight) {
      cudaError_t e = cudaEventQuery(v->event);
      if (e != cudaErrorNotReady) {
        v->kernelInFlight = false;
        ran = true;
        mb_ar_hdr total;
        int status = 0;
        mb_ar_result(reducer()->ctx(), (int)v->index, &total, &status);
        if (e != cudaSuccess || status < 0) {
          lastError_ = e != cudaSuccess ? std::string(cudaGetErrorString(e))
                                        : (status == MB_ETIMEOUT ? "allreduce barrier timed out" : "allreduce failed");
          v->reduceDone = true;  // abandon the round; the resync resets the slots
          onError();
        } else if (v->gated && status == MB_AR_SHORT) {
          // gate closed (src/accumulator.cc:1051): keep accumulating; the next reduce/skip call counts again
          ran = false;
          v->isCounting = false;
          ++shortRounds_;
          recordTiming(*v, /*reduced=*/false);
        } else {
          // later work on the compute stream (clip_grad_norm_, optimizer.step) is ordered after the kernel
          c10::cuda::CUDAGuard dg(device_);
          cudaStreamWaitEvent(c10::cuda::getCurrentCUDAStream(device_).stream(), v->event, 0);
          if (v->gated) {
            v->reduceStarted = true;
            recordTiming(*v, /*reduced=*/true);
            check(mb_ar_slot_advance(reducer()->ctx(), (int)v->index), "mb_ar_slot_advance");
            torch::NoGradGuard ng;
            pointGradsAt(viewsOf(v->resultBase));
            appliedBase_ = v->resultBase;
          }
          finishReduce(v, total);
        }
      }
    } else if (v->reduceOp && v->reduceOp->future->done()) {
      auto op = std::move(v->reduceOp);
      v->reduceOp.reset();
      ran = true;
      Bytes value;
      const int flags = op->future->snapshot(&value, nullptr);
      if (flags & 1) {
        torch::NoGradGuard ng;
        Reduction red = unpackReduction(value);
        if (red.grads.empty()) {
          actuallyZeroGradients();
        } else if (red.h.num_gradients) {
          auto gs = ensureGrads();
          if (gs.size() != red.grads.size()) throw std::runtime_error("grads shrank?");
          for (size_t i = 0; i < gs.size(); ++i) {
            gs[i].copy_(red.grads[i], true);
            gs[i].mul_(1.0f / red.h.num_gradients);
          }
        }
        red.h.has_grads = red.grads.empty() ? 0 : 1;
        finishReduce(v, red.h);
      } else {
        onError();
      }
    }
    if (ran) nextResultIndex_ = (nextResultIndex_ == slots_.size() - 1) ? 0 : nextResultIndex_ + 1;
  }

  void onError() {
    if (hSyncId_ == parts_.info->syncId.load()) resync();
  }
  void resync() {
    std::lock_guard<std::mutex> l(parts_.info->mutex);
    parts_.service->resync(*parts_.info);
  }

  // ---- model / state sync (src/accumulator.cc:464-488, 713-836) --------------------------------------------------
  void setupHandlers() {
    parts_.rpc->handle("Acc::requestModel/" + resName_, [this](const std::string&, const Bytes& p) {
      Reader r(p);
      uint32_t syncId = r.u32();
      std::string peer = r.str();
      const bool viaNvlink = !r.done() && r.u32() != 0;  // the requester has this leader's publish region mapped
      std::lock_guard<std::mutex> l(netMu_);
      if (syncId != netSyncId_) return;
      if (std::find(requestedModelUpdate_.begin(), requestedModelUpdate_.end(), peer) == requestedModelUpdate_.end())
        requestedModelUpdate_.push_back(peer);
      if (viaNvlink) requestedViaNvlink_.insert(peer);
      else requestedViaNvlink_.erase(peer);
    });
    parts_.rpc->handle("Acc::modelFetched/" + resName_, [this](const std::string&, const Bytes& p) {
      Reader r(p);
      uint32_t syncId = r.u32();
      std::string peer = r.str();
      std::lock_guard<std::mutex> l(netMu_);
      if (syncId == netSyncId_) publishPending_.erase(peer);
    });
    parts_.rpc->handle("Acc::modelUpdate/" + resName_, [this](const std::string&, const Bytes& p) {
      Reader r(p);
      uint32_t syncId = r.u32();
      const uint32_t kind = r.u32();
      const bool regular = (kind & 1u) != 0;
      const bool viaNvlink = (kind & 2u) != 0;  // float CUDA tensors wait in the sender's publish region
      int64_t version = r.i64();
      uint32_t np = r.u32();
      std::vector<Bytes> ps(np);
      for (auto& x : ps) x = r.str();
      uint32_t nb = r.u32();
      std::vector<Bytes> bs(nb);
      for (auto& x : bs) x = r.str();
      Bytes state = r.str();
      std::lock_guard<std::mutex> l(netMu_);
      if (syncId != netSyncId_) return;
      if (regular && version != netModelVersion_ && !netWaitingForModel_) return;
      if (np != params_.size() || nb != buffers_.size()) return;
      newParameters_ = std::move(ps);
      newBuffers_ = std::move(bs);
      newUserState_ = std::move(state);
      newModelVersion_ = version;
      newViaNvlink_ = viaNvlink;
      haveNewParameters_ = true;
    });
    parts_.rpc->handle("Acc::buffersUpdate/" + resName_, [this](const std::string&, const Bytes& p) {
      Reader r(p);
      uint32_t syncId = r.u32();
      uint32_t nb = r.u32();
      std::vector<Bytes> bs(nb);
      for (auto& x : bs) x = r.str();
      std::lock_guard<std::mutex> l(netMu_);
      if (syncId != netSyncId_ || nb != buffers_.size()) return;
      newBuffers_ = std::move(bs);
      haveNewBuffers_ = true;
    });
  }

  void requestModel() {
    if (syncLeader_ == myName_) return;
    isWaitingForModel_ = true;
    isWaitingForModelTimestamp_ = Clock::now();
    Writer w;
    w.u32(hSyncId_);
    w.str(myName_);
    // NVLink model sync (SURVEY 8(f)-3): possible once this peer's context is connected for the epoch, i.e. the leader's
    // publish region is mapped here
    w.u32(nvlinkSyncPossible() ? 1 : 0);
    parts_.rpc->send(syncLeader_, "Acc::requestModel/" + resName_, w.b);
  }

  bool nvlinkSyncPossible() {
    return gradsOnCuda_ && reducerReady_ && reducer_ && reducer_->syncId() == hSyncId_ && reducer_->world() > 1 && !nvlinkOff_;
  }
  // tensors that travel through the publish region: float32, on the accumulator's device (same predicate on both sides)
  bool viaPublishRegion(const torch::Tensor& t) const {
    return t.is_cuda() && t.get_device() == device_ && t.scalar_type() == torch::kFloat32 && t.numel() > 0;
  }
  uint64_t modelFlatBytes() {
    std::vector<uint64_t> n;
    for (auto* list : {&params_, &buffers_})
      for (auto& t : *list)
        if (viaPublishRegion(t)) n.push_back((uint64_t)t.numel());
    return n.empty() ? 0 : mb_ar_flat_numel(n.data(), (int)n.size()) * 4;
  }

  // kind bit 0: regular (periodic) update, bit 1: float CUDA tensors are published over NVLink instead of serialised
  Bytes packModel(bool regular, const Bytes& state, bool viaNvlink = false) {
    torch::NoGradGuard ng;
    Writer w;
    w.u32(hSyncId_);
    w.u32((regular ? 1u : 0u) | (viaNvlink ? 2u : 0u));
    w.i64(modelVersion_);
    if (viaNvlink) {
      // parameters + buffers -> this rank's publish region, ONE pack launch; the message below only goes out once
      // the stream has passed it (reference: every tensor .to(cpu), serialised, sent over the RPC transport)
      std::vector<const float*> ptrs;
      std::vector<uint64_t> numel;
      std::vector<torch::Tensor> keep;
      for (auto* list : {&params_, &buffers_})
        for (auto& t : *list)
          if (viaPublishRegion(t)) {
            keep.push_back(t.detach().contiguous());
            ptrs.push_back(keep.back().data_ptr<float>());
            numel.push_back((uint64_t)keep.back().numel());
          }
      c10::cuda::CUDAGuard dg(device_);
      if (!ptrs.empty())
        launch_counter() += check(mb_ar_xfer_pack(reducer()->ctx(), ptrs.data(), numel.data(), (int)ptrs.size(),
                                                  current_stream(device_)),
                                  "Accumulator model publish");
      cudaStreamSynchronize(c10::cuda::getCurrentCUDAStream(device_).stream());
      ++nvlinkPublishes_;
    }
    w.u32((uint32_t)params_.size());
    for (auto& p : params_) w.str(viaNvlink && viaPublishRegion(p) ? Bytes() : packTensor(p.detach().to(torch::kCPU)));
    w.u32((uint32_t)buffers_.size());
    for (auto& b : buffers_) w.str(viaNvlink && viaPublishRegion(b) ? Bytes() : packTensor(b.detach().to(torch::kCPU)));
    w.str(state);
    return w.b;
  }

  void setState(py::object userState) {
    MBH_PHASE("setState");
    userState = deepCopyToCpu(userState);
    Bytes pickled = pickleDumps(userState);
    std::lock_guard<std::mutex> l(mu_);
    userState_ = userState;
    wantsUserState_ = false;
    auto now = Clock::now();
    std::vector<std::string> requested;
    {
      std::lock_guard<std::mutex> nl(netMu_);
      requested.swap(requestedModelUpdate_);
    }
    // recipients that can pull over NVLink get the publish-region variant (packed once for all of them); the region is
    // not overwritten while a previous fetch is unacknowledged (10 s grace), such requests wait for a later tick
    std::vector<std::string> viaTcp, viaNvl, later;
    {
      std::lock_guard<std::mutex> nl(netMu_);
      if (!publishPending_.empty() && now - publishSince_ >= std::chrono::seconds(10)) publishPending_.clear();
      for (auto& n : requested) {
        if (n == myName_ || std::find(members_.begin(), members_.end(), n) == members_.end()) continue;
        if (requestedViaNvlink_.count(n) && nvlinkSyncPossible()) {
          if (publishPending_.empty()) viaNvl.push_back(n);
          else later.push_back(n);
        } else if (requestedViaNvlink_.count(n) && gradsOnCuda_ && !nvlinkOff_ && !reducerReady_ &&
                   now - epochStart_ < std::chrono::seconds(5)) {
          later.push_back(n);  // the requester is connected for this epoch, this peer not quite yet: next tick
        } else {
          viaTcp.push_back(n);
        }
      }
      for (auto& n : later) requestedModelUpdate_.push_back(n);
      for (auto& n : viaNvl) {
        publishPending_.insert(n);
        requestedViaNvlink_.erase(n);
      }
      if (!viaNvl.empty()) publishSince_ = now;
    }
    if (!viaTcp.empty()) {
      Bytes msg = packModel(false, pickled);
      for (auto& n : viaTcp) parts_.rpc->send(n, "Acc::modelUpdate/" + resName_, msg);
    }
    if (!viaNvl.empty()) {
      Bytes msg = packModel(false, pickled, /*viaNvlink=*/true);
      for (auto& n : viaNvl) parts_.rpc->send(n, "Acc::modelUpdate/" + resName_, msg);
    }
    if (!later.empty()) wantsUserState_ = true;
    if (syncLeader_ == myName_ && now - lastSentModel_ >= std::chrono::seconds(600)) {
      lastSentModel_ = now;
      Bytes reg = packModel(true, pickled);
      for (auto& n : members_)
        if (n != myName_) parts_.rpc->send(n, "Acc::modelUpdate/" + resName_, reg);
    }
  }

  py::object state() {
    std::lock_guard<std::mutex> l(mu_);
    hasNewUserState_ = false;
    return userState_ ? *userState_ : py::none();
  }

  void sendModelUpdates() {
    if (syncLeader_ != myName_) {
      wantsUserState_ = false;
      std::lock_guard<std::mutex> nl(netMu_);
      requestedModelUpdate_.clear();
      return;
    }
    auto now = Clock::now();
    bool requested;
    {
      std::lock_guard<std::mutex> nl(netMu_);
      requested = !requestedModelUpdate_.empty();
    }
    if (requested || now - lastSentModel_ >= std::chrono::seconds(600)) wantsUserState_ = true;
    if (now - lastSentBuffers_ >= std::chrono::seconds(12) && !buffers_.empty()) {
      lastSentBuffers_ = now;
      torch::NoGradGuard ng;
      Writer w;
      w.u32(hSyncId_);
      w.u32((uint32_t)buffers_.size());
      for (auto& b : buffers_) w.str(packTensor(b.detach().to(torch::kCPU)));
      for (auto& n : members_)
        if (n != myName_) parts_.rpc->send(n, "Acc::buffersUpdate/" + resName_, w.b);
    }
  }

  // Returns false when the update could not be applied and was requested again.
  bool commitModelUpdate() {
    MBH_PHASE("commitModelUpdate");
    torch::NoGradGuard ng;
    std::vector<Bytes> ps, bs;
    Bytes state;
    bool viaNvlink = false;
    {
      std::lock_guard<std::mutex> nl(netMu_);
      viaNvlink = newViaNvlink_;
    }
    if (viaNvlink && !nvlinkSyncPossible()) {
      // the NVLink context of this epoch went away between the request and the answer: drop the update and ask again
      // (the new request carries the current capability, i.e. the model then comes over the control plane)
      {
        std::lock_guard<std::mutex> nl(netMu_);
        haveNewParameters_ = false;
        newParameters_.clear();
        newBuffers_.clear();
        newUserState_.clear();
      }
      requestModel();
      return false;
    }
    {
      std::lock_guard<std::mutex> nl(netMu_);
      haveNewParameters_ = false;
      haveNewBuffers_ = false;
      modelVersion_ = newModelVersion_;
      ps.swap(newParameters_);
      bs.swap(newBuffers_);
      state.swap(newUserState_);
    }
    lastReceivedModel_ = Clock::now();
    if (ps.size() != params_.size()) throw std::runtime_error("Model parameters size mismatch in update!");
    if (bs.size() != buffers_.size()) throw std::runtime_error("Model buffers size mismatch in update!");
    if (viaNvlink) {
      // pull the leader's publish region straight into the parameter / buffer tensors: ONE launch of P2P loads
      auto it = std::find(members_.begin(), members_.end(), syncLeader_);
      if (it == members_.end()) throw std::runtime_error("moolib_b200: model update from a leader outside the group");
      std::vector<float*> ptrs;
      std::vector<uint64_t> numel;
      std::vector<std::pair<torch::Tensor, torch::Tensor>> fixups;  // (destination, contiguous temporary)
      for (auto* list : {&params_, &buffers_})
        for (auto& t : *list)
          if (viaPublishRegion(t)) {
            torch::Tensor d = t.detach();
            if (!d.is_contiguous()) {
              fixups.emplace_back(d, torch::empty_like(d, d.options().memory_format(c10::MemoryFormat::Contiguous)));
              d = fixups.back().second;
            }
            ptrs.push_back(d.data_ptr<float>());
            numel.push_back((uint64_t)d.numel());
          }
      c10::cuda::CUDAGuard dg(device_);
      if (!ptrs.empty())
        launch_counter() += check(mb_ar_xfer_unpack(reducer()->ctx(), (int)(it - members_.begin()), ptrs.data(), numel.data(),
                                                    (int)ptrs.size(), current_stream(device_)),
                                  "Accumulator model fetch");
      for (auto& f : fixups) f.first.copy_(f.second);
      cudaStreamSynchronize(c10::cuda::getCurrentCUDAStream(device_).stream());
      ++nvlinkFetches_;
      Writer ack;
      ack.u32(hSyncId_);
      ack.str(myName_);
      parts_.rpc->send(syncLeader_, "Acc::modelFetched/" + resName_, ack.b);  // the leader may reuse its region
    }
    for (size_t i = 0; i < params_.size(); ++i)
      if (!(viaNvlink && viaPublishRegion(params_[i]))) params_[i].copy_(unpackTensor(ps[i]).view_as(params_[i]), true);
    for (size_t i = 0; i < buffers_.size(); ++i)
      if (!(viaNvlink && viaPublishRegion(buffers_[i]))) buffers_[i].copy_(unpackTensor(bs[i]).view_as(buffers_[i]), true);
    userState_ = pickleLoads(state);
    hasNewUserState_ = true;
    hasReceivedModel_ = true;
    return true;
  }

  void commitBuffersUpdate() {
    torch::NoGradGuard ng;
    std::vector<Bytes> bs;
    {
      std::lock_guard<std::mutex> nl(netMu_);
      haveNewBuffers_ = false;
      bs.swap(newBuffers_);
    }
    if (bs.size() != buffers_.size()) throw std::runtime_error("Model buffers size mismatch in update!");
    for (size_t i = 0; i < buffers_.size(); ++i) buffers_[i].copy_(unpackTensor(bs[i]).view_as(buffers_[i]), true);
  }

  // ---- update (src/accumulator.cc:519-665) -------------------------------------------------------------------------
  void update() {
    torch::NoGradGuard ng;
    MBH_PHASE("update:enter");
    if (shouldUpdateGroup_) {
      py::gil_scoped_release nogil;
      parts_.service->update(*parts_.info, 0, 10 * 1000);
    }
    std::lock_guard<std::mutex> l(mu_);
    auto now = Clock::now();

    MBH_PHASE("update:locked");
    // leader election result
    if (findLeaderOp_ && findLeaderOp_->future->done()) {
      auto op = std::move(findLeaderOp_);
      findLeaderOp_.reset();
      Bytes value;
      const int flags = op->future->snapshot(&value, nullptr);
      if (flags & 1) {
        Reader r(value);
        int64_t version = r.i64();
        std::string leader = r.str();
        isFindingLeader_ = false;
        syncLeader_ = leader;
        {
          std::lock_guard<std::mutex> gl(parts_.info->mutex);
          members_ = parts_.info->members;
        }
        if (version != modelVersion_ || !hasReceivedModel_) {
          // CUDA models: wait (up to 2 s) for the NVLink context of this epoch, then the model comes over NVLink
          if (gradsOnCuda_ && !nvlinkOff_ && !reducerReady_ && syncLeader_ != myName_) {
            isWaitingForModel_ = true;
            isWaitingForModelTimestamp_ = now;
            deferredRequestSince_ = now;
            requestDeferred_ = true;
          } else {
            requestModel();
          }
        } else {
          lastReceivedModel_ = now;
        }
      } else if (hSyncId_ == parts_.info->syncId.load()) {
        resync();
      }
    }
    MBH_PHASE("update:reducer-poll");
    if (gradsOnCuda_ && hSyncId_ != 0 && !reducerReady_) {
      auto r = reducer();
      if (r->failed()) throw std::runtime_error(r->error());
      reducerReady_ = r->poll() && r->syncId() == hSyncId_;
      if (reducerReady_ && deviceGate() && gradsInArena()) {
        // new group epoch: the ring restarted at position 0; move .grad off whatever buffer it pointed at
        torch::NoGradGuard ng2;
        appliedBase_ = nullptr;
        repointForAccumulation();
      }
    }
    if (requestDeferred_ && (reducerReady_ || now - deferredRequestSince_ >= std::chrono::seconds(2))) {
      requestDeferred_ = false;
      if (hSyncId_ != 0 && !syncLeader_.empty()) requestModel();
    }
    MBH_PHASE("update:checkGradientResult");
    checkGradientResult();
    MBH_PHASE("update:after-check");

    uint32_t groupSync = parts_.info->syncId.load();
    if (hSyncId_ != groupSync) {
      hSyncId_ = groupSync;
      syncLeader_.clear();
      findLeaderOp_.reset();
      for (auto& v : slots_) v.reset();
      nextIndex_ = nextResultIndex_ = 0;
      {
        std::lock_guard<std::mutex> nl(netMu_);
        netSyncId_ = hSyncId_;
        requestedModelUpdate_.clear();
        requestedViaNvlink_.clear();
        publishPending_.clear();
        haveNewParameters_ = false;
      }
      hasNewUserState_ = false;
      wantsUserState_ = false;
      isFindingLeader_ = true;
      isWaitingForModel_ = false;
      requestDeferred_ = false;
      epochStart_ = now;
      hasGradients_ = false;
      reducerReady_ = false;
      members_.clear();
      if (hSyncId_ != 0) {
        Writer w;
        w.i64(modelVersion_);
        w.str(myName_);
        try {
          // max over (modelVersion, name) (src/accumulator.cc:589-596)
          findLeaderOp_ = parts_.service->allReduce(
              parts_.info, "Accumulator::findLeader/" + resName_, w.b, [](const Bytes& a, const Bytes& b) {
                Reader ra(a), rb(b);
                int64_t va = ra.i64(), vb = rb.i64();
                std::string na = ra.str(), nb = rb.str();
                return std::tie(va, na) < std::tie(vb, nb) ? b : a;
              });
        } catch (const std::exception&) {
          // the group changed again under us; the next update() sees the new syncId
          hSyncId_ = 0;
        }
        if (gradsOnCuda_) reducer()->poll();  // start the NVLink handle exchange alongside the election
      }
    }

    bool haveParams, haveBuffers;
    {
      std::lock_guard<std::mutex> nl(netMu_);
      haveParams = haveNewParameters_;
      haveBuffers = haveNewBuffers_;
      netModelVersion_ = modelVersion_;
      netWaitingForModel_ = isWaitingForModel_;
    }
    MBH_PHASE("update:model-sync");
    if (haveParams) {
      bool ignore;
      {
        std::lock_guard<std::mutex> nl(netMu_);
        ignore = !isWaitingForModel_ && modelVersion_ != newModelVersion_;
        if (ignore) haveNewParameters_ = false;
      }
      if (!ignore && commitModelUpdate()) isWaitingForModel_ = false;
    } else if (isWaitingForModel_ && now - isWaitingForModelTimestamp_ >= std::chrono::seconds(60)) {
      requestModel();
    } else if (!isWaitingForModel_ && connectedImpl() && syncLeader_ != myName_ &&
               now - lastReceivedModel_ >= std::chrono::minutes(30)) {
      lastReceivedModel_ = now;
      resync();
    }
    if (haveBuffers && !haveParams) commitBuffersUpdate();
    MBH_PHASE("update:sendModelUpdates");
    if (!members_.empty()) sendModelUpdates();
    MBH_PHASE("idle");
  }

  // ---- misc API --------------------------------------------------------------------------------------------------
  py::dict debugState() {
    std::lock_guard<std::mutex> l(mu_);
    py::dict d;
    d["sync_id"] = hSyncId_;
    d["group_sync_id"] = parts_.info->syncId.load();
    d["leader"] = syncLeader_;
    d["members"] = members_.size();
    d["finding_leader"] = isFindingLeader_;
    d["waiting_for_model"] = isWaitingForModel_;
    d["has_received_model"] = hasReceivedModel_;
    d["has_gradients"] = hasGradients_;
    d["reducer_ready"] = reducerReady_;
    d["reducer_failed"] = reducer_ ? reducer_->failed() : false;
    d["reducer_sync"] = reducer_ ? reducer_->syncId() : 0u;
    d["model_version"] = modelVersion_;
    d["last_error"] = lastError_;
    d["nvlink_model_publishes"] = nvlinkPublishes_;
    d["nvlink_model_fetches"] = nvlinkFetches_;
    d["next_index"] = nextIndex_;
    auto& v = slots_[nextResultIndex_];
    if (v) {
      d["slot_counting"] = v->isCounting;
      d["slot_count_op"] = (bool)v->countOp;
      d["slot_reduce_started"] = v->reduceStarted;
      d["slot_reduce_done"] = v->reduceDone;
      d["slot_kernel_in_flight"] = v->kernelInFlight;
      d["slot_num_gradients"] = v->data.num_gradients;
      d["slot_num_skipped"] = v->data.num_skipped;
      d["slot_batch"] = v->data.batch_size;
    }
    return d;
  }
  py::dict getGradientStats() {
    py::dict r;
    r["num_gradients"] = stats_.num_gradients;
    r["num_skipped"] = stats_.num_skipped;
    r["batch_size"] = stats_.batch_size;
    return r;
  }
  int64_t modelVersion() { return modelVersion_; }
  void setModelVersion(int64_t v) { modelVersion_ = v; }
  void setVirtualBatchSize(int n) {
    std::lock_guard<std::mutex> l(mu_);
    virtualBatchSize_ = (uint64_t)n;
  }
  void setParallelGradients(int n) {
    if (n < 1 || n > MB_AR_MAX_SLOTS)
      throw std::runtime_error("set_parallel_gradients: n must be in [1, " + std::to_string(MB_AR_MAX_SLOTS) + "]");
    std::lock_guard<std::mutex> l(mu_);
    releaseGradViews();
    slots_.clear();
    slots_.resize(n);
    nextIndex_ = nextResultIndex_ = 0;
    reducer_.reset();
    reducerReady_ = false;
  }

  // ---- device-side round timings (bench.py: roofline_nvlink) -------------------------------------------------------
  void recordTiming(ReduceSlot& v, bool reduced) {
    float gateUs = 0.f, reduceUs = 0.f;
    if (mb_ar_round_times(reducer()->ctx(), (int)v.index, &gateUs, &reduceUs) != MB_OK) return;  // no kernel ran
    if (timings_.size() >= 65536) return;
    timings_.push_back({gateUs, reduceUs, reduced});
  }
  py::dict reduceTimings(bool clear) {
    std::lock_guard<std::mutex> l(mu_);
    py::list gate, red, ok;
    for (auto& t : timings_) {
      gate.append(t.gateUs);
      red.append(t.reduceUs);
      ok.append(t.reduced);
    }
    py::dict d;
    d["gate_us"] = gate;      // K-A0: includes the wait for the slowest peer
    d["reduce_us"] = red;     // K-A2: the data movement
    d["reduced"] = ok;        // false: the gate stayed shut (short batch), K-A2 returned at once
    d["bytes"] = arena_ ? (int64_t)arena_->total : (int64_t)0;
    d["world"] = reducer_ ? reducer_->world() : 0;
    d["stage_launches"] = stageLaunches_;
    d["zero_copy_rounds"] = zeroCopyRounds_;
    d["short_rounds"] = shortRounds_;
    d["device_gate"] = deviceGate();
    if (clear) {
      timings_.clear();
      stageLaunches_ = zeroCopyRounds_ = shortRounds_ = 0;
    }
    return d;
  }
  std::string getLeader() {
    std::lock_guard<std::mutex> l(mu_);
    return syncLeader_;
  }
  bool isLeader() {
    std::lock_guard<std::mutex> l(mu_);
    return syncLeader_ == myName_;
  }

 private:
  std::mutex mu_;
  py::object ownGroup_;
  GroupParts parts_;
  bool shouldUpdateGroup_ = false;
  std::string resName_, myName_;
  std::vector<torch::Tensor> params_, buffers_;
  bool gradsOnCuda_ = false;
  int device_ = 0;
  std::shared_ptr<DeviceReducer> reducer_;
  bool reducerReady_ = false;
  cudaStream_t arStream_ = nullptr;
  bool nvlinkOff_ = [] {
    const char* e = std::getenv("MOOLIB_B200_NVLINK_MODEL_SYNC");
    return e && *e == '0';
  }();
  bool requestDeferred_ = false;
  Clock::time_point deferredRequestSince_{}, epochStart_ = Clock::now();
  uint64_t nvlinkPublishes_ = 0, nvlinkFetches_ = 0;
  std::unique_ptr<GradArena> arena_;
  void* appliedBase_ = nullptr;   // the buffer of the applied result that .grad currently shows (null: none)
  struct RoundTiming {
    float gateUs, reduceUs;
    bool reduced;
  };
  std::vector<RoundTiming> timings_;
  uint64_t stageLaunches_ = 0, zeroCopyRounds_ = 0, shortRounds_ = 0;
  bool strictCounting_ = [] {
    const char* e = std::getenv("MOOLIB_B200_STRICT_COUNTING");
    return !(e && *e == '0');
  }();
  std::vector<std::shared_ptr<ReduceSlot>> slots_;
  size_t nextIndex_ = 0, nextResultIndex_ = 0;
  uint64_t virtualBatchSize_ = 1;
  uint32_t hSyncId_ = 0;
  int64_t modelVersion_ = 0;
  std::string syncLeader_;
  std::vector<std::string> members_;
  bool isFindingLeader_ = false, isWaitingForModel_ = false, hasGradients_ = false, hasReceivedModel_ = false;
  bool wantsUserState_ = false;
  std::atomic<bool> hasNewUserState_{false};
  std::optional<py::object> userState_;
  mb_ar_hdr stats_{0, 0, 0, 0};
  std::shared_ptr<SmallReduce> findLeaderOp_;
  Clock::time_point isWaitingForModelTimestamp_{}, lastReceivedModel_ = Clock::now(), lastSentModel_ = Clock::now(),
                    lastSentBuffers_ = Clock::now();
  std::string lastError_;
  // state touched by the IO thread
  std::mutex netMu_;
  uint32_t netSyncId_ = 0;
  int64_t netModelVersion_ = 0;
  bool netWaitingForModel_ = false;
  std::vector<std::string> requestedModelUpdate_;
  std::set<std::string> requestedViaNvlink_;  // requesters that can pull from this peer's publish region
  std::set<std::string> publishPending_;      // NVLink recipients that have not acknowledged their fetch yet
  Clock::time_point publishSince_{};
  bool newViaNvlink_ = false;
  bool haveNewParameters_ = false, haveNewBuffers_ = false;
  int64_t newModelVersion_ = 0;
  std::vector<Bytes> newParameters_, newBuffers_;
  Bytes newUserState_;
};

void bind_accumulator(py::module_& m) {
  py::class_<Accumulator>(m, "Accumulator",
                          "Accumulate and synchronise gradients / model state across the peers of a group "
                          "(moolib.Accumulator API); CUDA gradients are reduced by the NVLink allreduce kernel.")
      .def(py::init<std::string, py::object, py::object, py::object>(), py::arg("name"), py::arg("parameters"),
           py::arg("buffers"), py::arg("group") = py::none())
      .def("connect", &Accumulator::connect, py::arg("address"))
      .def("update", &Accumulator::update)
      .def("connected", &Accumulator::connected)
      .def("wants_state", &Accumulator::wantsState)
      .def("has_new_state", &Accumulator::hasNewState)
      .def("set_state", &Accumulator::setState)
      .def("state", &Accumulator::state)
      .def("wants_gradients", &Accumulator::wantsGradients)
      .def("has_gradients", &Accumulator::hasGradients)
      .def("reduce_gradients", &Accumulator::reduceGradients, py::arg("batch_size"))
      .def("skip_gradients", &Accumulator::skipGradients)
      .def("zero_gradients", &Accumulator::zeroGradients)
      .def("model_version", &Accumulator::modelVersion)
      .def("set_model_version", &Accumulator::setModelVersion)
      .def("set_virtual_batch_size", &Accumulator::setVirtualBatchSize)
      .def("set_parallel_gradients", &Accumulator::setParallelGradients)
      .def("get_leader", &Accumulator::getLeader)
      .def("is_leader", &Accumulator::isLeader)
      .def("get_gradient_stats", &Accumulator::getGradientStats)
      .def("debug_state", &Accumulator::debugState)
      .def("reduce_timings", &Accumulator::reduceTimings, py::arg("clear") = false,
           "CUDA-event timings of every device-gated round: K-A0 (gate, waits for the slowest peer) and K-A2 (reduce)");
}

}  // namespace mbh
