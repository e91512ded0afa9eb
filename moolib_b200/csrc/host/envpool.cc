// EnvPool / EnvStepper (HP-B source side): Python environments stepped in forked worker processes that write their
// observations straight into a shared-memory slab laid out as the learner batch [B, *shape].
//
// Mirrors moolib.EnvPool (reference: src/env.h, src/env.cc; bound at src/moolib.cc:1613-1645): same constructor, same
// `step(batch_index, action) -> future`, `future.result() -> dict[str, Tensor]` of CPU tensors aliasing the slabs until
// the next step() on that buffer, same dtype/shape/index errors, same env protocol (reset on first step and on done;
// obs dict or array -> "state"; "done" bool and "reward" f32 appended; action mailbox counter encoding `prev + 1 + a`,
// src/env.cc:340-345 / src/env.h:279-292).
//
// What changes for a B200 learner:
//   * the slabs are sized for the pool's batch (not maxEnvs = 4096 rows as src/env.h:236) and, once a CUDA context
//     exists, registered as mapped pinned memory (cudaHostRegister): `result()` tensors are pinned, so the learner's
//     `.to(device, non_blocking=True)` is a real async DMA and the copy kernels can read the slabs in place
//     (mb_copy2d_batch with host-mapped sources -- one launch for all keys);
//   * a CUDA action tensor is scattered into the per-env mailboxes by the device (mb_scatter_actions) instead of
//     a pinned copy + stream synchronize + CPU loop (src/env.cc:310-319, 340-345).
// Process management is deliberately simpler than the reference's double-fork server (src/env.cc:176-223): the
// workers are forked directly in the constructor.
#include "common.h"

#include <optional>
#include "control.h"

#include <fcntl.h>
#include <pybind11/numpy.h>
#include <semaphore.h>
#include <signal.h>
#include <sys/mman.h>
#include <sys/prctl.h>
#include <sys/wait.h>
#include <unistd.h>

#include <cuda_runtime_api.h>

namespace mbh {

namespace {

constexpr size_t kMaxClients = 256;
constexpr size_t kMaxEnvs = 4096;
constexpr size_t kMaxBuffers = 4;
constexpr size_t kMaxKeys = 32;
constexpr size_t kQueueCap = 8;

struct KeyEntry {
  char key[64];
  int64_t shape[8];
  int32_t ndim;
  char dtype;  // numpy kind
  uint64_t elements, itemsize;
  uint64_t dataOffset;  // from the arena base
};

struct ClientCtl {
  std::atomic<uint64_t> nStepsIn, nStepsOut, resultOffset;
};

struct BufferCtl {
  std::atomic<uint32_t> batchAllocated, batchAllocating;
  uint32_t nkeys;
  KeyEntry keys[kMaxKeys];
  ClientCtl clients[kMaxClients];
  std::atomic<uint32_t> action[kMaxEnvs];  // src/env.h:96-98 EnvInput
};

struct ClientIO {
  sem_t inSem, outSem;
  std::atomic<uint32_t> qTop, qBot;
  int32_t queue[kQueueCap];
};

struct Shared {
  uint64_t size;
  std::atomic<uint64_t> allocated;
  std::atomic<uint32_t> clients, terminate, workerError;
  std::atomic<uint32_t> errorClaimed;  // the first failing worker writes errorText, then sets workerError
  char errorText[512];
  uint32_t batchSize, numBuffers, numClients;
  ClientIO io[kMaxClients];
  BufferCtl buffers[kMaxBuffers];

  uint64_t allocAligned(uint64_t n, uint64_t align) {
    uint64_t off = allocated.load(std::memory_order_relaxed), start;
    do {
      start = (off + align - 1) / align * align;
    } while (!allocated.compare_exchange_weak(off, start + n, std::memory_order_relaxed));
    if (start + n > size) throw std::runtime_error("Out of space in shared memory buffer");
    return start;
  }
};

torch::ScalarType dtypeOf(char kind, uint64_t itemsize) {
  switch (kind) {
    case 'f': return itemsize == 8 ? torch::kFloat64 : itemsize == 2 ? torch::kFloat16 : torch::kFloat32;
    case 'i': return itemsize == 8 ? torch::kInt64 : itemsize == 4 ? torch::kInt32 : itemsize == 2 ? torch::kInt16 : torch::kInt8;
    case 'u':
      if (itemsize == 1) return torch::kUInt8;
      throw std::runtime_error("EnvPool: unsigned observation dtypes wider than 8 bits are not supported by torch");
    case 'b': return torch::kBool;
  }
  throw std::runtime_error(std::string("EnvPool: unsupported observation dtype kind '") + kind + "'");
}

// ---- worker process -----------------------------------------------------------------------------------------------

struct WorkerEnv {
  py::object env, reset, step;
  uint64_t steps = 0;
  uint32_t prevAction = 0;
};

void fillKey(Shared* sh, BufferCtl& b, size_t row, const std::string& key, const void* src, size_t len) {
  for (uint32_t i = 0; i < b.nkeys; ++i) {
    KeyEntry& k = b.keys[i];
    if (key == k.key) {
      if (len != k.itemsize * k.elements) throw std::runtime_error("fill batch size mismatch");
      // src/env.h:258: one memcpy of the env's item into its row of the [B, *shape] slab
      std::memcpy(reinterpret_cast<char*>(sh) + k.dataOffset + k.itemsize * k.elements * row, src, len);
      return;
    }
  }
  throw std::runtime_error(key + ": batch key not found");
}

void allocateBatch(Shared* sh, BufferCtl& b, const std::vector<std::pair<std::string, py::array>>& obs) {
  auto add = [&](const std::string& key, int ndim, const ssize_t* shape, uint64_t itemsize, char kind) {
    if (b.nkeys >= kMaxKeys) throw std::runtime_error("EnvPool: too many observation keys");
    KeyEntry& k = b.keys[b.nkeys];
    std::memset(&k, 0, sizeof(k));
    std::snprintf(k.key, sizeof(k.key), "%s", key.c_str());
    k.ndim = ndim;
    k.elements = 1;
    for (int i = 0; i < ndim; ++i) {
      k.shape[i] = shape[i];
      k.elements *= (uint64_t)shape[i];
    }
    k.itemsize = itemsize;
    k.dtype = kind;
    const uint64_t bytes = (k.itemsize * k.elements * sh->batchSize + 4095) / 4096 * 4096;
    k.dataOffset = sh->allocAligned(bytes, 4096);  // page aligned: each slab can be cudaHostRegister'ed on its own
    ++b.nkeys;
  };
  for (auto& [key, arr] : obs) add(key, (int)arr.ndim(), arr.shape(), (uint64_t)arr.itemsize(), arr.dtype().kind());
  add("done", 0, nullptr, 1, 'b');
  add("reward", 0, nullptr, 4, 'f');
}

// reference: Env::step, src/env.h:265-339
void stepEnv(Shared* sh, size_t bufferIndex, size_t row, WorkerEnv& e, py::object& createEnv) {
  BufferCtl& b = sh->buffers[bufferIndex];
  ++e.steps;
  uint32_t action = e.prevAction;
  auto start = Clock::now();
  uint32_t spins = 0;
  while ((action = b.action[row].load(std::memory_order_acquire)) == e.prevAction) {
    if (sh->terminate.load(std::memory_order_relaxed)) return;
    if ((++spins & 0xfff) == 0) {
      if (getppid() == 1) _exit(0);
      if (Clock::now() - start >= std::chrono::seconds(120)) throw std::runtime_error("Timed out waiting for env action");
      if (spins > 0x100000) usleep(50);
    }
  }
  uint32_t decoded = action - (e.prevAction + 1);
  e.prevAction = action;
  bool done = false;
  float reward = 0.0f;
  py::object rawObs;
  if (e.steps == 1) {
    if (!e.env) {
      e.env = createEnv();
      e.reset = e.env.attr("reset");
      e.step = e.env.attr("step");
    }
    rawObs = e.reset();
  } else {
    py::tuple tup = e.step(decoded);
    rawObs = tup[0];
    reward = py::cast<float>(tup[1]);
    done = py::cast<bool>(tup[2]);
    if (done) rawObs = e.reset();
  }
  std::vector<std::pair<std::string, py::array>> obs;
  auto toArray = [](py::handle h) {
    return py::array::ensure(py::reinterpret_borrow<py::object>(h), py::array::c_style | py::array::forcecast);
  };
  if (py::isinstance<py::dict>(rawObs)) {
    for (auto kv : py::reinterpret_borrow<py::dict>(rawObs)) obs.emplace_back(py::cast<std::string>(kv.first), toArray(kv.second));
  } else {
    obs.emplace_back("state", toArray(rawObs));
  }
  for (auto& kv : obs)
    if (!kv.second) throw std::runtime_error("EnvPool: observation '" + kv.first + "' is not array-like");
  if (!b.batchAllocated.load(std::memory_order_acquire)) {
    if (b.batchAllocating.exchange(1)) {
      while (!b.batchAllocated.load(std::memory_order_acquire)) usleep(10);
    } else {
      allocateBatch(sh, b, obs);
      b.batchAllocated.store(1, std::memory_order_release);
    }
  }
  fillKey(sh, b, row, "done", &done, 1);
  fillKey(sh, b, row, "reward", &reward, 4);
  for (auto& [key, arr] : obs) fillKey(sh, b, row, key, arr.data(), (size_t)arr.nbytes());
}

// reference: EnvRunner::run, src/env.h:407-453
[[noreturn]] void workerMain(Shared* sh, int myIndex, py::object createEnv) {
  prctl(PR_SET_PDEATHSIG, SIGKILL);
  signal(SIGINT, SIG_IGN);
  std::vector<std::vector<WorkerEnv>> envs(kMaxBuffers);
  ClientIO& io = sh->io[myIndex];
  try {
    sh->clients.fetch_add(1);
    while (!sh->terminate.load()) {
      if (io.qTop.load(std::memory_order_acquire) == io.qBot.load(std::memory_order_relaxed)) {
        timespec ts;
        clock_gettime(CLOCK_REALTIME, &ts);
        ts.tv_sec += 1;
        sem_timedwait(&io.inSem, &ts);
        if (getppid() == 1) break;
        continue;
      }
      uint32_t bot = io.qBot.load(std::memory_order_relaxed);
      size_t bufferIndex = (size_t)io.queue[bot % kQueueCap];
      io.qBot.store(bot + 1, std::memory_order_release);
      BufferCtl& b = sh->buffers[bufferIndex];
      ClientCtl& c = b.clients[myIndex];
      uint64_t done = c.nStepsOut.load(), want = c.nStepsIn.load();
      if (want != done) {
        size_t offset = (size_t)c.resultOffset.load(), n = (size_t)(want - done);
        auto& list = envs[bufferIndex];
        if (list.size() < n) list.resize(n);
        for (size_t i = 0; i < n; ++i) stepEnv(sh, bufferIndex, offset + i, list[i], createEnv);
        c.nStepsOut.store(want, std::memory_order_release);
        sem_post(&io.outSem);
      }
    }
  } catch (const std::exception& ex) {
    if (!sh->errorClaimed.exchange(1)) {
      // the learner throws errorText as soon as it sees workerError: the text must be complete before the flag is set
      std::snprintf(sh->errorText, sizeof(sh->errorText), "Error in env: %s", ex.what());
      sh->workerError.store(1, std::memory_order_release);
    }
    for (size_t i = 0; i < kMaxClients; ++i) sem_post(&sh->io[i].outSem);
  }
  _exit(0);
}

}  // namespace

// ---- learner side ---------------------------------------------------------------------------------------------------

class EnvStepper;

struct EnvStepperFuture {
  EnvStepper* stepper;
  std::shared_ptr<void> keep;
  int bufferIndex;
  size_t size, stride;
  // device = None: CPU tensors aliasing the (pinned, device-mapped) slabs, as the reference (src/env.cc:389-401).
  // device = "cuda:i": every key on the device, read from the slabs by ONE launch of the copy kernel -- what the actor
  // loop otherwise does with one `.to(device)` per key (examples/vtrace/experiment.py:492-494).
  py::object result(std::optional<std::string> device);
};

class EnvStepper : public std::enable_shared_from_this<EnvStepper> {
 public:
  EnvStepper(py::object createEnv, int numProcesses, int batchSize, int numBatches)
      : batchSize_(batchSize), numBatches_(numBatches) {
    if (numProcesses < 1 || (size_t)numProcesses > kMaxClients) throw std::runtime_error("EnvPool: bad num_processes");
    if (batchSize < 1 || (size_t)batchSize > kMaxEnvs) throw std::runtime_error("EnvPool: bad batch_size");
    if (numBatches < 1 || (size_t)numBatches > kMaxBuffers)
      throw std::runtime_error("EnvPool: num_batches must be in [1, " + std::to_string(kMaxBuffers) + "]");
    numClients_ = std::min(numProcesses, batchSize);
    const char* e = std::getenv("MOOLIB_B200_ENVPOOL_BYTES");
    arenaBytes_ = e ? std::strtoull(e, nullptr, 0) : (2ull << 30);  // sparse: only touched pages are backed
    arenaBytes_ = std::max<uint64_t>(arenaBytes_, sizeof(Shared) + (1 << 20));
    void* mem = mmap(nullptr, arenaBytes_, PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
    if (mem == MAP_FAILED) throw std::runtime_error("EnvPool: mmap of the shared arena failed");
    shared_ = new (mem) Shared();
    shared_->size = arenaBytes_;
    shared_->allocated = (sizeof(Shared) + 4095) / 4096 * 4096;
    shared_->batchSize = (uint32_t)batchSize;
    shared_->numBuffers = (uint32_t)numBatches;
    shared_->numClients = (uint32_t)numClients_;
    for (int i = 0; i < numClients_; ++i) {
      sem_init(&shared_->io[i].inSem, 1, 0);
      sem_init(&shared_->io[i].outSem, 1, 0);
    }
    for (int i = 0; i < numClients_; ++i) {
      pid_t pid = fork();
      if (pid < 0) throw std::runtime_error(std::string("EnvPool: fork failed: ") + std::strerror(errno));
      if (pid == 0) {
        PyOS_AfterFork_Child();
        workerMain(shared_, i, createEnv);
      }
      pids_.push_back(pid);
    }
    for (auto& b : bufferBusy_) b = false;
  }

  ~EnvStepper() {
    shared_->terminate = 1;
    for (int i = 0; i < numClients_; ++i) sem_post(&shared_->io[i].inSem);
    for (pid_t p : pids_) {
      int st;
      bool gone = false;
      for (int k = 0; k < 200 && !gone; ++k) {
        gone = waitpid(p, &st, WNOHANG) != 0;
        if (!gone) usleep(5000);
      }
      if (!gone) {
        kill(p, SIGKILL);
        waitpid(p, &st, 0);
      }
    }
    for (auto& r : registered_) cudaHostUnregister(r);
    munmap(shared_, arenaBytes_);
  }

  // reference: EnvPoolWrapper::step (src/moolib.cc:1396-1409) + EnvStepper::step (src/env.cc:273-349)
  EnvStepperFuture step(int bufferIndex, py::object actionObject) {
    if (is_tensor(actionObject)) {
      torch::Tensor t = to_tensor(actionObject);
      if (t.dim() == 1 && t.size(0) != batchSize_)
        throw std::runtime_error("env step was passed an action tensor with batch size " + std::to_string(t.size(0)) +
                                 ", expected " + std::to_string(batchSize_));
    }
    if (bufferIndex < 0 || bufferIndex >= numBatches_)
      throw std::runtime_error("env step was passed an out-of-range batch index " + std::to_string(bufferIndex) +
                               " (valid range is [0," + std::to_string(numBatches_) + "))");
    if (!is_tensor(actionObject))
      throw std::runtime_error(
          "EnvStepper::step function was passed an action argument that could not be converted to a Tensor");
    torch::Tensor action = to_tensor(actionObject);
    if (action.scalar_type() != torch::kInt64)
      throw std::runtime_error("EnvStepper::step expected action tensor with data type long");
    if (action.dim() != 1) throw std::runtime_error("EnvStepper::step expected a 1-dimensional tensor");
    if (bufferBusy_[bufferIndex].exchange(true))
      throw std::runtime_error("EnvStepper: attempt to step buffer index " + std::to_string(bufferIndex) +
                               " twice concurrently");
    checkWorkers();
    BufferCtl& b = shared_->buffers[bufferIndex];
    const size_t size = (size_t)action.size(0);
    const size_t stride = (size + numClients_ - 1) / numClients_;
    size_t client = 0;
    for (size_t i = 0; i < size; i += stride, ++client) {
      size_t n = std::min(size - i, stride);
      ClientCtl& c = b.clients[client];
      c.resultOffset.store(i);
      c.nStepsIn.fetch_add(n);
      ClientIO& io = shared_->io[client];
      uint32_t top = io.qTop.load(std::memory_order_relaxed);
      if (top - io.qBot.load(std::memory_order_acquire) >= kQueueCap) throw std::runtime_error("EnvStepper: shared queue is full");
      io.queue[top % kQueueCap] = bufferIndex;
      io.qTop.store(top + 1, std::memory_order_release);
      sem_post(&io.inSem);
    }
    if (action.is_cuda()) {
      // B3 on the device: mailbox[i] += 1 + action[i], written straight into the (host-mapped) shared arena
      ensureRegistered(reinterpret_cast<char*>(shared_), sizeof(Shared));  // header (mailboxes) as one registration
      torch::Tensor a = action.contiguous();
      c10::cuda::CUDAGuard g(a.get_device());
      uint32_t* dev = nullptr;
      if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&dev), &b.action[0], 0) != cudaSuccess)
        throw std::runtime_error("EnvPool: the action mailboxes are not device-mapped");
      launch_counter() += check(mb_scatter_actions(dev, 1, a.data_ptr<int64_t>(), size, current_stream(a.get_device())),
                                "EnvPool.step");
      keepAction_[bufferIndex] = a;  // alive until the kernel has run
    } else {
      // Host-written mailboxes release the workers immediately.  If the slabs are pinned/mapped, device reads of the
      // previous result (async H2D copies, Batcher kernels) may still be queued: wait for them before the workers may
      // overwrite the slab.  (With CUDA actions this ordering is free: the scatter kernel above is enqueued behind
      // those reads on the same stream.)
      if (!registered_.empty()) {
        py::gil_scoped_release nogil;
        cudaStreamSynchronize(c10::cuda::getCurrentCUDAStream().stream());
      }
      torch::Tensor a = action.contiguous();
      const int64_t* acc = a.data_ptr<int64_t>();
      for (size_t i = 0; i < size; ++i) {
        auto& m = b.action[i];
        m.store(m.load(std::memory_order_relaxed) + 1 + (uint32_t)acc[i], std::memory_order_release);
      }
    }
    return EnvStepperFuture{this, shared_from_this(), bufferIndex, size, stride};
  }

  // reference: EnvStepperFuture::result, src/env.cc:351-412
  py::object result(int bufferIndex, size_t size, size_t stride) {
    BufferCtl& b = shared_->buffers[bufferIndex];
    {
      py::gil_scoped_release nogil;
      auto start = Clock::now();
      size_t client = 0;
      for (size_t i = 0; i < size; i += stride, ++client) {
        ClientCtl& c = b.clients[client];
        uint64_t want = c.nStepsIn.load();
        while (c.nStepsOut.load(std::memory_order_acquire) != want) {
          if (shared_->workerError.load()) throw std::runtime_error(shared_->errorText);
          if (Clock::now() - start >= std::chrono::seconds(1800)) throw std::runtime_error("Timed out waiting for env");
          timespec ts;
          clock_gettime(CLOCK_REALTIME, &ts);
          ts.tv_nsec += 2000000;
          if (ts.tv_nsec >= 1000000000) ts.tv_sec += 1, ts.tv_nsec -= 1000000000;
          sem_timedwait(&shared_->io[client].outSem, &ts);
          checkWorkers();
        }
      }
    }
    auto& map = outputMap_[bufferIndex];
    if (map.empty()) {
      for (uint32_t i = 0; i < b.nkeys; ++i) {
        KeyEntry& k = b.keys[i];
        std::vector<int64_t> sizes(k.shape, k.shape + k.ndim);
        sizes.insert(sizes.begin(), (int64_t)size);
        char* data = reinterpret_cast<char*>(shared_) + k.dataOffset;
        ensureRegistered(data, (k.itemsize * k.elements * shared_->batchSize + 4095) / 4096 * 4096);
        map.emplace_back(k.key, torch::from_blob(data, sizes, torch::TensorOptions().dtype(dtypeOf(k.dtype, k.itemsize))));
      }
    }
    bufferBusy_[bufferIndex] = false;
    py::dict r;
    for (auto& [key, t] : map) r[py::str(key)] = to_python(t);
    return std::move(r);
  }

 private:
  void checkWorkers() {
    if (shared_->workerError.load()) throw std::runtime_error(shared_->errorText);
  }
  // Pin + map a page-aligned piece of the arena once a CUDA context exists (no-op on a CPU-only process).
  void ensureRegistered(char* p, size_t bytes) {
    if (!torch::cuda::is_available()) return;
    char* base = reinterpret_cast<char*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)4095);
    size_t len = ((p - base) + bytes + 4095) / 4096 * 4096;
    for (auto& r : registered_)
      if (r == base) return;
    if (cudaHostRegister(base, len, cudaHostRegisterMapped | cudaHostRegisterPortable) == cudaSuccess) registered_.push_back(base);
    else cudaGetLastError();
  }

  int batchSize_, numBatches_, numClients_ = 0;
  uint64_t arenaBytes_ = 0;
  Shared* shared_ = nullptr;
  std::vector<pid_t> pids_;
  std::array<std::atomic<bool>, kMaxBuffers> bufferBusy_;
  std::array<std::vector<std::pair<std::string, torch::Tensor>>, kMaxBuffers> outputMap_;
  std::array<torch::Tensor, kMaxBuffers> keepAction_;
  std::vector<void*> registered_;
};

py::object EnvStepperFuture::result(std::optional<std::string> device) {
  py::object host = stepper->result(bufferIndex, size, stride);
  if (!device || *device == "cpu") return host;
  return nestToDevice(host, *device);
}

void bind_envpool(py::module_& m) {
  py::class_<EnvStepperFuture>(m, "EnvStepperFuture").def("result", &EnvStepperFuture::result, py::arg("device") = py::none());
  py::class_<EnvStepper, std::shared_ptr<EnvStepper>>(m, "EnvPool",
                                                      "Batched Python environments in worker processes "
                                                      "(moolib.EnvPool API) writing into pinned, device-mapped slabs.")
      .def(py::init<py::object, int, int, int>(), py::arg("create_env"), py::arg("num_processes"), py::arg("batch_size"),
           py::arg("num_batches"))
      .def("step", &EnvStepper::step, py::arg("batch_index"), py::arg("action"));
  m.attr("EnvStepper") = m.attr("EnvPool");
}

}  // namespace mbh
