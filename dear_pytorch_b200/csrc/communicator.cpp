// communicator.cpp — see communicator.h.
#include "communicator.h"

#include <c10/cuda/CUDAStream.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include "dear_msg.h"
#include <stdexcept>

namespace dear {

#define DEAR_CHECK(cond, msg)                                                        \
  do {                                                                               \
    if (!(cond)) {                                                                   \
      dear::Msg _oss;                                                                     \
      _oss << "dear: " << msg;                                                       \
      throw std::runtime_error(_oss.str());                                          \
    }                                                                                \
  } while (0)

#define DEAR_CUDA(expr)                                                              \
  do {                                                                               \
    cudaError_t _e = (expr);                                                         \
    if (_e != cudaSuccess) {                                                         \
      dear::Msg _oss;                                                                     \
      _oss << "dear: CUDA error '" << cudaGetErrorString(_e) << "' in " #expr " ("   \
           << __FILE__ << ":" << __LINE__ << ")";                                    \
      throw std::runtime_error(_oss.str());                                          \
    }                                                                                \
  } while (0)

static inline cudaStream_t S(void* p) { return reinterpret_cast<cudaStream_t>(p); }
static inline cudaEvent_t E(void* p) { return reinterpret_cast<cudaEvent_t>(p); }

static cudaStream_t current_stream(int device) {
  return c10::cuda::getCurrentCUDAStream(static_cast<c10::DeviceIndex>(device)).stream();
}

static bool is_capturing(cudaStream_t s) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &st) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return st != cudaStreamCaptureStatusNone;
}

static cudaStream_t make_priority_stream() {
  int lo = 0, hi = 0;
  DEAR_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  cudaStream_t s;
  DEAR_CUDA(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, hi));
  return s;
}

static cudaEvent_t make_event() {
  cudaEvent_t e;
  DEAR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return e;
}

int dtype_of(const torch::Tensor& t) {
  switch (t.scalar_type()) {
    case torch::kFloat: return DT_F32;
    case torch::kBFloat16: return DT_BF16;
    case torch::kHalf: return DT_F16;
    default: return -1;
  }
}

static torch::ScalarType scalar_of(int dt) {
  switch (dt) {
    case DT_F32: return torch::kFloat;
    case DT_BF16: return torch::kBFloat16;
    case DT_F16: return torch::kHalf;
    default: throw std::runtime_error("dear: bad dtype");
  }
}

// ===========================================================================
// Communicator
// ===========================================================================
ArenaOptions Communicator::arena_options() const {
  ArenaOptions a;
  a.provider = is_cuda() ? static_cast<Provider>(opt_.provider) : Provider::HOST_SHM;
  a.want_multicast = opt_.multicast;
  a.device = opt_.device;
  a.timeout_s = opt_.rendezvous_timeout_s;
  return a;
}

std::string Communicator::unique_key(const std::string& what) {
  return name_ + "/" + what + "/" + std::to_string(key_seq_++);
}

Communicator::Communicator(int rank, int world, c10::intrusive_ptr<c10d::Store> store, std::string name,
                           CommOptions opt)
    : rank_(rank), world_(world), store_(std::move(store)), name_(std::move(name)), opt_(opt) {
  DEAR_CHECK(opt_.nstreams >= 1 && opt_.nstreams <= 16, "nstreams must be in [1,16]");
  if (is_cuda()) {
    DEAR_CHECK(cuda_runtime_usable(), "CUDA device requested but no CUDA runtime/driver is usable");
    DEAR_CUDA(cudaSetDevice(opt_.device));
  }
  for (int i = 0; i < opt_.nstreams; ++i) add_slot();
  (void)status_word_host();
}

void Communicator::add_slot() {
  arenas_.push_back(SymmArena::create(static_cast<size_t>(opt_.staging_bytes), rank_, world_, store_, unique_key("general"),
                                      arena_options()));
  Slot s;
  if (is_cuda()) {
    s.stream = make_priority_stream();
    s.ev_in = make_event();
    s.ev_out = make_event();
  }
  slots_.push_back(s);
}

void Communicator::extend_streams(int n) {
  DEAR_CHECK(n >= 1 && n <= 16, "nstreams must be in [1,16]");
  while (static_cast<int>(slots_.size()) < n) add_slot();
}

Communicator::~Communicator() {
  if (is_cuda()) {
    for (auto& s : slots_) {
      if (s.stream) {
        cudaStreamSynchronize(S(s.stream));
        cudaStreamDestroy(S(s.stream));
      }
      if (s.ev_in) cudaEventDestroy(E(s.ev_in));
      if (s.ev_out) cudaEventDestroy(E(s.ev_out));
    }
    cudaGetLastError();
  }
}

int Communicator::next_slot() {
  int s = cur_slot_;
  cur_slot_ = (cur_slot_ + 1) % static_cast<int>(slots_.size());
  return s;
}

void Communicator::check_status() {
  uint32_t* st = status_word_host();
  uint32_t v = __atomic_load_n(st, __ATOMIC_ACQUIRE);
  if (v != ST_OK) {
    __atomic_store_n(st, 0u, __ATOMIC_RELEASE);
    static const char* names[] = {"ok", "reduce-scatter: peers never packed", "reduce-scatter: peers never released the bucket",
                                  "all-gather: peers never arrived", "all-gather: peers never pushed", "general collective"};
    std::string msg = "dear: rank " + std::to_string(rank_) + ": cross-GPU wait timed out (";
    msg += (v < 6 ? names[v] : "unknown");
    msg += ", code " + std::to_string(v) +
           "); a peer is missing, crashed, or issued collectives in a different order";
    throw std::runtime_error(msg);
  }
}

void Communicator::gen_chunked(int slot, int op, const char* src, char* dst, uint64_t nelems, int dtype,
                               uint32_t elem_bytes, int root_or_peer, float scale, uint64_t dst_stride_elems) {
  SymmArena& arena = *arenas_.at(slot);
  GenParams p;
  std::memset(&p, 0, sizeof(p));
  p.stage = arena.data_table(0);
  p.mc_stage = nullptr;
  p.op = op;
  p.root_or_peer = root_or_peer;
  p.scale = scale;
  p.ready_chan = 1;
  p.done_chan = 2;
  p.sig = arena.sig_table();
  p.ctrl = arena.ctrl();
  p.rank = rank_;
  p.world = world_;
  p.dtype = dtype < 0 ? DT_F32 : dtype;
  p.elem_bytes = elem_bytes;
  p.status = is_cuda() ? status_word_device() : status_word_host();
  p.timeout_ns = timeout_ns();
  p.dst_stride_bytes = dst_stride_elems * elem_bytes;

  const uint64_t max_elems = (static_cast<uint64_t>(opt_.staging_bytes) / elem_bytes) & ~uint64_t(15);
  uint64_t done = 0;
  do {
    const uint64_t n = std::min<uint64_t>(nelems - done, max_elems);
    p.src = src ? src + done * elem_bytes : nullptr;
    p.dst = dst ? dst + done * elem_bytes : nullptr;
    p.nelems = n;
    if (is_cuda()) {
      int grid = static_cast<int>(std::min<uint64_t>(std::max<uint64_t>(1, (n * elem_bytes) / (16 * 512 * 4)), opt_.gen_grid));
      launch_gen(p, grid, S(slots_[slot].stream));
    } else {
      emu_gen(p);
    }
    count_launch();
    done += n;
  } while (done < nelems);
}

int Communicator::run_gen(int op, const void* src, void* dst, uint64_t nelems, int dtype, uint32_t elem_bytes,
                          int root_or_peer, float scale) {
  const int slot = next_slot();
  cudaStream_t cur = nullptr;
  if (is_cuda()) {
    cur = current_stream(opt_.device);
    DEAR_CUDA(cudaEventRecord(E(slots_[slot].ev_in), cur));
    DEAR_CUDA(cudaStreamWaitEvent(S(slots_[slot].stream), E(slots_[slot].ev_in), 0));
  }
  gen_chunked(slot, op, reinterpret_cast<const char*>(src), reinterpret_cast<char*>(dst), nelems, dtype, elem_bytes,
              root_or_peer, scale, 0);
  if (is_cuda()) DEAR_CUDA(cudaEventRecord(E(slots_[slot].ev_out), S(slots_[slot].stream)));
  return slot;
}

static void check_tensor(const torch::Tensor& t, bool cuda, int device, const char* what) {
  DEAR_CHECK(t.is_contiguous(), what << ": tensor must be contiguous");
  if (cuda) {
    DEAR_CHECK(t.is_cuda() && t.device().index() == device, what << ": tensor must live on cuda:" << device);
  } else {
    DEAR_CHECK(t.device().is_cpu(), what << ": tensor must be a CPU tensor for the host-emulation backend");
  }
}

int Communicator::allreduce_(torch::Tensor t, double scale) {
  check_tensor(t, is_cuda(), opt_.device, "allreduce");
  const int dt = dtype_of(t);
  DEAR_CHECK(dt >= 0, "allreduce: dtype must be float32/bfloat16/float16");
  return run_gen(GEN_ALLREDUCE, t.data_ptr(), t.data_ptr(), t.numel(), dt, t.element_size(), 0, static_cast<float>(scale));
}

int Communicator::reduce_(torch::Tensor t, int root, double scale) {
  check_tensor(t, is_cuda(), opt_.device, "reduce");
  const int dt = dtype_of(t);
  DEAR_CHECK(dt >= 0, "reduce: dtype must be float32/bfloat16/float16");
  DEAR_CHECK(root >= 0 && root < world_, "reduce: bad root");
  return run_gen(GEN_REDUCE, t.data_ptr(), t.data_ptr(), t.numel(), dt, t.element_size(), root, static_cast<float>(scale));
}

int Communicator::bcast_(torch::Tensor t, int root) {
  check_tensor(t, is_cuda(), opt_.device, "bcast");
  DEAR_CHECK(root >= 0 && root < world_, "bcast: bad root");
  // raw byte move: any dtype (fp32, int64 for BN num_batches_tracked, ...)
  return run_gen(GEN_BCAST, t.data_ptr(), rank_ == root ? nullptr : t.data_ptr(), t.numel(), DT_F32, t.element_size(), root, 1.f);
}

int Communicator::sendrecv(torch::Tensor send, torch::Tensor recv, int peer) {
  check_tensor(send, is_cuda(), opt_.device, "sendrecv(send)");
  check_tensor(recv, is_cuda(), opt_.device, "sendrecv(recv)");
  DEAR_CHECK(send.numel() == recv.numel() && send.element_size() == recv.element_size(), "sendrecv: size mismatch");
  DEAR_CHECK(peer >= 0 && peer < world_, "sendrecv: bad peer");
  return run_gen(GEN_SENDRECV, send.data_ptr(), recv.data_ptr(), send.numel(), DT_F32, send.element_size(), peer, 1.f);
}

int Communicator::device_barrier() { return run_gen(GEN_BARRIER, nullptr, nullptr, 0, DT_F32, 4, 0, 1.f); }

int Communicator::allgather(torch::Tensor send, torch::Tensor recv) {
  check_tensor(send, is_cuda(), opt_.device, "allgather(send)");
  check_tensor(recv, is_cuda(), opt_.device, "allgather(recv)");
  DEAR_CHECK(recv.numel() == send.numel() * world_ && send.element_size() == recv.element_size(),
             "allgather: recv must hold world*send elements");
  const int slot = next_slot();
  if (is_cuda()) {
    DEAR_CUDA(cudaEventRecord(E(slots_[slot].ev_in), current_stream(opt_.device)));
    DEAR_CUDA(cudaStreamWaitEvent(S(slots_[slot].stream), E(slots_[slot].ev_in), 0));
  }
  gen_chunked(slot, GEN_ALLGATHER, reinterpret_cast<const char*>(send.data_ptr()), reinterpret_cast<char*>(recv.data_ptr()),
              send.numel(), DT_F32, send.element_size(), 0, 1.f, send.numel());
  if (is_cuda()) DEAR_CUDA(cudaEventRecord(E(slots_[slot].ev_out), S(slots_[slot].stream)));
  return slot;
}

int Communicator::reduce_scatter(torch::Tensor send, torch::Tensor recv, double scale) {
  check_tensor(send, is_cuda(), opt_.device, "reduce_scatter(send)");
  check_tensor(recv, is_cuda(), opt_.device, "reduce_scatter(recv)");
  const int dt = dtype_of(send);
  DEAR_CHECK(dt >= 0 && dtype_of(recv) == dt, "reduce_scatter: dtype must be float32/bfloat16/float16");
  DEAR_CHECK(send.numel() == recv.numel() * world_, "reduce_scatter: send must hold world*recv elements");
  const int slot = next_slot();
  const uint64_t per = recv.numel();
  const uint32_t eb = send.element_size();
  const char* sp = reinterpret_cast<const char*>(send.data_ptr());
  char* rp = reinterpret_cast<char*>(recv.data_ptr());
  char* stage = arenas_.at(slot)->local_data();
  cudaStream_t st = is_cuda() ? S(slots_[slot].stream) : nullptr;
  if (is_cuda()) {
    DEAR_CUDA(cudaEventRecord(E(slots_[slot].ev_in), current_stream(opt_.device)));
    DEAR_CUDA(cudaStreamWaitEvent(st, E(slots_[slot].ev_in), 0));
  }
  // chunk over the shard so that world*chunk fits the staging buffer
  const uint64_t max_chunk = ((static_cast<uint64_t>(opt_.staging_bytes) / eb / world_) & ~uint64_t(15));
  DEAR_CHECK(max_chunk > 0, "staging buffer too small");
  for (uint64_t a = 0; a < per || a == 0; a += max_chunk) {
    const uint64_t n = std::min<uint64_t>(per - a, max_chunk);
    if (n == 0) break;
    // gather the P row-chunks contiguously into my staging buffer
    // NOTE: the previous op on this slot may still be read by peers; the
    // kernel's step (0) waits for them, so the staging copy must happen inside
    // the same stream AFTER a device barrier on the done flags: we run a
    // zero-size barrier op first to inherit that guarantee.
    gen_chunked(slot, GEN_BARRIER, nullptr, nullptr, 0, DT_F32, 4, 0, 1.f, 0);
    for (int q = 0; q < world_; ++q) {
      const char* s = sp + (uint64_t(q) * per + a) * eb;
      char* d = stage + uint64_t(q) * n * eb;
      if (is_cuda()) DEAR_CUDA(cudaMemcpyAsync(d, s, n * eb, cudaMemcpyDeviceToDevice, st));
      else std::memcpy(d, s, n * eb);
    }
    gen_chunked(slot, GEN_REDUCE_SCATTER, nullptr, rp + a * eb, n * world_, dt, eb, 0, static_cast<float>(scale), 0);
  }
  if (is_cuda()) DEAR_CUDA(cudaEventRecord(E(slots_[slot].ev_out), st));
  return slot;
}

int Communicator::allreduce_rsag_(torch::Tensor t, double scale) {
  // all-reduce as reduce-scatter followed by all-gather (reference communicator.cpp:198-235)
  const int64_t n = t.numel();
  if (n < world_ || n % world_ != 0) return allreduce_(t, scale);   // the reference pads; we fall back
  auto flat = t.view({-1});
  const int64_t per = n / world_;
  auto shard = flat.narrow(0, rank_ * per, per);
  auto tmp = torch::empty_like(shard);
  const int h = reduce_scatter(flat, tmp, scale);
  wait_stream(h);
  const int h2 = allgather(tmp, flat);
  wait_stream(h2);   // `tmp` is freed in current-stream order, i.e. after the all-gather consumed it
  return h2;
}

int Communicator::allreduce_rb_(torch::Tensor t, double scale) {
  // all-reduce as reduce(root 0) + broadcast(root 0) (reference communicator.cpp:185-196)
  int h = reduce_(t, 0, scale);
  wait_stream(h);
  return bcast_(t, 0);
}

void Communicator::synchronize() {
  if (is_cuda())
    for (auto& s : slots_) DEAR_CUDA(cudaStreamSynchronize(S(s.stream)));
  check_status();
}

void Communicator::sync_stream(int handle) {
  DEAR_CHECK(handle >= 0 && handle < static_cast<int>(slots_.size()), "bad stream handle");
  if (is_cuda()) DEAR_CUDA(cudaStreamSynchronize(S(slots_[handle].stream)));
  check_status();
}

void Communicator::wait_stream(int handle) {
  DEAR_CHECK(handle >= 0 && handle < static_cast<int>(slots_.size()), "bad stream handle");
  if (is_cuda()) DEAR_CUDA(cudaStreamWaitEvent(current_stream(opt_.device), E(slots_[handle].ev_out), 0));
}

int Communicator::num_free_streams() {
  if (!is_cuda()) return static_cast<int>(slots_.size());
  int n = 0;
  for (auto& s : slots_) {
    cudaError_t e = cudaStreamQuery(S(s.stream));
    if (e == cudaSuccess) ++n; else if (e != cudaErrorNotReady) DEAR_CUDA(e);
  }
  cudaGetLastError();
  return n;
}

void Communicator::barrier() {
  if (world_ == 1) return;
  const std::string base = name_ + "/hostbar/" + std::to_string(barrier_seq_++) + "/";
  store_->set(base + std::to_string(rank_), std::vector<uint8_t>{1});
  std::vector<std::string> keys;
  for (int r = 0; r < world_; ++r) keys.push_back(base + std::to_string(r));
  store_->wait(keys, std::chrono::milliseconds(static_cast<int64_t>(opt_.rendezvous_timeout_s * 1000)));
}

// ===========================================================================
// BucketSet
// ===========================================================================
BucketSet::BucketSet(std::shared_ptr<Communicator> comm, std::vector<int64_t> padded_numels, int dtype,
                     bool with_grad_buckets)
    : comm_(std::move(comm)), dtype_(dtype), with_grad_(with_grad_buckets) {
  const int world = comm_->size();
  const size_t es = dtype_size(dtype);
  DEAR_CHECK(static_cast<int>(padded_numels.size()) * kChannelsPerBucket + kGeneralChannels <= kNumChannels,
             "too many buckets (" << static_cast<long long>(padded_numels.size()) << ")");
  size_t off = 0;
  for (int64_t n : padded_numels) {
    DEAR_CHECK(n > 0 && n % world == 0, "bucket size must be a positive multiple of the world size");
    const int64_t shard = n / world;
    DEAR_CHECK((shard * es) % 16 == 0, "shard bytes must be a multiple of 16");
    Bucket b;
    b.padded = n;
    b.shard = shard;
    b.param_off = off;
    off += (n * es + 255) / 256 * 256;
    if (with_grad_) {
      b.grad_off = off;
      off += (n * es + 255) / 256 * 256;
    }
    buckets_.push_back(std::move(b));
  }
  arena_ = SymmArena::create(off, comm_->rank(), world, comm_->store(), comm_->unique_key("buckets"),
                             comm_->arena_options());
  // ---- per-bucket reduce-scatter plan (north star: "picked per bucket size") -------------------------------
  const CommOptions& o = comm_->options();
  for (auto& b : buckets_) {
    const int64_t bytes = b.padded * static_cast<int64_t>(es);
    const int64_t shard_bytes = b.shard * static_cast<int64_t>(es);
    int algo = o.rs_algo;
    if (algo < 0) algo = (world > 1 && bytes >= o.pipe_min_bytes) ? RS_ALGO_PIPE : RS_ALGO_ONESHOT;
    // (the host emulation runs one algorithm; a FORCED pipe plan is still built there so that the stripe-major work
    // list of set_pack can be tested without a GPU)
    if (world == 1 || (!comm_->is_cuda() && o.rs_algo != RS_ALGO_PIPE)) algo = RS_ALGO_ONESHOT;
    if (algo == RS_ALGO_NVLS && !arena_->has_multicast()) algo = RS_ALGO_ONESHOT;
    b.rs_algo = algo;
    if (algo == RS_ALGO_PIPE) {
      int64_t k = std::max<int64_t>(1, std::min<int64_t>(16, bytes / std::max<int64_t>(1, o.stripe_target_bytes)));
      int64_t cs = (shard_bytes + k - 1) / k;
      cs = (cs + kPipePackPiece - 1) / kPipePackPiece * kPipePackPiece;
      b.stripe_bytes = static_cast<uint64_t>(cs);
      b.nstripes = static_cast<uint32_t>((shard_bytes + cs - 1) / cs);
      // one CTA per 16 KB chunk of a stripe is the most that can be busy
      const int64_t chunks = std::max<int64_t>(1, std::min<int64_t>(cs, shard_bytes) / kPipeChunk);
      b.rs_grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(o.rs_grid, chunks)));
    } else {
      b.nstripes = 1;
      b.stripe_bytes = static_cast<uint64_t>(shard_bytes);
      b.rs_grid = grid_for(bytes, (world > 1 && bytes >= o.big_bucket_bytes) ? std::max(o.rs_grid, o.rs_grid_big) : o.rs_grid);
    }
  }
  if (comm_->is_cuda()) {
    stream_ = make_priority_stream();
    ag_stream_ = o.separate_ag_stream ? make_priority_stream() : stream_;
    ev_fence_ = make_event();
    ev_fence_ag_ = make_event();
    for (auto& b : buckets_) {
      b.ev_in = make_event();
      b.rs_done = make_event();
      b.ag_done = make_event();
      for (auto* st : {&b.stage_pack, &b.stage_hyper}) {
        st->ev[0] = make_event();
        st->ev[1] = make_event();
      }
    }
  }
}

BucketSet::~BucketSet() {
  if (comm_->is_cuda()) {
    if (stream_) cudaStreamSynchronize(S(stream_));
    if (ag_stream_) cudaStreamSynchronize(S(ag_stream_));
    for (auto& b : buckets_) {
      for (void* e : {b.ev_in, b.rs_done, b.ag_done}) if (e) cudaEventDestroy(E(e));
      for (auto* st : {&b.stage_pack, &b.stage_hyper}) {
        for (void* e : st->ev) if (e) cudaEventDestroy(E(e));
        for (void* p : st->pinned) if (p) cudaFreeHost(p);
      }
      for (void* p : b.captured_tables) cudaFree(p);
      if (b.pack_dev) cudaFree(b.pack_dev);
      if (b.hyper_dev) cudaFree(b.hyper_dev);
    }
    if (ev_fence_) cudaEventDestroy(E(ev_fence_));
    if (ev_fence_ag_) cudaEventDestroy(E(ev_fence_ag_));
    if (upload_stream_) cudaStreamDestroy(S(upload_stream_));
    if (ag_stream_ && ag_stream_ != stream_) {
      cudaStreamSynchronize(S(ag_stream_));
      cudaStreamDestroy(S(ag_stream_));
    }
    if (stream_) cudaStreamDestroy(S(stream_));
    cudaGetLastError();
  }
}

static torch::Tensor wrap(char* ptr, int64_t numel, int dtype, bool cuda, int device, std::shared_ptr<SymmArena> keep) {
  auto opts = torch::TensorOptions().dtype(scalar_of(dtype));
  if (cuda) opts = opts.device(torch::kCUDA, device);
  return torch::from_blob(ptr, {numel}, [keep](void*) mutable { keep.reset(); }, opts);
}

torch::Tensor BucketSet::param_buffer(int g) {
  auto& b = buckets_.at(g);
  return wrap(arena_->local_data() + b.param_off, b.padded, dtype_, comm_->is_cuda(), comm_->options().device, arena_);
}

torch::Tensor BucketSet::grad_buffer(int g) {
  DEAR_CHECK(with_grad_, "this BucketSet has no gradient buckets");
  auto& b = buckets_.at(g);
  return wrap(arena_->local_data() + b.grad_off, b.padded, dtype_, comm_->is_cuda(), comm_->options().device, arena_);
}

void BucketSet::set_step(int g, int64_t t) {
  buckets_.at(g);
  const uint32_t v = static_cast<uint32_t>(t);
  uint32_t* dst = arena_->ctrl() + 2 * kNumChannels + g;
  if (comm_->is_cuda()) {
    DEAR_CUDA(cudaStreamSynchronize(S(stream_)));
    if (ag_stream_ != stream_) DEAR_CUDA(cudaStreamSynchronize(S(ag_stream_)));
    DEAR_CUDA(cudaMemcpy(dst, &v, sizeof(v), cudaMemcpyHostToDevice));
  } else {
    *dst = v;
  }
}

void BucketSet::set_shards(int g, torch::Tensor grad_shard, std::optional<torch::Tensor> mom,
                           std::optional<torch::Tensor> master, std::optional<torch::Tensor> var) {
  auto& b = buckets_.at(g);
  auto chk = [&](const torch::Tensor& t, const char* what) {
    DEAR_CHECK(t.scalar_type() == torch::kFloat && t.is_contiguous() && t.numel() == b.shard,
               what << " must be a contiguous float32 tensor of " << b.shard << " elements");
    DEAR_CHECK(t.is_cuda() == comm_->is_cuda(), what << " is on the wrong device type");
  };
  chk(grad_shard, "grad_shard");
  b.grad_shard = grad_shard;
  b.mom = torch::Tensor();
  b.master = torch::Tensor();
  if (mom.has_value() && mom->defined()) { chk(*mom, "momentum shard"); b.mom = *mom; }
  if (master.has_value() && master->defined()) { chk(*master, "master shard"); b.master = *master; }
  b.var = torch::Tensor();
  if (var.has_value() && var->defined()) { chk(*var, "second-moment shard"); b.var = *var; }
  // (low-precision buckets must have a master shard by the time allgather_update() runs)
}

void BucketSet::upload(Bucket& b, bool is_pack, const void* host, size_t bytes, void** dev, size_t* cap) {
  if (bytes == 0) return;
  const cudaStream_t cur = current_stream(comm_->options().device);
  // a capture may be in progress on the compute stream before the comm stream has joined it
  const bool capturing = is_capturing(S(stream_)) || is_capturing(cur);
  if (capturing) {
    //  * hyper-parameters must never be frozen into a graph (an LR scheduler could not change them any more):
    //    TrainStep uploads them before the capture starts and after every change, outside the graph;
    //  * a pack table holds the gradient addresses of THIS capture.  It gets a device buffer of its own that only the
    //    captured kernels ever read (the pointer is baked into their launch parameters), filled right now on a private
    //    stream outside the capture.  A replay therefore needs no H2D copy node — round 2 first used memcpy nodes, and
    //    in the end-to-end benchmark they queued behind the 38 MB batch upload on the same copy engine — and eager
    //    steps between replays keep using (and overwriting) the bucket's ordinary table without disturbing the graph.
    DEAR_CHECK(is_pack, "optimizer hyper-parameters changed during CUDA-graph capture; upload them before capturing "
                        "(DearEngine.refresh_hyper_outside_graph)");
    void* dtab = nullptr;
    void* pin = nullptr;
    cudaError_t err = cudaSuccess;
    {
      // allocation / synchronisation calls are "potentially unsafe" under a thread-local capture: relax the mode
      cudaStreamCaptureMode mode = cudaStreamCaptureModeRelaxed;
      DEAR_CUDA(cudaThreadExchangeStreamCaptureMode(&mode));
      if (upload_stream_ == nullptr) {
        cudaStream_t us;
        err = cudaStreamCreateWithFlags(&us, cudaStreamNonBlocking);
        if (err == cudaSuccess) upload_stream_ = us;
      }
      if (err == cudaSuccess) err = cudaMalloc(&dtab, bytes);
      if (err == cudaSuccess) err = cudaHostAlloc(&pin, bytes, cudaHostAllocDefault);
      if (err == cudaSuccess) {
        std::memcpy(pin, host, bytes);
        err = cudaMemcpyAsync(dtab, pin, bytes, cudaMemcpyHostToDevice, S(upload_stream_));
      }
      if (err == cudaSuccess) err = cudaStreamSynchronize(S(upload_stream_));
      if (pin) cudaFreeHost(pin);
      if (err != cudaSuccess && dtab != nullptr) { cudaFree(dtab); dtab = nullptr; }   // nothing leaks on the error path
      cudaThreadExchangeStreamCaptureMode(&mode);
    }
    DEAR_CUDA(err);
    b.captured_tables.push_back(dtab);
    b.capture_table = dtab;
    b.eager_table_stale = true;      // pack_host now mirrors the capture's table, not what pack_dev holds
    return;
  }
  if (*cap < bytes) {
    // the old table may still be read by an in-flight kernel on the comm streams
    DEAR_CUDA(cudaStreamSynchronize(S(stream_)));
    if (ag_stream_ != stream_) DEAR_CUDA(cudaStreamSynchronize(S(ag_stream_)));
    if (*dev) DEAR_CUDA(cudaFree(*dev));
    size_t ncap = std::max<size_t>(bytes * 2, 4096);
    DEAR_CUDA(cudaMalloc(dev, ncap));
    *cap = ncap;
  }
  if (is_pack) b.eager_table_stale = false;
  if (!is_pack && ag_stream_ != stream_) {
    // the hyper table is read by update kernels on the all-gather stream: overwrite it only after they finished
    DEAR_CUDA(cudaEventRecord(E(ev_fence_ag_), S(ag_stream_)));
    DEAR_CUDA(cudaStreamWaitEvent(S(stream_), E(ev_fence_ag_), 0));
  }
  Bucket::Staging& st = is_pack ? b.stage_pack : b.stage_hyper;
  const int slot = st.next;
  st.next ^= 1;
  DEAR_CUDA(cudaEventSynchronize(E(st.ev[slot])));   // the copy that last read this slot; normally long complete
  if (st.cap[slot] < bytes) {
    if (st.pinned[slot]) DEAR_CUDA(cudaFreeHost(st.pinned[slot]));
    size_t ncap = std::max<size_t>(bytes * 2, 4096);
    DEAR_CUDA(cudaHostAlloc(&st.pinned[slot], ncap, cudaHostAllocDefault));
    st.cap[slot] = ncap;
  }
  std::memcpy(st.pinned[slot], host, bytes);
  DEAR_CUDA(cudaMemcpyAsync(*dev, st.pinned[slot], bytes, cudaMemcpyHostToDevice, S(stream_)));
  DEAR_CUDA(cudaEventRecord(E(st.ev[slot]), S(stream_)));
}

bool BucketSet::set_pack(int g, const std::vector<int64_t>& src_ptrs, const std::vector<int64_t>& dst_off_bytes,
                         const std::vector<int64_t>& nbytes, const std::vector<int64_t>& flags) {
  auto& b = buckets_.at(g);
  const size_t n = src_ptrs.size();
  DEAR_CHECK(dst_off_bytes.size() == n && nbytes.size() == n && flags.size() == n, "set_pack: ragged arguments");
  const size_t es = dtype_size(dtype_);
  std::vector<PackSeg> segs;
  segs.reserve(n);
  uint32_t tiles = 0;
  bool inplace = false;
  // the stripe-pipelined kernel walks the table in bucket order
  std::vector<size_t> order(n);
  for (size_t i = 0; i < n; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b2) { return dst_off_bytes[a] < dst_off_bytes[b2]; });
  for (size_t oi = 0; oi < n; ++oi) {
    const size_t i = order[oi];
    if (nbytes[i] == 0) continue;
    if (src_ptrs[i] == 0 && !(flags[i] & SEG_ZERO_FILL)) { inplace = true; continue; }   // already in the bucket
    PackSeg s;
    s.src = reinterpret_cast<const void*>(static_cast<uintptr_t>(src_ptrs[i]));
    s.dst_off = static_cast<uint64_t>(dst_off_bytes[i]);
    s.nbytes = static_cast<uint64_t>(nbytes[i]);
    s.tile_begin = tiles;
    s.flags = static_cast<uint32_t>(flags[i]);
    DEAR_CHECK(s.dst_off % 16 == 0, "set_pack: destination offsets must be 16-byte aligned");
    DEAR_CHECK((reinterpret_cast<uintptr_t>(s.src) % 16) == 0, "set_pack: gradient storage must be 16-byte aligned");
    DEAR_CHECK(s.nbytes % 2 == 0 && s.dst_off + s.nbytes <= static_cast<uint64_t>(b.padded) * es, "set_pack: segment out of range");
    DEAR_CHECK(segs.empty() || segs.back().dst_off + segs.back().nbytes <= s.dst_off, "set_pack: segments overlap");
    tiles += static_cast<uint32_t>((s.nbytes + kPackTileBytes - 1) / kPackTileBytes);
    segs.push_back(s);
  }
  const bool same = segs.size() == b.pack_host.size() &&
                    (segs.empty() || std::memcmp(segs.data(), b.pack_host.data(), segs.size() * sizeof(PackSeg)) == 0);
  b.pack_inplace = inplace;
  // (a capture always builds its own table; an eager call after a capture must refresh the bucket's table)
  const bool capturing_now = comm_->is_cuda() && (is_capturing(S(stream_)) || is_capturing(current_stream(comm_->options().device)));
  if (same && !b.eager_table_stale && !capturing_now) return false;
  b.pack_host = std::move(segs);
  b.ntiles = tiles;
  if (b.rs_algo == RS_ALGO_PIPE) {
    // work list of the pipelined kernel: every segment cut at shard and stripe boundaries and into pieces of at
    // most kPipePackPiece bytes, ordered stripe-major (stripe k of EVERY shard before stripe k+1)
    const uint64_t SB = static_cast<uint64_t>(b.shard) * es, cs = b.stripe_bytes;
    std::vector<std::vector<PackSeg>> per_stripe(b.nstripes);
    for (const PackSeg& sg : b.pack_host) {
      uint64_t o = sg.dst_off;
      const uint64_t end = sg.dst_off + sg.nbytes;
      while (o < end) {
        const uint64_t in_shard = o % SB;
        const uint64_t k = in_shard / cs;
        const uint64_t stripe_end = o - in_shard + std::min<uint64_t>(SB, (k + 1) * cs);
        const uint64_t n = std::min<uint64_t>({end - o, stripe_end - o, static_cast<uint64_t>(kPipePackPiece)});
        PackSeg pc = sg;
        pc.src = sg.src ? reinterpret_cast<const char*>(sg.src) + (o - sg.dst_off) : nullptr;
        pc.dst_off = o;
        pc.nbytes = n;
        pc.tile_begin = static_cast<uint32_t>(k);
        per_stripe.at(k).push_back(pc);
        o += n;
      }
    }
    b.pieces_host.clear();
    for (uint32_t k = 0; k < b.nstripes; ++k) {
      b.piece_first[k] = static_cast<uint32_t>(b.pieces_host.size());
      b.pieces_host.insert(b.pieces_host.end(), per_stripe[k].begin(), per_stripe[k].end());
    }
    for (uint32_t k = b.nstripes; k < 17; ++k) b.piece_first[k] = static_cast<uint32_t>(b.pieces_host.size());
    if (comm_->is_cuda())
      upload(b, true, b.pieces_host.data(), b.pieces_host.size() * sizeof(PackSeg), reinterpret_cast<void**>(&b.pack_dev), &b.pack_cap);
    return true;
  }
  if (comm_->is_cuda())
    upload(b, true, b.pack_host.data(), b.pack_host.size() * sizeof(PackSeg), reinterpret_cast<void**>(&b.pack_dev), &b.pack_cap);
  return true;
}

bool BucketSet::set_hyper(int g, const std::vector<int64_t>& ends, const std::vector<double>& lr,
                          const std::vector<double>& wd, const std::vector<double>& mom,
                          const std::vector<double>& damp, const std::vector<int64_t>& nesterov,
                          const std::vector<int64_t>& opt, const std::vector<double>& beta2, const std::vector<double>& eps) {
  auto& b = buckets_.at(g);
  const size_t n = ends.size();
  DEAR_CHECK(n >= 1 && lr.size() == n && wd.size() == n && mom.size() == n && damp.size() == n && nesterov.size() == n,
             "set_hyper: ragged arguments");
  std::vector<HyperSeg> segs(n);
  for (size_t i = 0; i < n; ++i) {
    segs[i].end = static_cast<uint64_t>(ends[i]);
    segs[i].lr = static_cast<float>(lr[i]);
    segs[i].weight_decay = static_cast<float>(wd[i]);
    segs[i].momentum = static_cast<float>(mom[i]);
    segs[i].dampening = static_cast<float>(damp[i]);
    segs[i].nesterov = static_cast<uint32_t>(nesterov[i]) & (HYPER_NESTEROV | HYPER_SKIP);
    segs[i].opt = i < opt.size() ? static_cast<uint32_t>(opt[i]) : OPT_SGD;
    segs[i].beta2 = i < beta2.size() ? static_cast<float>(beta2[i]) : 0.f;
    segs[i].eps = i < eps.size() ? static_cast<float>(eps[i]) : 0.f;
    DEAR_CHECK(i == 0 || segs[i].end > segs[i - 1].end, "set_hyper: segment ends must increase");
  }
  DEAR_CHECK(segs.back().end >= static_cast<uint64_t>(b.padded), "set_hyper: segments must cover the bucket");
  const bool same = segs.size() == b.hyper_host.size() &&
                    std::memcmp(segs.data(), b.hyper_host.data(), segs.size() * sizeof(HyperSeg)) == 0;
  bool any_adam = false, all_adam = true;
  for (const auto& sg : segs) { any_adam |= sg.opt != OPT_SGD; all_adam &= sg.opt != OPT_SGD; }
  DEAR_CHECK(!any_adam || all_adam, "a bucket cannot mix SGD and Adam parameter groups");
  b.adam = all_adam;
  if (same) return false;
  b.hyper_host = std::move(segs);
  if (comm_->is_cuda())
    upload(b, false, b.hyper_host.data(), b.hyper_host.size() * sizeof(HyperSeg), reinterpret_cast<void**>(&b.hyper_dev), &b.hyper_cap);
  return true;
}

int BucketSet::grid_for(int64_t bytes, int max_grid) const {
  int64_t g = (bytes + (512 * 16 * 8) - 1) / (512 * 16 * 8);
  if (g < 1) g = 1;
  if (g > max_grid) g = max_grid;
  return static_cast<int>(g);
}

void BucketSet::fence_current_to_comm() {
  if (!comm_->is_cuda()) return;
  DEAR_CUDA(cudaEventRecord(E(ev_fence_), current_stream(comm_->options().device)));
  DEAR_CUDA(cudaStreamWaitEvent(S(stream_), E(ev_fence_), 0));
  if (ag_stream_ != stream_) DEAR_CUDA(cudaStreamWaitEvent(S(ag_stream_), E(ev_fence_), 0));
}

void BucketSet::reduce_scatter(int g, bool pack) {
  auto& b = buckets_.at(g);
  DEAR_CHECK(with_grad_, "reduce_scatter needs gradient buckets");
  DEAR_CHECK(b.grad_shard.defined(), "set_shards() must be called before reduce_scatter()");
  RSParams p;
  std::memset(&p, 0, sizeof(p));
  p.grad = arena_->data_table(b.grad_off);
  p.mc_grad = arena_->has_multicast() ? arena_->mc_data() + b.grad_off : nullptr;
  p.out = b.grad_shard.data_ptr<float>();
  p.shard_elems = static_cast<uint64_t>(b.shard);
  p.scale = grad_scale_ / static_cast<float>(comm_->size());
  const bool cuda = comm_->is_cuda();
  // a capturing launch reads the capture's private table (set by set_pack during this capture)
  const bool cap_now = cuda && is_capturing(current_stream(comm_->options().device));
  PackSeg* table_dev = (cap_now && b.capture_table != nullptr) ? static_cast<PackSeg*>(b.capture_table) : b.pack_dev;
  if (pack && !b.pack_host.empty()) {
    p.segs = cuda ? table_dev : b.pack_host.data();
    p.nseg = static_cast<uint32_t>(b.pack_host.size());
    p.ntiles = b.ntiles;
    // one GPU: the pack writes the fp32 shard directly (fp32: copy; bf16 / fp16: widening, CUDA kernel only).  The
    // fp32 copy cannot apply a gradient scale (1/loss_scale), so a scaled fp32 bucket packs into the gradient bucket
    // and the reduce pass applies the scale.
    const bool direct_ok = dtype_ == DT_F32 ? grad_scale_ == 1.f : cuda;
    p.direct_out = (comm_->size() == 1 && direct_ok && !b.pack_inplace) ? 1u : 0u;
  }
  p.sig = arena_->sig_table();
  p.ctrl = arena_->ctrl();
  p.bucket = static_cast<uint32_t>(g);
  p.rank = comm_->rank();
  p.world = comm_->size();
  p.dtype = dtype_;
  p.status = cuda ? status_word_device() : status_word_host();
  p.timeout_ns = comm_->timeout_ns();
  if (b.rs_algo == RS_ALGO_PIPE) {
    // stripe-pipelined variant: stripe-major work list instead of the segment table (device kernel and host emulation)
    p.nstripes = b.nstripes;
    p.stripe_bytes = b.stripe_bytes;
    p.mc_grad = nullptr;
    p.pieces = (pack && !b.pieces_host.empty()) ? (cuda ? table_dev : b.pieces_host.data()) : nullptr;
    std::memcpy(p.piece_first, b.piece_first, sizeof(p.piece_first));
    p.segs = nullptr;
    p.nseg = 0;
    p.ntiles = 0;
    p.direct_out = 0;
  }
  if (cuda) {
    DEAR_CUDA(cudaEventRecord(E(b.ev_in), current_stream(comm_->options().device)));
    DEAR_CUDA(cudaStreamWaitEvent(S(stream_), E(b.ev_in), 0));
    // the previous update kernel of this bucket (other stream) must have consumed the reduced shard it overwrites
    // (a capturing stream may only wait on events of its own capture, and vice versa; across that boundary the
    // capture / replay is ordered after the eager work by the stream it is launched on)
    if (ag_stream_ != stream_ && b.ag_pending && b.ag_done_captured == is_capturing(S(stream_)))
      DEAR_CUDA(cudaStreamWaitEvent(S(stream_), E(b.ag_done), 0));
    if (b.rs_algo == RS_ALGO_PIPE) {
      launch_rs_pipe(p, b.rs_grid, S(stream_));
    } else {
      if (b.rs_algo != RS_ALGO_NVLS) p.mc_grad = nullptr;
      launch_rs(p, b.rs_grid, S(stream_));
    }
    DEAR_CUDA(cudaEventRecord(E(b.rs_done), S(stream_)));
  } else {
    emu_rs(p);
  }
  b.rs_pending = true;
  comm_->count_launch();
}

void BucketSet::allgather_update(int g, bool do_update, bool first_step, bool entry_barrier, bool zero_grad) {
  auto& b = buckets_.at(g);
  const bool cuda = comm_->is_cuda();
  AGParams p;
  std::memset(&p, 0, sizeof(p));
  p.param = arena_->data_table(b.param_off);
  p.mc_param = arena_->has_multicast() ? arena_->mc_data() + b.param_off : nullptr;
  if (do_update) {
    DEAR_CHECK(b.grad_shard.defined(), "set_shards() must be called before allgather_update()");
    DEAR_CHECK(!b.hyper_host.empty(), "set_hyper() must be called before allgather_update()");
    p.grad_shard = b.grad_shard.data_ptr<float>();
    p.mom_shard = b.mom.defined() ? b.mom.data_ptr<float>() : nullptr;
    p.adam = b.adam ? 1u : 0u;
    if (b.adam) {
      DEAR_CHECK(b.mom.defined() && b.var.defined(), "Adam needs exp_avg and exp_avg_sq shards (set_shards)");
      p.var_shard = b.var.data_ptr<float>();
    }
    p.step_ctr = arena_->ctrl() + 2 * kNumChannels + g;
    p.hyper = cuda ? b.hyper_dev : b.hyper_host.data();
    p.nhyper = static_cast<uint32_t>(b.hyper_host.size());
  }
  p.master_shard = b.master.defined() ? b.master.data_ptr<float>() : nullptr;
  DEAR_CHECK(dtype_ == DT_F32 || p.master_shard != nullptr, "low-precision parameter buckets need an fp32 master shard");
  if (zero_grad && with_grad_) {
    p.zero_grad = arena_->local_data() + b.grad_off;
    p.zero_bytes = static_cast<uint64_t>(b.padded) * dtype_size(dtype_);
  }
  p.shard_elems = static_cast<uint64_t>(b.shard);
  p.first_step = first_step ? 1u : 0u;
  p.entry_barrier = entry_barrier ? 1u : 0u;
  p.do_update = do_update ? 1u : 0u;
  p.sig = arena_->sig_table();
  p.ctrl = arena_->ctrl();
  p.bucket = static_cast<uint32_t>(g);
  p.rank = comm_->rank();
  p.world = comm_->size();
  p.dtype = dtype_;
  p.status = cuda ? status_word_device() : status_word_host();
  p.timeout_ns = comm_->timeout_ns();
  if (cuda) {
    if (ag_stream_ != stream_) {
      // everything queued on the reduce-scatter stream so far (this step's reduce-scatters, table uploads)
      DEAR_CUDA(cudaEventRecord(E(ev_fence_ag_), S(stream_)));
      DEAR_CUDA(cudaStreamWaitEvent(S(ag_stream_), E(ev_fence_ag_), 0));
    }
    launch_ag(p, grid_for(b.shard * 16, comm_->options().ag_grid), S(ag_stream_));
    DEAR_CUDA(cudaEventRecord(E(b.ag_done), S(ag_stream_)));
    b.ag_done_captured = is_capturing(S(ag_stream_));
  } else {
    emu_ag(p);
  }
  b.ag_pending = true;
  comm_->count_launch();
}

void BucketSet::wait_bucket(int g) {
  auto& b = buckets_.at(g);
  if (comm_->is_cuda() && b.ag_pending)
    DEAR_CUDA(cudaStreamWaitEvent(current_stream(comm_->options().device), E(b.ag_done), 0));
}

void BucketSet::wait_rs(int g) {
  auto& b = buckets_.at(g);
  if (comm_->is_cuda() && b.rs_pending)
    DEAR_CUDA(cudaStreamWaitEvent(current_stream(comm_->options().device), E(b.rs_done), 0));
}

void BucketSet::wait_all() {
  if (!comm_->is_cuda()) return;
  // each comm stream is ordered, so one fresh event per stream covers all buckets.  A capturing stream may only wait
  // on streams of the same capture (and an eager one only on eager streams): a comm stream on the other side of that
  // boundary has nothing this wait could be about — eager work precedes the capture, which TrainStep starts only
  // after a full synchronisation.
  const cudaStream_t cur = current_stream(comm_->options().device);
  const bool cc = is_capturing(cur);
  if (is_capturing(S(stream_)) == cc) {
    DEAR_CUDA(cudaEventRecord(E(ev_fence_), S(stream_)));
    DEAR_CUDA(cudaStreamWaitEvent(cur, E(ev_fence_), 0));
  }
  if (ag_stream_ != stream_ && is_capturing(S(ag_stream_)) == cc) {
    DEAR_CUDA(cudaEventRecord(E(ev_fence_ag_), S(ag_stream_)));
    DEAR_CUDA(cudaStreamWaitEvent(cur, E(ev_fence_ag_), 0));
  }
}

std::vector<std::vector<int64_t>> BucketSet::pack_pieces(int g) const {
  const auto& b = buckets_.at(g);
  std::vector<std::vector<int64_t>> out;
  for (const PackSeg& pc : b.pieces_host)
    out.push_back({static_cast<int64_t>(reinterpret_cast<uintptr_t>(pc.src)), static_cast<int64_t>(pc.dst_off),
                   static_cast<int64_t>(pc.nbytes), static_cast<int64_t>(pc.tile_begin), static_cast<int64_t>(pc.flags)});
  return out;
}

std::string BucketSet::rs_plan(int g) const {
  const auto& b = buckets_.at(g);
  static const char* names[] = {"oneshot", "pipe", "nvls"};
  Msg o;
  o << names[b.rs_algo] << ":grid=" << b.rs_grid << ":stripes=" << b.nstripes << ":stripe_bytes=" << b.stripe_bytes;
  return o.str();
}

void BucketSet::synchronize() {
  if (comm_->is_cuda()) {
    DEAR_CUDA(cudaStreamSynchronize(S(stream_)));
    if (ag_stream_ != stream_) DEAR_CUDA(cudaStreamSynchronize(S(ag_stream_)));
  }
  comm_->check_status();
}

}  // namespace dear
