// comm.cpp — replica communicator: binds one worker replica to one GPU, owns its symmetric heap
// (CUDA VMM, exported as POSIX fds), exchanges handles with the job's other replicas over a unix
// socket, optionally binds an NVSwitch multicast object, re-forms the group in place on elastic
// add/drop, and plans + launches the allreduce kernels of allreduce.cu.
//
// Reference side: this is what stands behind the env contract of
// TorchJobReconciler.SetClusterSpec (controllers/train/torchjob_controller.go:394-446):
// RANK / WORLD_SIZE keep their meaning, MASTER_ADDR:MASTER_PORT is replaced by a unix-socket path
// (single box, no DNS/Services).  The elastic path replaces restartStalePod /
// restartPodInKruiseProtocol (controllers/train/elastic_scale.go:303-397): survivors are not
// restarted, only the membership changes.
#include <cuda.h>
#include <cuda_runtime.h>
#include <errno.h>
#include <math.h>
#include <fcntl.h>
#include <poll.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/socket.h>
#include <sys/stat.h>
#include <sys/time.h>
#include <sys/types.h>
#include <sys/un.h>
#include <time.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <random>
#include <string>
#include <vector>

#include "tok_internal.h"

namespace tok {

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
}

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

const char* last_error_cstr() { return g_err.c_str(); }

// ------------------------------------------------------------------------------------------------
// driver API, resolved through the runtime so that libtok8s.so has no link-time dependency on
// libcuda.so (it must load — and its control plane must work — on a box without a driver).
// ------------------------------------------------------------------------------------------------
#define TOK_DRV_FNS(X)             \
  X(cuGetErrorString)              \
  X(cuDeviceGet)                   \
  X(cuDeviceGetAttribute)          \
  X(cuMemGetAllocationGranularity) \
  X(cuMemCreate)                   \
  X(cuMemRelease)                  \
  X(cuMemAddressReserve)           \
  X(cuMemAddressFree)              \
  X(cuMemMap)                      \
  X(cuMemUnmap)                    \
  X(cuMemSetAccess)                \
  X(cuMemExportToShareableHandle)  \
  X(cuMemImportFromShareableHandle) \
  X(cuMulticastCreate)             \
  X(cuMulticastAddDevice)          \
  X(cuMulticastBindMem)            \
  X(cuMulticastUnbind)             \
  X(cuMulticastGetGranularity)

struct Drv {
#define X(n) decltype(&n) n##_ = nullptr;
  TOK_DRV_FNS(X)
#undef X
  bool ok = false;
  std::string why;
};

static Drv& drv() {
  static Drv d;
  static std::once_flag once;
  std::call_once(once, [] {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
      d.why = std::string("no CUDA device: ") + cudaGetErrorString(e);
      cudaGetLastError();
      return;
    }
#define X(n)                                                                          \
  {                                                                                   \
    void* fp = nullptr;                                                               \
    cudaDriverEntryPointQueryResult qr;                                               \
    e = cudaGetDriverEntryPoint(#n, &fp, cudaEnableDefault, &qr);                     \
    if (e != cudaSuccess || fp == nullptr || qr != cudaDriverEntryPointSuccess) {     \
      d.why = std::string("driver entry point missing: ") + #n;                       \
      cudaGetLastError();                                                             \
      return;                                                                         \
    }                                                                                 \
    d.n##_ = reinterpret_cast<decltype(&n)>(fp);                                      \
  }
    TOK_DRV_FNS(X)
#undef X
    d.ok = true;
  });
  return d;
}

static const char* cu_err(CUresult r) {
  const char* s = nullptr;
  if (drv().cuGetErrorString_ && drv().cuGetErrorString_(r, &s) == CUDA_SUCCESS && s) return s;
  return "unknown CUresult";
}

#define CU_CHECK(call)                                                                 \
  do {                                                                                 \
    CUresult _r = (call);                                                              \
    if (_r != CUDA_SUCCESS)                                                            \
      return fail(TOK_ERR_CUDA, "%s failed: %s (%d)", #call, cu_err(_r), (int)_r);     \
  } while (0)
#define RT_CHECK(call)                                                                 \
  do {                                                                                 \
    cudaError_t _e = (call);                                                           \
    if (_e != cudaSuccess)                                                             \
      return fail(TOK_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e));       \
  } while (0)

static size_t env_size(const char* name, size_t dflt) {
  const char* v = getenv(name);
  if (!v || !*v) return dflt;
  char* end = nullptr;
  unsigned long long x = strtoull(v, &end, 10);
  if (end == v) return dflt;
  return static_cast<size_t>(x);
}

static size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static double now_s() {
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec + ts.tv_nsec * 1e-9;
}

// ------------------------------------------------------------------------------------------------
// unix-socket plumbing (star topology around the group's rank 0)
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kMagic = 0x746f6b38u;  // "tok8"

struct Hello {
  uint32_t magic;
  uint32_t abi;
  uint64_t epoch;
  int32_t rank;
  int32_t world;
  int32_t device;
  int32_t pid;
  uint64_t uid;
  uint64_t heap_bytes;
  uint64_t cap_bytes;
  int32_t mc_supported;
  int32_t reserved;
  char bus_id[32];
  char job[64];
};

static int wait_fd(int fd, short events, double deadline) {
  for (;;) {
    double left = deadline - now_s();
    if (left <= 0) return 0;
    struct pollfd p = {fd, events, 0};
    int r = poll(&p, 1, static_cast<int>(std::min(left, 1.0) * 1000) + 1);
    if (r > 0) return 1;
    if (r < 0 && errno != EINTR) return -1;
  }
}

// Sends buf (len bytes) with nfds descriptors attached to the first byte.
static int send_msg(int sock, const void* buf, size_t len, const int* fds, int nfds,
                    double deadline) {
  const char* p = static_cast<const char*>(buf);
  size_t sent = 0;
  bool first = true;
  while (sent < len) {
    if (wait_fd(sock, POLLOUT, deadline) <= 0) return -1;
    struct msghdr msg;
    memset(&msg, 0, sizeof(msg));
    struct iovec iov = {const_cast<char*>(p + sent), len - sent};
    msg.msg_iov = &iov;
    msg.msg_iovlen = 1;
    std::vector<char> ctrl;
    if (first && nfds > 0) {
      ctrl.resize(CMSG_SPACE(sizeof(int) * nfds));
      msg.msg_control = ctrl.data();
      msg.msg_controllen = ctrl.size();
      struct cmsghdr* c = CMSG_FIRSTHDR(&msg);
      c->cmsg_level = SOL_SOCKET;
      c->cmsg_type = SCM_RIGHTS;
      c->cmsg_len = CMSG_LEN(sizeof(int) * nfds);
      memcpy(CMSG_DATA(c), fds, sizeof(int) * nfds);
    }
    ssize_t n = sendmsg(sock, &msg, MSG_NOSIGNAL);
    if (n < 0) {
      if (errno == EINTR || errno == EAGAIN) continue;
      return -1;
    }
    sent += static_cast<size_t>(n);
    first = false;
  }
  return 0;
}

// Receives exactly len bytes; descriptors that arrive with them are appended to fds_out.
static int recv_msg(int sock, void* buf, size_t len, std::vector<int>* fds_out, double deadline) {
  char* p = static_cast<char*>(buf);
  size_t got = 0;
  while (got < len) {
    if (wait_fd(sock, POLLIN, deadline) <= 0) return -1;
    struct msghdr msg;
    memset(&msg, 0, sizeof(msg));
    struct iovec iov = {p + got, len - got};
    msg.msg_iov = &iov;
    msg.msg_iovlen = 1;
    char ctrl[CMSG_SPACE(sizeof(int) * 16)];
    msg.msg_control = ctrl;
    msg.msg_controllen = sizeof(ctrl);
    ssize_t n = recvmsg(sock, &msg, 0);
    if (n < 0) {
      if (errno == EINTR || errno == EAGAIN) continue;
      return -1;
    }
    if (n == 0) return -1;  // peer closed
    for (struct cmsghdr* c = CMSG_FIRSTHDR(&msg); c; c = CMSG_NXTHDR(&msg, c)) {
      if (c->cmsg_level == SOL_SOCKET && c->cmsg_type == SCM_RIGHTS) {
        int cnt = static_cast<int>((c->cmsg_len - CMSG_LEN(0)) / sizeof(int));
        for (int i = 0; i < cnt; ++i) {
          int fd;
          memcpy(&fd, CMSG_DATA(c) + i * sizeof(int), sizeof(int));
          if (fds_out)
            fds_out->push_back(fd);
          else
            close(fd);
        }
      }
    }
    got += static_cast<size_t>(n);
  }
  return 0;
}

struct Star {
  bool root = false;
  int world = 0;
  int listen_fd = -1;
  std::vector<int> conn;  // root: conn[rank] for rank != 0 ; member: conn[0] = link to root
  std::string path;
  double deadline = 0;

  ~Star() { close_all(); }
  void close_all() {
    for (int& c : conn)
      if (c >= 0) {
        close(c);
        c = -1;
      }
    if (listen_fd >= 0) {
      close(listen_fd);
      listen_fd = -1;
      unlink(path.c_str());
    }
  }
  // Collective AND of a per-member status, returned to everyone.
  int all_ok(int my_ok, int* out) {
    if (root) {
      int acc = my_ok ? 1 : 0;
      for (int r = 1; r < world; ++r) {
        int v = 0;
        if (recv_msg(conn[r], &v, sizeof(v), nullptr, deadline) != 0)
          return fail(TOK_ERR_RENDEZVOUS, "rendezvous: lost rank %d during barrier", r);
        acc &= (v ? 1 : 0);
      }
      for (int r = 1; r < world; ++r)
        if (send_msg(conn[r], &acc, sizeof(acc), nullptr, 0, deadline) != 0)
          return fail(TOK_ERR_RENDEZVOUS, "rendezvous: cannot release rank %d", r);
      *out = acc;
    } else {
      int v = my_ok ? 1 : 0;
      if (send_msg(conn[0], &v, sizeof(v), nullptr, 0, deadline) != 0 ||
          recv_msg(conn[0], &v, sizeof(v), nullptr, deadline) != 0)
        return fail(TOK_ERR_RENDEZVOUS, "rendezvous: lost the group root during barrier");
      *out = v;
    }
    return TOK_OK;
  }
};

}  // namespace tok

// ------------------------------------------------------------------------------------------------
// the communicator
// ------------------------------------------------------------------------------------------------
using namespace tok;

struct PeerMap {
  uint64_t uid = 0;
  CUmemGenericAllocationHandle handle = 0;
  CUdeviceptr va = 0;
  bool own = false;
};

struct tok_comm {
  std::string job_id;
  std::string rdzv_path;
  int rank = 0, world = 1, max_world = 1, device = 0;
  uint64_t uid = 0;
  uint64_t epoch = 0;
  CUdevice cu_dev = 0;
  char bus_id[32] = {0};
  int sm_count = 148;
  int mc_supported = 0;

  size_t gran = 0;
  size_t cap_bytes = 0;
  size_t pool_bytes = 0;   // symmetric pool for zero-copy buckets
  size_t pool_used = 0;    // bump pointer (identical allocation sequence on every replica)
  std::vector<std::pair<size_t, size_t>> pool_free;  // (offset, bytes) of released segments, by offset
  std::mutex pool_mu;      // tok_pool_malloc may be entered from any allocator-calling thread
  size_t heap_bytes = 0;
  bool zero_copy = true;
  CUmemGenericAllocationHandle local_handle = 0;
  CUdeviceptr local_va = 0;

  std::vector<PeerMap> cache;      // every heap currently mapped (including our own)
  char* peer[kMaxWorld] = {0};     // by current rank

  bool mc_bound = false;
  CUmemGenericAllocationHandle mc_handle = 0;
  CUdeviceptr mc_va = 0;

  unsigned long long* dbg = nullptr;    // device, only with TOK_DEBUG_PHASES=1
  uint32_t* ctr = nullptr;              // device
  volatile uint32_t* hostctl = nullptr; // pinned host page
  uint32_t* hostctl_dev = nullptr;

  // tunables
  int max_ctas = 64;
  int zc_ctas = 0;          // 0 = built-in rule for the zero-copy kernels
  size_t cta_bytes = 65536;
  size_t one_shot_max = 256 << 10;
  bool one_shot_max_env = false;
  size_t nvls_min = 0;
  int force_algo = 0;
  bool disable_nvls = false;
  unsigned long long barrier_timeout_ns = 600000ull * 1000000ull;
  double rdzv_timeout_s = 120;
  int local_tma = 1;        // world 1, one dtype: 1 = cp.async.bulk variant, 0 = LDG.128 wave
  int nvls_unroll = 8;      // multimem.ld_reduce in flight per thread in the zero-copy NVLS kernel

  std::atomic<uint64_t> launches{0};    // exchange / broadcast / local kernels
  std::atomic<uint64_t> arrivals{0};    // arrive kernels
  std::atomic<uint64_t> elided{0};      // world-1 identity buckets that needed no launch
  std::atomic<uint64_t> broadcasts{0};
  std::atomic<int> last_algo{0};
  std::atomic<int> last_ctas{0};
  bool membership_dirty = false;  // exchange() got far enough to touch the peer mappings
};

static std::atomic<tok_comm*> g_pool_comm{nullptr};  // communicator behind tok_pool_malloc()

namespace {

struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) {
      cudaSetDevice(dev);
      changed = true;
    }
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
};

int map_heap(tok_comm* c, CUmemGenericAllocationHandle h, CUdeviceptr* va) {
  Drv& d = drv();
  CU_CHECK(d.cuMemAddressReserve_(va, c->heap_bytes, c->gran, 0, 0));
  CUresult r = d.cuMemMap_(*va, c->heap_bytes, 0, h, 0);
  if (r != CUDA_SUCCESS) {
    d.cuMemAddressFree_(*va, c->heap_bytes);
    return fail(TOK_ERR_CUDA, "cuMemMap failed: %s", cu_err(r));
  }
  CUmemAccessDesc acc;
  memset(&acc, 0, sizeof(acc));
  acc.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  acc.location.id = c->cu_dev;
  acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  r = d.cuMemSetAccess_(*va, c->heap_bytes, &acc, 1);
  if (r != CUDA_SUCCESS) {
    d.cuMemUnmap_(*va, c->heap_bytes);
    d.cuMemAddressFree_(*va, c->heap_bytes);
    return fail(TOK_ERR_CUDA,
                "cuMemSetAccess on a peer heap failed: %s (no P2P path between the replicas' GPUs?)",
                cu_err(r));
  }
  return TOK_OK;
}

void unmap_heap(tok_comm* c, PeerMap& m) {
  Drv& d = drv();
  if (m.va) {
    d.cuMemUnmap_(m.va, c->heap_bytes);
    d.cuMemAddressFree_(m.va, c->heap_bytes);
  }
  if (m.handle && !m.own) d.cuMemRelease_(m.handle);
  m = PeerMap();
}

void teardown_multicast(tok_comm* c) {
  Drv& d = drv();
  if (c->mc_va) {
    d.cuMemUnmap_(c->mc_va, c->heap_bytes);
    d.cuMemAddressFree_(c->mc_va, c->heap_bytes);
    c->mc_va = 0;
  }
  if (c->mc_handle) {
    if (c->mc_bound) d.cuMulticastUnbind_(c->mc_handle, c->cu_dev, 0, c->heap_bytes);
    d.cuMemRelease_(c->mc_handle);
    c->mc_handle = 0;
  }
  c->mc_bound = false;
}

int alloc_local(tok_comm* c) {
  Drv& d = drv();
  CUmemAllocationProp prop;
  memset(&prop, 0, sizeof(prop));
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = c->cu_dev;
  prop.requestedHandleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
  size_t gran = 0;
  CU_CHECK(d.cuMemGetAllocationGranularity_(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
  c->gran = std::max<size_t>(gran, 2u << 20);

  int mc = 0;
  d.cuDeviceGetAttribute_(&mc, CU_DEVICE_ATTRIBUTE_MULTICAST_SUPPORTED, c->cu_dev);
  c->mc_supported = (mc && !c->disable_nvls) ? 1 : 0;
  size_t total = kFlagBytes + 2 * c->cap_bytes + c->pool_bytes;
  if (c->mc_supported && c->max_world > 1) {
    CUmulticastObjectProp mp;
    memset(&mp, 0, sizeof(mp));
    mp.numDevices = static_cast<unsigned>(c->max_world);
    mp.size = round_up(total, c->gran);
    mp.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
    size_t mg = 0;
    if (d.cuMulticastGetGranularity_(&mg, &mp, CU_MULTICAST_GRANULARITY_RECOMMENDED) ==
            CUDA_SUCCESS &&
        mg > 0 && mg <= (1ull << 30))
      c->gran = std::max(c->gran, mg);
    else if (d.cuMulticastGetGranularity_(&mg, &mp, CU_MULTICAST_GRANULARITY_MINIMUM) ==
                 CUDA_SUCCESS &&
             mg > 0)
      c->gran = std::max(c->gran, mg);
  }
  c->heap_bytes = round_up(total, c->gran);
  c->pool_bytes = c->heap_bytes - kFlagBytes - 2 * c->cap_bytes;  // rounding slack joins the pool
  CU_CHECK(d.cuMemCreate_(&c->local_handle, c->heap_bytes, &prop, 0));
  int rc = map_heap(c, c->local_handle, &c->local_va);
  if (rc != TOK_OK) return rc;
  RT_CHECK(cudaMemset(reinterpret_cast<void*>(c->local_va), 0, kFlagBytes));
  RT_CHECK(cudaMalloc(reinterpret_cast<void**>(&c->ctr), kCtrWords * sizeof(uint32_t)));
  RT_CHECK(cudaMemset(c->ctr, 0, kCtrWords * sizeof(uint32_t)));
  if (env_size("TOK_DEBUG_PHASES", 0)) {
    RT_CHECK(cudaMalloc(reinterpret_cast<void**>(&c->dbg), kMaxCtas * 8 * sizeof(unsigned long long)));
    RT_CHECK(cudaMemset(c->dbg, 0, kMaxCtas * 8 * sizeof(unsigned long long)));
  }
  void* hp = nullptr;
  RT_CHECK(cudaHostAlloc(&hp, 4096, cudaHostAllocMapped | cudaHostAllocPortable));
  memset(hp, 0, 4096);
  c->hostctl = static_cast<volatile uint32_t*>(hp);
  void* dp = nullptr;
  RT_CHECK(cudaHostGetDevicePointer(&dp, hp, 0));
  c->hostctl_dev = static_cast<uint32_t*>(dp);
  PeerMap self;
  self.uid = c->uid;
  self.handle = c->local_handle;
  self.va = c->local_va;
  self.own = true;
  c->cache.push_back(self);
  return TOK_OK;
}

// One membership exchange: gathers every member's Hello + heap fd at the group's rank 0 and
// scatters the full table back, then (re)builds the peer table and the multicast binding.
int exchange(tok_comm* c) {
  Drv& d = drv();
  c->membership_dirty = false;
  Star star;
  star.root = (c->rank == 0);
  star.world = c->world;
  star.deadline = now_s() + c->rdzv_timeout_s;
  char suffix[32];
  snprintf(suffix, sizeof(suffix), ".e%llu", static_cast<unsigned long long>(c->epoch));
  star.path = c->rdzv_path + suffix;
  struct sockaddr_un addr;
  memset(&addr, 0, sizeof(addr));
  addr.sun_family = AF_UNIX;
  // sun_path holds 107 characters.  A longer path names the same socket file through this
  // process's descriptor of its directory, /proc/self/fd/<dir>/<name>, which every replica opens
  // for itself; the directory descriptor only has to live until bind() / connect().
  std::string sock = star.path;
  struct DirFd {
    int fd = -1;
    ~DirFd() {
      if (fd >= 0) close(fd);
    }
  } dir;
  if (sock.size() >= sizeof(addr.sun_path)) {
    const size_t slash = star.path.rfind('/');
    const std::string parent =
        slash == std::string::npos ? "." : (slash == 0 ? "/" : star.path.substr(0, slash));
    dir.fd = open(parent.c_str(), O_PATH | O_DIRECTORY | O_CLOEXEC);
    if (dir.fd < 0)
      return fail(TOK_ERR_RENDEZVOUS, "rendezvous directory %s: %s", parent.c_str(),
                  strerror(errno));
    sock = "/proc/self/fd/" + std::to_string(dir.fd) + "/" +
           star.path.substr(slash == std::string::npos ? 0 : slash + 1);
  }
  if (sock.size() >= sizeof(addr.sun_path))
    return fail(TOK_ERR_INVALID, "rendezvous file name too long (%zu >= %zu): %s", sock.size(),
                sizeof(addr.sun_path), star.path.c_str());
  strcpy(addr.sun_path, sock.c_str());

  Hello me;
  memset(&me, 0, sizeof(me));
  me.magic = kMagic;
  me.abi = TOK_ABI_VERSION;
  me.epoch = c->epoch;
  me.rank = c->rank;
  me.world = c->world;
  me.device = c->device;
  me.pid = static_cast<int32_t>(getpid());
  me.uid = c->uid;
  me.heap_bytes = c->heap_bytes;
  me.cap_bytes = c->cap_bytes;
  me.mc_supported = c->mc_supported;
  memcpy(me.bus_id, c->bus_id, sizeof(me.bus_id));
  snprintf(me.job, sizeof(me.job), "%s", c->job_id.c_str());

  std::vector<Hello> table(c->world);
  std::vector<int> fds(c->world, -1);
  auto close_fds = [&] {
    for (int& f : fds)
      if (f >= 0) {
        close(f);
        f = -1;
      }
  };

  int my_fd = -1;
  if (c->world > 1)
    CU_CHECK(d.cuMemExportToShareableHandle_(&my_fd, c->local_handle,
                                             CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0));

  if (c->world == 1) {
    table[0] = me;
  } else if (star.root) {
    star.listen_fd = socket(AF_UNIX, SOCK_STREAM | SOCK_CLOEXEC, 0);
    if (star.listen_fd < 0) {
      close(my_fd);
      return fail(TOK_ERR_RENDEZVOUS, "socket(): %s", strerror(errno));
    }
    unlink(star.path.c_str());
    if (bind(star.listen_fd, reinterpret_cast<struct sockaddr*>(&addr), sizeof(addr)) != 0 ||
        listen(star.listen_fd, kMaxWorld) != 0) {
      close(my_fd);
      return fail(TOK_ERR_RENDEZVOUS, "bind/listen(%s): %s", star.path.c_str(), strerror(errno));
    }
    star.conn.assign(c->world, -1);
    table[0] = me;
    fds[0] = my_fd;
    for (int joined = 1; joined < c->world; ++joined) {
      if (wait_fd(star.listen_fd, POLLIN, star.deadline) <= 0) {
        close_fds();
        return fail(TOK_ERR_RENDEZVOUS,
                    "rendezvous %s: only %d of %d replicas joined within %.0f s", star.path.c_str(),
                    joined, c->world, c->rdzv_timeout_s);
      }
      int s = accept4(star.listen_fd, nullptr, nullptr, SOCK_CLOEXEC);
      if (s < 0) {
        --joined;
        continue;
      }
      Hello h;
      std::vector<int> got;
      if (recv_msg(s, &h, sizeof(h), &got, star.deadline) != 0 || h.magic != kMagic ||
          got.size() != 1) {
        for (int f : got) close(f);
        close(s);
        close_fds();
        return fail(TOK_ERR_RENDEZVOUS, "rendezvous %s: malformed hello", star.path.c_str());
      }
      const bool bad = h.abi != TOK_ABI_VERSION || h.epoch != c->epoch || h.world != c->world ||
                       h.rank <= 0 || h.rank >= c->world || star.conn[h.rank] >= 0 ||
                       h.heap_bytes != c->heap_bytes || h.cap_bytes != c->cap_bytes ||
                       strncmp(h.job, me.job, sizeof(h.job)) != 0;
      if (bad) {
        close(got[0]);
        close(s);
        close_fds();
        return fail(TOK_ERR_RENDEZVOUS,
                    "rendezvous %s: replica rank=%d world=%d epoch=%llu heap=%llu job=%.63s does not "
                    "match this group (world=%d epoch=%llu heap=%llu job=%s)",
                    star.path.c_str(), h.rank, h.world, (unsigned long long)h.epoch,
                    (unsigned long long)h.heap_bytes, h.job, c->world,
                    (unsigned long long)c->epoch, (unsigned long long)c->heap_bytes, me.job);
      }
      star.conn[h.rank] = s;
      table[h.rank] = h;
      fds[h.rank] = got[0];
    }
    for (int r = 1; r < c->world; ++r) {
      if (send_msg(star.conn[r], table.data(), sizeof(Hello) * c->world, fds.data(), c->world,
                   star.deadline) != 0) {
        close_fds();
        return fail(TOK_ERR_RENDEZVOUS, "rendezvous: cannot send the table to rank %d", r);
      }
    }
  } else {
    int s = -1;
    for (;;) {
      s = socket(AF_UNIX, SOCK_STREAM | SOCK_CLOEXEC, 0);
      if (s < 0) {
        close(my_fd);
        return fail(TOK_ERR_RENDEZVOUS, "socket(): %s", strerror(errno));
      }
      if (connect(s, reinterpret_cast<struct sockaddr*>(&addr), sizeof(addr)) == 0) break;
      close(s);
      if (now_s() > star.deadline) {
        close(my_fd);
        return fail(TOK_ERR_RENDEZVOUS, "rendezvous %s: the group root never appeared (%.0f s)",
                    star.path.c_str(), c->rdzv_timeout_s);
      }
      usleep(20000);
    }
    star.conn.assign(1, s);
    int rc = send_msg(s, &me, sizeof(me), &my_fd, 1, star.deadline);
    close(my_fd);
    my_fd = -1;
    if (rc != 0) return fail(TOK_ERR_RENDEZVOUS, "rendezvous: cannot send hello");
    std::vector<int> got;
    if (recv_msg(s, table.data(), sizeof(Hello) * c->world, &got, star.deadline) != 0 ||
        static_cast<int>(got.size()) != c->world) {
      for (int f : got) close(f);
      return fail(TOK_ERR_RENDEZVOUS,
                  "rendezvous %s: no membership table from the root (it rejected this replica or "
                  "timed out)",
                  star.path.c_str());
    }
    for (int r = 0; r < c->world; ++r) fds[r] = got[r];
  }

  // ---- build the peer table, reusing mappings of surviving peers (in-place re-form) -------------
  c->membership_dirty = true;
  std::vector<PeerMap> next;
  int rc = TOK_OK;
  for (int r = 0; r < c->world && rc == TOK_OK; ++r) {
    auto it = std::find_if(c->cache.begin(), c->cache.end(),
                           [&](const PeerMap& m) { return m.uid == table[r].uid && m.va != 0; });
    if (it != c->cache.end()) {
      next.push_back(*it);
      it->va = 0;  // moved
      it->handle = 0;
    } else {
      PeerMap m;
      m.uid = table[r].uid;
      CUresult cr = d.cuMemImportFromShareableHandle_(
          &m.handle, reinterpret_cast<void*>(static_cast<uintptr_t>(fds[r])),
          CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR);
      if (cr != CUDA_SUCCESS) {
        rc = fail(TOK_ERR_CUDA, "cuMemImportFromShareableHandle(rank %d) failed: %s", r, cu_err(cr));
        break;
      }
      rc = map_heap(c, m.handle, &m.va);
      if (rc != TOK_OK) {
        d.cuMemRelease_(m.handle);
        break;
      }
      next.push_back(m);
    }
  }
  close_fds();
  // whatever is left in the old cache belongs to replicas that were dropped (never our own heap:
  // our uid is always in the table)
  for (PeerMap& m : c->cache)
    if (m.va != 0 && !m.own) unmap_heap(c, m);
  for (PeerMap& m : c->cache)
    if (m.va != 0 && m.own) next.push_back(m);  // only reachable after a failed exchange
  c->cache.swap(next);
  int all = 0;
  int brc = c->world > 1 ? star.all_ok(rc == TOK_OK, &all) : (all = (rc == TOK_OK), TOK_OK);
  if (rc != TOK_OK) return rc;
  if (brc != TOK_OK) return brc;
  if (!all) return fail(TOK_ERR_RENDEZVOUS, "a peer failed to map the group's heaps");
  for (int r = 0; r < kMaxWorld; ++r) c->peer[r] = reinterpret_cast<char*>(c->local_va);
  for (int r = 0; r < c->world; ++r) {
    auto it = std::find_if(c->cache.begin(), c->cache.end(),
                           [&](const PeerMap& m) { return m.uid == table[r].uid; });
    c->peer[r] = reinterpret_cast<char*>(it->va);
  }

  // ---- NVSwitch multicast (NVLS) -----------------------------------------------------------------
  teardown_multicast(c);
  bool mc_possible = c->world > 1;
  for (int r = 0; r < c->world; ++r) {
    if (!table[r].mc_supported) mc_possible = false;
    for (int q = 0; q < r; ++q)
      if (strncmp(table[r].bus_id, table[q].bus_id, sizeof(table[r].bus_id)) == 0)
        mc_possible = false;  // two replicas share a GPU (single-GPU test mode)
  }
  if (mc_possible) {
    int ok = 1;
    int mc_fd = -1;
    if (star.root) {
      CUmulticastObjectProp mp;
      memset(&mp, 0, sizeof(mp));
      mp.numDevices = static_cast<unsigned>(c->world);
      mp.size = c->heap_bytes;
      mp.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
      CUresult cr = d.cuMulticastCreate_(&c->mc_handle, &mp);
      if (cr == CUDA_SUCCESS)
        cr = d.cuMemExportToShareableHandle_(&mc_fd, c->mc_handle,
                                             CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0);
      if (cr != CUDA_SUCCESS) {
        set_error("multicast create/export failed: %s", cu_err(cr));
        ok = 0;
      }
      for (int r = 1; r < c->world; ++r) {
        int32_t hdr = ok;
        if (send_msg(star.conn[r], &hdr, sizeof(hdr), ok ? &mc_fd : nullptr, ok ? 1 : 0,
                     star.deadline) != 0)
          return fail(TOK_ERR_RENDEZVOUS, "rendezvous: cannot send the multicast handle");
      }
      if (mc_fd >= 0) close(mc_fd);
    } else {
      int32_t hdr = 0;
      std::vector<int> got;
      if (recv_msg(star.conn[0], &hdr, sizeof(hdr), &got, star.deadline) != 0)
        return fail(TOK_ERR_RENDEZVOUS, "rendezvous: no multicast handle from the root");
      ok = hdr;
      if (ok && got.size() == 1) {
        CUresult cr = d.cuMemImportFromShareableHandle_(
            &c->mc_handle, reinterpret_cast<void*>(static_cast<uintptr_t>(got[0])),
            CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR);
        if (cr != CUDA_SUCCESS) {
          set_error("multicast import failed: %s", cu_err(cr));
          c->mc_handle = 0;
          ok = 0;
        }
      } else {
        ok = 0;
      }
      for (int f : got) close(f);
    }
    if (ok && d.cuMulticastAddDevice_(c->mc_handle, c->cu_dev) != CUDA_SUCCESS) ok = 0;
    int all_added = 0;
    rc = star.all_ok(ok, &all_added);
    if (rc != TOK_OK) return rc;
    int bound = 0;
    if (all_added) {
      CUresult cr = d.cuMulticastBindMem_(c->mc_handle, 0, c->local_handle, 0, c->heap_bytes, 0);
      if (cr == CUDA_SUCCESS) {
        c->mc_bound = true;
        bound = 1;
      } else {
        set_error("cuMulticastBindMem failed: %s", cu_err(cr));
      }
    }
    int all_bound = 0;
    rc = star.all_ok(bound, &all_bound);
    if (rc != TOK_OK) return rc;
    int mapped = 0;
    if (all_bound) {
      CUdeviceptr va = 0;
      if (d.cuMemAddressReserve_(&va, c->heap_bytes, c->gran, 0, 0) == CUDA_SUCCESS) {
        CUmemAccessDesc acc;
        memset(&acc, 0, sizeof(acc));
        acc.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
        acc.location.id = c->cu_dev;
        acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        if (d.cuMemMap_(va, c->heap_bytes, 0, c->mc_handle, 0) == CUDA_SUCCESS) {
          if (d.cuMemSetAccess_(va, c->heap_bytes, &acc, 1) == CUDA_SUCCESS) {
            c->mc_va = va;
            mapped = 1;
          } else {
            d.cuMemUnmap_(va, c->heap_bytes);
            d.cuMemAddressFree_(va, c->heap_bytes);
          }
        } else {
          d.cuMemAddressFree_(va, c->heap_bytes);
        }
      }
    }
    int all_mapped = 0;
    rc = star.all_ok(mapped, &all_mapped);
    if (rc != TOK_OK) return rc;
    if (!all_mapped) teardown_multicast(c);  // NVLS is optional: fall back to P2P algorithms
  }

  // ---- fresh barrier state for the new group ------------------------------------------------------
  RT_CHECK(cudaMemset(reinterpret_cast<void*>(c->local_va), 0, kFlagBytes));
  RT_CHECK(cudaMemset(c->ctr, 0, kCtrWords * sizeof(uint32_t)));
  RT_CHECK(cudaDeviceSynchronize());
  c->hostctl[kCtlAbort] = 0;
  c->hostctl[kCtlStatus] = 0;
  c->hostctl[kCtlWhere] = 0;
  // identity token at the end of the control page: after the host barrier every replica reads every
  // peer's token THROUGH ITS PEER MAPPING and compares it with the uid the membership table lists for
  // that rank — a wrong or stale mapping fails here, loudly, instead of as a silent hang later
  RT_CHECK(cudaMemcpy(reinterpret_cast<char*>(c->local_va) + kTokenOff, &c->uid, sizeof(c->uid),
                      cudaMemcpyHostToDevice));
  RT_CHECK(cudaDeviceSynchronize());
  if (c->world > 1) {
    int all_reset = 0;
    rc = star.all_ok(1, &all_reset);
    if (rc != TOK_OK) return rc;
    int good = 1;
    for (int r = 0; r < c->world; ++r) {
      uint64_t seen = 0;
      if (cudaMemcpy(&seen, c->peer[r] + kTokenOff, sizeof(seen), cudaMemcpyDeviceToHost) != cudaSuccess ||
          seen != table[r].uid) {
        set_error("peer mapping check failed: rank %d's heap as mapped by rank %d carries token %llx, "
                  "the membership table says %llx",
                  r, c->rank, (unsigned long long)seen, (unsigned long long)table[r].uid);
        cudaGetLastError();
        good = 0;
      }
    }
    int all_good = 0;
    rc = star.all_ok(good, &all_good);
    if (rc != TOK_OK) return rc;
    if (!good) return TOK_ERR_STATE;
    if (!all_good) return fail(TOK_ERR_STATE, "a peer's mapping check failed");
  }
  return TOK_OK;
}

int create_impl(const char* job_id, int rank, int world, int max_world, int device_ordinal,
                const char* rendezvous_path, uint64_t epoch, tok_comm_t** out) {
  if (!out) return fail(TOK_ERR_INVALID, "comm out pointer is null");
  *out = nullptr;
  if (!job_id || !rendezvous_path) return fail(TOK_ERR_INVALID, "job_id / rendezvous_path is null");
  if (world < 1 || world > kMaxWorld || rank < 0 || rank >= world)
    return fail(TOK_ERR_INVALID, "invalid rank %d / world %d (1..%d)", rank, world, kMaxWorld);
  if (max_world < world) max_world = world;
  if (max_world > kMaxWorld)
    return fail(TOK_ERR_INVALID, "max_world %d exceeds %d", max_world, kMaxWorld);
  Drv& d = drv();
  if (!d.ok)
    return fail(TOK_ERR_NO_DEVICE, "libtok8s data path needs a CUDA GPU (no CPU fallback): %s",
                d.why.c_str());
  int ndev = 0;
  RT_CHECK(cudaGetDeviceCount(&ndev));
  if (device_ordinal < 0 || device_ordinal >= ndev)
    return fail(TOK_ERR_INVALID, "device ordinal %d out of range (0..%d)", device_ordinal, ndev - 1);

  DeviceGuard guard(device_ordinal);
  RT_CHECK(cudaFree(nullptr));  // make sure the primary context exists
  tok_comm* c = new tok_comm();
  c->job_id = job_id;
  c->rdzv_path = rendezvous_path;
  c->rank = rank;
  c->world = world;
  c->max_world = max_world;
  c->device = device_ordinal;
  c->epoch = epoch;
  std::random_device rd;
  c->uid = (static_cast<uint64_t>(rd()) << 32) ^ rd() ^ (static_cast<uint64_t>(getpid()) << 20) ^
           static_cast<uint64_t>(now_s() * 1e6);
  if (c->uid == 0) c->uid = 1;
  c->cap_bytes = round_up(env_size("TOK_STAGING_MB", 128) << 20, 2u << 20);
  c->pool_bytes = round_up(env_size("TOK_SYMM_POOL_MB", 1024) << 20, 2u << 20);
  c->zero_copy = env_size("TOK_DISABLE_ZERO_COPY", 0) == 0;
  c->max_ctas = static_cast<int>(std::min<size_t>(env_size("TOK_MAX_CTAS", 64), kMaxCtas));
  if (c->max_ctas < 1) c->max_ctas = 1;
  c->zc_ctas = static_cast<int>(std::min<size_t>(env_size("TOK_ZC_CTAS", getenv("TOK_MAX_CTAS") ? c->max_ctas : 0), kMaxCtas));
  c->cta_bytes = std::max<size_t>(env_size("TOK_CTA_BYTES", 65536), 4096);
  c->one_shot_max_env = getenv("TOK_ONE_SHOT_MAX") != nullptr;
  c->one_shot_max = env_size("TOK_ONE_SHOT_MAX", 256 << 10);
  c->nvls_min = env_size("TOK_NVLS_MIN", 0);
  c->force_algo = static_cast<int>(env_size("TOK_ALGO", 0));
  c->disable_nvls = env_size("TOK_DISABLE_NVLS", 0) != 0;
  // NCCL's watchdog default is 600 s; replicas legitimately skew by tens of seconds (first-iteration
  // cuDNN autotune, evaluation or a checkpoint on rank 0)
  c->barrier_timeout_ns = env_size("TOK_BARRIER_TIMEOUT_MS", 600000) * 1000000ull;
  // measured (profiles/r02_local_bench_n1.json): the cp.async.bulk ring beats the LDG.128 wave at
  // every size from 4 MB to 1 GiB (12.4 vs 14.5 us at the 28 MB DDP bucket, 0.97 vs 0.71-0.90 of the
  // measured HBM peak at 1 GiB)
  c->local_tma = static_cast<int>(env_size("TOK_LOCAL_TMA", 1));
  c->nvls_unroll = env_size("TOK_NVLS_UNROLL", 8) == 16 ? 16 : 8;
  c->rdzv_timeout_s = static_cast<double>(env_size("TOK_RDZV_TIMEOUT_S", 120));

  int rc = TOK_OK;
  do {
    CUresult cr = d.cuDeviceGet_(&c->cu_dev, device_ordinal);
    if (cr != CUDA_SUCCESS) {
      rc = fail(TOK_ERR_CUDA, "cuDeviceGet failed: %s", cu_err(cr));
      break;
    }
    cudaDeviceGetPCIBusId(c->bus_id, sizeof(c->bus_id), device_ordinal);
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device_ordinal);
    rc = alloc_local(c);
    if (rc != TOK_OK) break;
    rc = exchange(c);
  } while (0);
  if (rc != TOK_OK) {
    std::string keep = last_error_cstr();
    tok_comm_destroy(c);
    set_error("%s", keep.c_str());
    return rc;
  }
  *out = c;
  return TOK_OK;
}

// Algorithm selector.  Thresholds come from the measured sweeps on 2/4/8 B200 (profiles/): one-shot
// moves (N-1)*S per GPU but needs a single barrier, so it wins while the bucket is latency-bound —
// the smaller the group, the longer; NVLS wins as soon as there are >= 3 replicas and the bucket is
// past the one-shot range; at N == 2 the in-switch reduction saves nothing and two-shot is faster.
size_t one_shot_limit(const tok_comm* c) {
  if (c->one_shot_max_env) return c->one_shot_max;
  const bool mc = c->mc_va != 0;
  switch (c->world) {
    case 2: return 16u << 20;
    case 3:
    case 4: return mc ? (2u << 20) : (8u << 20);
    case 5:
    case 6: return mc ? (64u << 10) : (2u << 20);
    default: return mc ? (32u << 10) : (1u << 20);
  }
}

int pick_algo(const tok_comm* c, size_t wire_bytes) {
  if (c->world == 1) return TOK_ALGO_LOCAL;
  if (c->force_algo >= TOK_ALGO_ONE_SHOT && c->force_algo <= TOK_ALGO_NVLS) {
    if (c->force_algo == TOK_ALGO_NVLS && !c->mc_va) return TOK_ALGO_TWO_SHOT;
    return c->force_algo;
  }
  const size_t slot = c->cap_bytes / kMaxWorld;
  if (wire_bytes <= one_shot_limit(c) && wire_bytes <= slot) return TOK_ALGO_ONE_SHOT;
  // staged path: with 3-4 replicas the in-switch reduction stops paying off past ~12 MiB (measured:
  // two-shot 385 vs NVLS 335 GB/s busbw at 16 MiB, N=4); zero-copy buckets re-promote to NVLS
  const bool nvls_ok = c->mc_va && c->world >= 3 && wire_bytes >= c->nvls_min;
  if (nvls_ok && (c->world >= 5 || wire_bytes < (12u << 20))) return TOK_ALGO_NVLS;
  return TOK_ALGO_TWO_SHOT;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* tok_last_error(void) { return tok::last_error_cstr(); }

const char* tok_version(void) { return "libtok8s 0.2 (sm_100a, abi 2)"; }

void tok_free(void* p) { free(p); }

int tok_comm_create(const char* job_id, int rank, int world, int max_world, int device_ordinal,
                    const char* rendezvous_path, tok_comm_t** comm) {
  return create_impl(job_id, rank, world, max_world, device_ordinal, rendezvous_path, 0, comm);
}

int tok_comm_join(const char* job_id, int rank, int world, int max_world, int device_ordinal,
                  const char* rendezvous_path, uint64_t epoch, tok_comm_t** comm) {
  return create_impl(job_id, rank, world, max_world, device_ordinal, rendezvous_path, epoch, comm);
}

int tok_comm_reform(tok_comm_t* c, int new_world, int new_rank, uint64_t member_mask,
                    uint64_t epoch) {
  if (!c) return fail(TOK_ERR_INVALID, "comm is null");
  if (new_world < 1 || new_world > c->max_world || new_rank < 0 || new_rank >= new_world)
    return fail(TOK_ERR_INVALID, "invalid new rank %d / world %d (max_world %d)", new_rank,
                new_world, c->max_world);
  if (epoch <= c->epoch)
    return fail(TOK_ERR_STATE, "epoch must grow: have %llu, got %llu",
                (unsigned long long)c->epoch, (unsigned long long)epoch);
  if (!(member_mask & (1ull << c->rank)))
    return fail(TOK_ERR_INVALID,
                "member_mask 0x%llx drops this replica (old rank %d): destroy it instead",
                (unsigned long long)member_mask, c->rank);
  DeviceGuard guard(c->device);
  RT_CHECK(cudaDeviceSynchronize());  // no collective of the old group may still be in flight
  const int old_rank = c->rank, old_world = c->world;
  const uint64_t old_epoch = c->epoch;
  c->rank = new_rank;
  c->world = new_world;
  c->epoch = epoch;
  const int rc = exchange(c);
  if (rc == TOK_ERR_RENDEZVOUS && !c->membership_dirty) {
    // The membership exchange never completed (peers that were announced did not show up): nothing
    // of the old group was unmapped yet, so the communicator stays usable with its previous
    // membership and a later epoch (e.g. the controller's revert) can still be applied.
    c->rank = old_rank;
    c->world = old_world;
    c->epoch = old_epoch;
  }
  return rc;
}

int tok_comm_abort(tok_comm_t* c) {
  if (!c || !c->hostctl) return fail(TOK_ERR_INVALID, "comm is null");
  c->hostctl[kCtlAbort] = 1;
  return TOK_OK;
}

int tok_comm_status(tok_comm_t* c) {
  if (!c || !c->hostctl) return fail(TOK_ERR_INVALID, "comm is null");
  const uint32_t s = c->hostctl[kCtlStatus];
  if (s == 1) {
    const uint32_t where = c->hostctl[kCtlWhere];
    return fail(TOK_ERR_TIMEOUT,
                "a peer replica never reached the in-kernel barrier within %llu ms (rank %d of %d; "
                "given up in %s, CTA %u, ranks still behind: mask 0x%x, waited for value %u)",
                c->barrier_timeout_ns / 1000000ull, c->rank, c->world,
                (where & 0xff) == 1 ? "the bucket arrival" : (where & 0xff) == 2 ? "a CTA barrier" : "?",
                where >> 8, c->hostctl[kCtlBehind], c->hostctl[kCtlWant]);
  }
  if (s == 2) return fail(TOK_ERR_ABORTED, "collective aborted by tok_comm_abort()");
  if (s == 3)
    return fail(TOK_ERR_STATE,
                "zero-copy bucket is not at the same symmetric-pool offset on every replica (the "
                "replicas' pool allocation sequences differ); set TOK_DISABLE_ZERO_COPY=1");
  return TOK_OK;
}

int tok_comm_destroy(tok_comm_t* c) {
  if (!c) return TOK_OK;
  {
    tok_comm* expect = c;
    g_pool_comm.compare_exchange_strong(expect, nullptr);
  }
  if (drv().ok) {
    DeviceGuard guard(c->device);
    cudaDeviceSynchronize();
    teardown_multicast(c);
    for (PeerMap& m : c->cache) {
      if (m.own) {
        if (m.va) {
          drv().cuMemUnmap_(m.va, c->heap_bytes);
          drv().cuMemAddressFree_(m.va, c->heap_bytes);
        }
      } else {
        unmap_heap(c, m);
      }
    }
    c->cache.clear();
    if (c->local_handle) drv().cuMemRelease_(c->local_handle);
    if (c->ctr) cudaFree(c->ctr);
    if (c->dbg) cudaFree(c->dbg);
    if (c->hostctl) cudaFreeHost(const_cast<uint32_t*>(c->hostctl));
    cudaGetLastError();
  }
  delete c;
  return TOK_OK;
}

int tok_comm_caps(tok_comm_t* c, tok_caps_t* caps) {
  if (!c || !caps) return fail(TOK_ERR_INVALID, "comm / caps is null");
  memset(caps, 0, sizeof(*caps));
  caps->abi_version = TOK_ABI_VERSION;
  caps->rank = c->rank;
  caps->world = c->world;
  caps->max_world = c->max_world;
  caps->device = c->device;
  caps->multicast = c->mc_va ? 1 : 0;
  caps->p2p = 1;
  caps->epoch = c->epoch;
  caps->staging_bytes = c->cap_bytes;
  caps->heap_bytes = c->heap_bytes;
  caps->one_shot_max = one_shot_limit(c);
  caps->nvls_min = c->nvls_min;
  caps->max_ctas = c->max_ctas;
  caps->sm_count = c->sm_count;
  return TOK_OK;
}

int tok_allreduce_algo(tok_comm_t* c, size_t wire_bytes, int* algo) {
  if (!c || !algo) return fail(TOK_ERR_INVALID, "comm / algo is null");
  *algo = pick_algo(c, wire_bytes);
  return TOK_OK;
}

// ---- symmetric pool ---------------------------------------------------------------------------
// First-fit over the released segments (lowest offset first), else bump.  Deterministic: replicas
// that perform the same allocate/release sequence get the same offsets — which is all the zero-copy
// path needs, and the arrive kernel verifies it for every bucket.
static size_t pool_base_off(const tok_comm* c) { return kFlagBytes + 2 * c->cap_bytes; }

int tok_comm_symm_alloc(tok_comm_t* c, size_t bytes, void** ptr) {
  if (!c || !ptr) return fail(TOK_ERR_INVALID, "comm / ptr is null");
  const size_t need = round_up(std::max<size_t>(bytes, 1), 2u << 20);  // segment-friendly alignment
  std::lock_guard<std::mutex> lock(c->pool_mu);
  char* base = reinterpret_cast<char*>(c->local_va) + pool_base_off(c);
  for (size_t i = 0; i < c->pool_free.size(); ++i) {
    auto& blk = c->pool_free[i];
    if (blk.second < need) continue;
    *ptr = base + blk.first;
    if (blk.second == need) {
      c->pool_free.erase(c->pool_free.begin() + static_cast<long>(i));
    } else {
      blk.first += need;
      blk.second -= need;
    }
    return TOK_OK;
  }
  if (c->pool_used + need > c->pool_bytes)
    return fail(TOK_ERR_INVALID,
                "symmetric pool exhausted: %zu MiB used + %zu MiB requested > %zu MiB (TOK_SYMM_POOL_MB)",
                c->pool_used >> 20, need >> 20, c->pool_bytes >> 20);
  *ptr = base + c->pool_used;
  c->pool_used += need;
  return TOK_OK;
}

int tok_comm_symm_free(tok_comm_t* c, void* ptr, size_t bytes) {
  if (!c) return fail(TOK_ERR_INVALID, "comm is null");
  if (!ptr) return TOK_OK;
  const size_t size = round_up(std::max<size_t>(bytes, 1), 2u << 20);
  std::lock_guard<std::mutex> lock(c->pool_mu);
  const char* base = reinterpret_cast<const char*>(c->local_va) + pool_base_off(c);
  const char* p = static_cast<const char*>(ptr);
  if (p < base || p + size > base + c->pool_used || ((p - base) & ((2u << 20) - 1)))
    return fail(TOK_ERR_INVALID, "pointer %p (+%zu) is not a live symmetric-pool segment", ptr, size);
  const size_t off = static_cast<size_t>(p - base);
  auto it = std::lower_bound(c->pool_free.begin(), c->pool_free.end(), std::make_pair(off, size_t{0}));
  if ((it != c->pool_free.end() && it->first < off + size) ||
      (it != c->pool_free.begin() && (it - 1)->first + (it - 1)->second > off))
    return fail(TOK_ERR_STATE, "symmetric-pool segment at offset %zu released twice", off);
  it = c->pool_free.insert(it, std::make_pair(off, size));
  if (it + 1 != c->pool_free.end() && it->first + it->second == (it + 1)->first) {  // merge right
    it->second += (it + 1)->second;
    c->pool_free.erase(it + 1);
  }
  if (it != c->pool_free.begin() && (it - 1)->first + (it - 1)->second == it->first) {  // merge left
    (it - 1)->second += it->second;
    it = c->pool_free.erase(it) - 1;
  }
  if (it->first + it->second == c->pool_used) {  // the top of the pool shrinks back
    c->pool_used = it->first;
    c->pool_free.erase(it);
  }
  return TOK_OK;
}

int tok_comm_symm_info(tok_comm_t* c, void** base, size_t* bytes, size_t* used) {
  if (!c) return fail(TOK_ERR_INVALID, "comm is null");
  if (base) *base = reinterpret_cast<char*>(c->local_va) + pool_base_off(c);
  if (bytes) *bytes = c->pool_bytes;
  if (used) {
    std::lock_guard<std::mutex> lock(c->pool_mu);
    size_t freed = 0;
    for (auto& b : c->pool_free) freed += b.second;
    *used = c->pool_used - freed;
  }
  return TOK_OK;
}

int tok_comm_use_as_pool(tok_comm_t* c) {
  g_pool_comm.store(c);
  return TOK_OK;
}

// torch.cuda.memory.CUDAPluggableAllocator entry points: segments of a torch.cuda.MemPool are carved
// from the symmetric pool of the communicator selected with tok_comm_use_as_pool() and go back to
// its free list when torch releases them (DDP drops its first-generation buckets after iteration 1).
void* tok_pool_malloc(ptrdiff_t size, int device, void* stream) {
  (void)stream;
  tok_comm* c = g_pool_comm.load();
  if (!c || size <= 0 || device != c->device) return nullptr;
  void* p = nullptr;
  if (tok_comm_symm_alloc(c, static_cast<size_t>(size), &p) != TOK_OK) return nullptr;
  return p;
}

void tok_pool_free(void* ptr, size_t size, int device, void* stream) {
  (void)stream;
  tok_comm* c = g_pool_comm.load();
  if (!c || device != c->device) return;  // communicator already gone: the heap went with it
  tok_comm_symm_free(c, ptr, size);
}

int tok_comm_debug_read(tok_comm_t* c, uint64_t* out, size_t words) {
  if (!c || !out) return fail(TOK_ERR_INVALID, "comm / out is null");
  if (!c->dbg) return fail(TOK_ERR_STATE, "phase timestamps are off (set TOK_DEBUG_PHASES=1 before tok_comm_create)");
  const size_t n = std::min<size_t>(words, kMaxCtas * 8);
  DeviceGuard guard(c->device);
  RT_CHECK(cudaMemcpy(out, c->dbg, n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return TOK_OK;
}

int tok_comm_launches(tok_comm_t* c, uint64_t* launches) {
  if (!c || !launches) return fail(TOK_ERR_INVALID, "comm / launches is null");
  *launches = c->launches.load() + c->arrivals.load();
  return TOK_OK;
}

int tok_comm_stats(tok_comm_t* c, tok_stats_t* st) {
  if (!c || !st) return fail(TOK_ERR_INVALID, "comm / stats is null");
  memset(st, 0, sizeof(*st));
  st->launches = c->launches.load();
  st->arrivals = c->arrivals.load();
  st->elided = c->elided.load();
  st->broadcasts = c->broadcasts.load();
  st->last_algo = c->last_algo.load();
  st->last_ctas = c->last_ctas.load();
  return TOK_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// planning: which kernel a bucket takes
// ------------------------------------------------------------------------------------------------
namespace {

bool is_pow2_scale(float s) {
  int e = 0;
  return s > 0.f && frexpf(s, &e) == 0.5f;
}

struct Plan {
  int algo = 0;          // TOK_ALGO_* or an internal id
  bool inplace = false;  // zero-copy (preceded by an arrival)
  size_t buf_off = 0;
  bool elide = false;
};

void fill_common(const tok_comm* c, KArgs* a) {
  memset(a, 0, sizeof(*a));
  a->stage_off[0] = kFlagBytes;
  a->stage_off[1] = kFlagBytes + c->cap_bytes;
  a->slot_bytes = c->cap_bytes / kMaxWorld;
  for (int r = 0; r < kMaxWorld; ++r) a->peer[r] = c->peer[r];
  a->mc = reinterpret_cast<char*>(c->mc_va);
  a->ctr = c->ctr;
  a->hostctl = c->hostctl_dev;
  a->timeout_ns = c->barrier_timeout_ns;
  a->dbg = c->dbg;
  a->rank = c->rank;
  a->world = c->world;
  a->unroll = c->nvls_unroll;
}

bool in_pool(const tok_comm* c, const void* p, size_t bytes) {
  const char* lo = reinterpret_cast<const char*>(c->local_va) + kFlagBytes + 2 * c->cap_bytes;
  const char* q = static_cast<const char*>(p);
  return q >= lo && q + bytes <= lo + c->pool_bytes;
}

int plan_bucket(const tok_comm* c, const void* in, const void* out, size_t count, int in_dtype,
                int wire_dtype, int out_dtype, float scale, unsigned flags, Plan* pl) {
  const size_t wsz = dtype_size(wire_dtype);
  const size_t isz = dtype_size(in_dtype);
  const bool same_dt = in_dtype == wire_dtype && wire_dtype == out_dtype;
  int algo = static_cast<int>((flags & TOK_FLAG_ALGO_MASK) >> TOK_FLAG_ALGO_SHIFT);
  const bool forced = algo != TOK_ALGO_AUTO;
  if (algo == TOK_ALGO_AUTO) algo = pick_algo(c, count * wsz);
  if (algo == TOK_ALGO_LOCAL_TMA) {
    if (c->world != 1 || !same_dt)
      return fail(TOK_ERR_INVALID, "TOK_ALGO_LOCAL_TMA needs world == 1 and one dtype");
    algo = kAlgoLocalTma;
  } else if (algo < TOK_ALGO_LOCAL || algo > TOK_ALGO_NVLS) {
    return fail(TOK_ERR_INVALID, "unknown algorithm %d", algo);
  }
  if ((algo == TOK_ALGO_LOCAL || algo == kAlgoLocalTma) && c->world != 1)
    return fail(TOK_ERR_INVALID, "TOK_ALGO_LOCAL is only valid for world == 1 (world is %d)",
                c->world);
  if (algo == TOK_ALGO_NVLS && !c->mc_va)
    return fail(TOK_ERR_UNSUPPORTED,
                "NVLS requested but no multicast object is bound for this group");
  if (c->world == 1) {
    // a bucket that is already what the caller asked for needs no pass over HBM at all
    pl->elide = !forced && in == out && same_dt && scale == 1.0f && !(flags & TOK_FLAG_NO_ELIDE);
    if (algo == TOK_ALGO_LOCAL && !forced && same_dt && c->local_tma &&
        count * wsz >= (1u << 20))
      algo = kAlgoLocalTma;
    pl->algo = algo;
    return TOK_OK;
  }
  // Zero-copy: the bucket lives in the symmetric pool (same offset on every replica), is exchanged
  // in place, in its own dtype, in whole 16-byte packs -> peers read / multicast it directly.
  const bool pool_ok = c->zero_copy && !(flags & TOK_FLAG_NO_ZERO_COPY) && in == out && same_dt &&
                       in_pool(c, in, count * isz) && (count * wsz) % 16 == 0;
  // a pool bucket leaves the one-shot range earlier: its exchange needs no staging pass (measured at
  // N=2, profiles/r02_sweep_n2.json: in place 30.9 vs one-shot 30.0 us at 8 MiB, 43.6 vs 47.0 at 16)
  if (!forced && algo == TOK_ALGO_ONE_SHOT && pool_ok && c->world == 2 && count * wsz >= (8u << 20))
    algo = TOK_ALGO_TWO_SHOT;
  bool inplace = pool_ok && (algo == TOK_ALGO_TWO_SHOT || algo == TOK_ALGO_NVLS);
  if (inplace) {
    // The switch can only scale the SUM.  That equals the specified PRE semantics (scale every
    // contribution, then sum) when the caller asked for POST or the factor is a power of two; a
    // 16-bit float sum may also overflow before the 1/N is applied.  Everything else takes the P2P
    // in-place kernel, which applies PRE exactly as the staged path does.
    const bool post = (flags & TOK_FLAG_SCALE_POST) != 0;
    const bool nvls_exact = (post || is_pow2_scale(scale)) && (wire_dtype != TOK_F16 || post);
    // (pick_algo's rule stands for pool buckets too: with 3-4 replicas the in-switch reduction stops
    // paying off past ~12 MiB — measured in place at N=4 on the 22.9 / 28.3 MB DDP buckets: P2P
    // reduce+push 83.0 us vs NVLS 95.7 us, profiles/r02_zc_tune_n4.json; with >= 5 replicas NVLS wins:
    // 81 vs 98 us at N=8, profiles/r02_zc_tune_n8.json)
    if (algo == TOK_ALGO_NVLS && !nvls_exact) {
      if (forced)
        inplace = false;  // honour the forced algorithm through the staged kernel
      else
        algo = TOK_ALGO_TWO_SHOT;
    }
  }
  if (inplace) {
    pl->buf_off = static_cast<size_t>(static_cast<const char*>(in) -
                                      reinterpret_cast<const char*>(c->local_va));
    algo = (algo == TOK_ALGO_NVLS) ? kAlgoNvlsInplace : kAlgoTwoShotInplace;
  }
  pl->inplace = inplace;
  pl->algo = algo;
  return TOK_OK;
}

int check_bucket_args(tok_comm* c, const void* in, const void* out, int in_dtype, int wire_dtype,
                      int out_dtype) {
  if (!c) return fail(TOK_ERR_INVALID, "comm is null");
  auto bad_dt = [](int d) { return d != TOK_F32 && d != TOK_BF16 && d != TOK_F16; };
  if (bad_dt(in_dtype) || bad_dt(wire_dtype) || bad_dt(out_dtype))
    return fail(TOK_ERR_INVALID, "unsupported dtype (in %d wire %d out %d)", in_dtype, wire_dtype,
                out_dtype);
  if (!in || !out) return fail(TOK_ERR_INVALID, "in / out is null");
  if ((reinterpret_cast<uintptr_t>(in) & 15) || (reinterpret_cast<uintptr_t>(out) & 15))
    return fail(TOK_ERR_ALIGN, "bucket pointers must be 16-byte aligned (in %p out %p)", in, out);
  return tok_comm_status(c);
}

int do_arrive(tok_comm* c, size_t buf_off, void* stream) {
  KArgs a;
  fill_common(c, &a);
  a.buf_off = buf_off;
  int e = launch_arrive(a, stream);
  if (e != 0)
    return fail(TOK_ERR_CUDA, "arrive kernel launch failed: %s",
                cudaGetErrorString(static_cast<cudaError_t>(e)));
  c->arrivals.fetch_add(1);
  return TOK_OK;
}

}  // namespace

extern "C" {

int tok_bucket_arrive(tok_comm_t* c, const void* bucket, size_t count, int dtype, float scale,
                      unsigned flags, void* cuda_stream, int* arrived) {
  if (arrived) *arrived = 0;
  if (count == 0) return TOK_OK;
  int st = check_bucket_args(c, bucket, bucket, dtype, dtype, dtype);
  if (st != TOK_OK) return st;
  Plan pl;
  st = plan_bucket(c, bucket, bucket, count, dtype, dtype, dtype, scale, flags, &pl);
  if (st != TOK_OK) return st;
  if (!pl.inplace) return TOK_OK;  // staged kernels carry their own barriers
  DeviceGuard guard(c->device);
  st = do_arrive(c, pl.buf_off, cuda_stream);
  if (st == TOK_OK && arrived) *arrived = 1;
  return st;
}

int tok_allreduce_bucket(tok_comm_t* c, const void* in, void* out, size_t count, int in_dtype,
                         int wire_dtype, int out_dtype, float scale, unsigned flags,
                         void* cuda_stream) {
  if (c && count == 0) return TOK_OK;
  int st = check_bucket_args(c, in, out, in_dtype, wire_dtype, out_dtype);
  if (st != TOK_OK) return st;
  Plan pl;
  st = plan_bucket(c, in, out, count, in_dtype, wire_dtype, out_dtype, scale, flags, &pl);
  if (st != TOK_OK) return st;
  if (pl.elide) {
    c->elided.fetch_add(1);
    return TOK_OK;
  }
  const int algo = pl.algo;
  const bool inplace = pl.inplace;
  const int P = pack_elems(in_dtype, wire_dtype, out_dtype);
  const size_t wsz = dtype_size(wire_dtype);
  const size_t isz = dtype_size(in_dtype);
  const size_t osz = dtype_size(out_dtype);
  const bool local = algo == TOK_ALGO_LOCAL || algo == kAlgoLocalTma;

  // largest element count one launch may take (multiple of 8 elements -> 16-byte aligned chunks)
  size_t launch_cap = c->cap_bytes / wsz;
  if (algo == TOK_ALGO_ONE_SHOT) launch_cap = (c->cap_bytes / kMaxWorld) / wsz;
  launch_cap = launch_cap / (static_cast<size_t>(P) * kMaxWorld) * (static_cast<size_t>(P) * kMaxWorld);
  if (local || inplace) launch_cap = (static_cast<size_t>(1) << 40);

  DeviceGuard guard(c->device);
  if (inplace && !(flags & TOK_FLAG_ARRIVED)) {
    st = do_arrive(c, pl.buf_off, cuda_stream);
    if (st != TOK_OK) return st;
  }
  KArgs a;
  fill_common(c, &a);
  a.buf_off = pl.buf_off;
  a.scale = scale;
  a.flags = flags & TOK_FLAG_SCALE_POST;

  for (size_t off = 0; off < count; off += launch_cap) {
    const size_t n = std::min(launch_cap, count - off);
    a.in = static_cast<const char*>(in) + off * isz;
    a.out = static_cast<char*>(out) + off * osz;
    a.count = n;
    a.total_packs = (n + P - 1) / P;
    int ctas;
    if (algo == TOK_ALGO_LOCAL) {
      // one even wave, at most 2 CTAs per SM, >= 8 packs per thread
      const size_t full = n / P;
      const size_t want = (full + kThreads * 8 - 1) / (kThreads * 8);
      const size_t g = std::min<size_t>(std::max<size_t>(want, 1), static_cast<size_t>(c->sm_count) * 2);
      a.packs_per_cta = (std::max<size_t>(full, 1) + g - 1) / g;
      ctas = static_cast<int>(g);
    } else if (algo == kAlgoLocalTma) {
      const size_t tiles = (n / P * 16 + 16383) / 16384;
      ctas = static_cast<int>(std::min<size_t>(std::max<size_t>(tiles, 1), static_cast<size_t>(c->sm_count) * 2));
      a.packs_per_cta = 0;
    } else {
      const size_t bytes = a.total_packs * P * wsz;
      size_t cap_ctas = c->max_ctas;
      if (inplace) {
        // In-place NVLS saturates the NVSwitch reduction path with few requesters: in the isolated
        // sweeps (profiles/r01_sweep_n{4,8}_zero_copy_cta_tuning.json) 16 CTAs beat 64 from 32 MiB
        // up at N=8 (91 vs 112 us at 32 MiB, 160 vs 184 at 64 MiB).  Below that the evidence is
        // within run-to-run noise, and the ResNet-50 buckets (22.9 / 28.3 MB) measured best with 64
        // CTAs inside bench.py (77 us/bucket vs 87 with 16-32 CTAs), so 64 stays the default there.
        if (c->zc_ctas)
          cap_ctas = c->zc_ctas;
        else if (algo == kAlgoNvlsInplace && bytes >= (32u << 20))
          cap_ctas = 16;
        else
          cap_ctas = 64;
      }
      size_t g = std::min<size_t>(std::max<size_t>((bytes + c->cta_bytes - 1) / c->cta_bytes, 1),
                                  cap_ctas);
      size_t L = (a.total_packs + g - 1) / g;
      if (algo != TOK_ALGO_ONE_SHOT) L = round_up(L, c->world);
      if (inplace) a.buf_off = pl.buf_off + off * isz;
      a.packs_per_cta = L;
      ctas = static_cast<int>((a.total_packs + L - 1) / L);
    }
    int e = launch_allreduce(algo, in_dtype, wire_dtype, out_dtype, ctas, a, cuda_stream);
    if (e != 0)
      return fail(TOK_ERR_CUDA, "allreduce kernel launch failed: %s",
                  cudaGetErrorString(static_cast<cudaError_t>(e)));
    c->launches.fetch_add(1);
    c->last_algo.store(algo);
    c->last_ctas.store(ctas);
  }
  return TOK_OK;
}

int tok_comm_debug_peek(tok_comm_t* c, int rank, size_t byte_off, uint32_t* out, size_t words) {
  if (!c || !out) return fail(TOK_ERR_INVALID, "comm / out is null");
  if (rank < 0 || rank >= c->world || byte_off + words * 4 > kFlagBytes)
    return fail(TOK_ERR_INVALID, "rank / offset out of range");
  DeviceGuard guard(c->device);
  RT_CHECK(cudaMemcpy(out, c->peer[rank] + byte_off, words * 4, cudaMemcpyDeviceToHost));
  return TOK_OK;
}

int tok_comm_debug_barrier(tok_comm_t* c, int variant, int ctas, size_t count, void* cuda_stream) {
  if (!c) return fail(TOK_ERR_INVALID, "comm is null");
  if (variant < 0 || variant > 4 || ctas < 1 || ctas > 64)
    return fail(TOK_ERR_INVALID, "variant 0..4, ctas 1..64");
  if (c->world < 2) return fail(TOK_ERR_STATE, "a barrier needs world >= 2");
  int st = tok_comm_status(c);
  if (st != TOK_OK) return st;
  DeviceGuard guard(c->device);
  KArgs a;
  fill_common(c, &a);
  a.count = count;
  a.flags = static_cast<uint32_t>(variant);
  int e = launch_barrier_bench(ctas, a, cuda_stream);
  if (e != 0)
    return fail(TOK_ERR_CUDA, "barrier bench launch failed: %s",
                cudaGetErrorString(static_cast<cudaError_t>(e)));
  return TOK_OK;
}

int tok_broadcast(tok_comm_t* c, void* buf, size_t bytes, int root, void* cuda_stream) {
  if (!c) return fail(TOK_ERR_INVALID, "comm is null");
  if (root < 0 || root >= c->world)
    return fail(TOK_ERR_INVALID, "broadcast root %d out of range (world %d)", root, c->world);
  if (bytes == 0 || c->world == 1) return TOK_OK;
  if (!buf) return fail(TOK_ERR_INVALID, "buf is null");
  if (reinterpret_cast<uintptr_t>(buf) & 15)
    return fail(TOK_ERR_ALIGN, "broadcast buffer must be 16-byte aligned (%p)", buf);
  int st = tok_comm_status(c);
  if (st != TOK_OK) return st;
  DeviceGuard guard(c->device);
  const bool pooled = c->zero_copy && in_pool(c, buf, bytes) && bytes % 16 == 0;
  KArgs a;
  fill_common(c, &a);
  a.root = root;
  auto grid = [&](size_t nbytes, KArgs* k) {
    const size_t packs = std::max<size_t>(nbytes / 16, 1);
    const size_t g = std::min<size_t>(std::max<size_t>((nbytes + c->cta_bytes - 1) / c->cta_bytes, 1), 128);
    k->packs_per_cta = (packs + g - 1) / g;
    return static_cast<int>((packs + k->packs_per_cta - 1) / k->packs_per_cta);
  };
  if (pooled) {
    const size_t off = static_cast<size_t>(static_cast<char*>(buf) - reinterpret_cast<char*>(c->local_va));
    st = do_arrive(c, off, cuda_stream);
    if (st != TOK_OK) return st;
    a.buf_off = off;
    a.in = buf;
    a.out = buf;
    a.count = bytes;
    // one multimem.st stream feeds N-1 receivers; with a single receiver it saves nothing and a
    // pull (the receiver's own LDG.128 over NVLink) is the faster copy
    const int mode = (c->mc_va && c->world >= 3) ? kBcastMcPush : kBcastPull;
    const int ctas = grid(bytes, &a);
    int e = launch_broadcast(mode, ctas, a, cuda_stream);
    if (e != 0)
      return fail(TOK_ERR_CUDA, "broadcast kernel launch failed: %s",
                  cudaGetErrorString(static_cast<cudaError_t>(e)));
    c->launches.fetch_add(1);
    c->last_algo.store(mode);
    c->last_ctas.store(ctas);
  } else {
    const size_t cap = c->cap_bytes;  // one staging buffer per launch
    for (size_t off = 0; off < bytes; off += cap) {
      const size_t n = std::min(cap, bytes - off);
      a.in = static_cast<char*>(buf) + off;
      a.out = static_cast<char*>(buf) + off;
      a.count = n;
      const int ctas = grid(n, &a);
      int e = launch_broadcast(kBcastStaged, ctas, a, cuda_stream);
      if (e != 0)
        return fail(TOK_ERR_CUDA, "broadcast kernel launch failed: %s",
                    cudaGetErrorString(static_cast<cudaError_t>(e)));
      c->launches.fetch_add(1);
      c->last_algo.store(kBcastStaged);
      c->last_ctas.store(ctas);
    }
  }
  c->broadcasts.fetch_add(1);
  return TOK_OK;
}

}  // extern "C"
