// sb_exchange.cuh -- the collectives of a contig-sharded run (SURVEY.md 8e, mode 2).
//
// When the reference genome's index does not fit one GPU, its contigs are partitioned over the
// ranks; every rank sees every read chunk, searches / sorts / chains against its own contigs
// and three small exchanges per pipeline step make the result identical to the unsharded run:
//   1. all-reduce MAX of a 4-double control vector after the search (anchor overflow is a
//      collective decision, the batch-size estimate stays identical on every rank);
//   2. all-reduce MAX of seg_max[] -- one fp32 running max per (read chunk, contig, strand)
//      bucket, so each rank can apply the reference's global `max_chaining_score / 2` filter in
//      the reference's bucket order (spatial_index.cc:419-422, :542-549);
//   3. all-gather of the fixed-size chain candidate records (k_chain.cuh CandRec), after which
//      GeneratePrimaryChains / MAPQ / the StreamingMap decision run redundantly on every rank.
// Carried anchors never move: they stay on the rank that owns their contig.
//
// Two backends behind one interface:
//   NcclExchange   one process per GPU (torchrun): ncclAllReduce / ncclAllGather on the context's
//                  stream, i.e. over NVLink 5 / NVSwitch on a B200 box.  NCCL is bound at run
//                  time with dlopen("libnccl.so.2") -- inside a torch process that is torch's own
//                  copy -- so the library has no link-time dependency on it.
//   LocalExchange  several contexts inside ONE process, each driven by its own host thread
//                  (same GPU or peers): rendezvous on a host barrier, cudaMemcpyPeerAsync and a
//                  reduction kernel.  This is how the sharded path is parity-tested on one GPU.
#ifndef SB_EXCHANGE_CUH
#define SB_EXCHANGE_CUH

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdint.h>

#include <condition_variable>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include <algorithm>

#include "sb_device.cuh"

namespace sb {

enum ExDType { EX_F32 = 0, EX_F64 = 1, EX_U32 = 2 };
enum ExOp { EX_MAX = 0, EX_SUM = 1 };

// dst[i] = op(dst[i], src[r][i]) over the gathered copies (own copy included in src, skipped)
template <class T>
__global__ void k_ex_reduce(T *__restrict__ dst, const T *__restrict__ gathered, size_t n, uint32_t world,
                            uint32_t self, int op) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  T v = dst[i];
  for (uint32_t r = 0; r < world; ++r) {
    if (r == self) continue;
    const T o = gathered[(size_t)r * n + i];
    v = op == EX_MAX ? (o > v ? o : v) : (T)(v + o);
  }
  dst[i] = v;
}

struct Exchange {
  int rank = 0, world = 1;
  virtual ~Exchange() {}
  // in place on a device buffer of n elements; ordered on stream s
  virtual int allreduce(void *d_buf, size_t n, ExDType t, ExOp op, cudaStream_t s, std::string &err) = 0;
  // d_recv receives world * bytes (rank-major); d_send may NOT alias d_recv
  virtual int allgather(const void *d_send, void *d_recv, size_t bytes, cudaStream_t s, std::string &err) = 0;
  // root's d_buf -> everybody's d_buf (in place)
  virtual int broadcast(void *d_buf, size_t bytes, int root, cudaStream_t s, std::string &err) = 0;
};

// ------------------------------------------------------------------ in-process group
struct LocalGroup {
  int world = 0;
  std::mutex m;
  std::condition_variable cv;
  int arrived = 0;
  uint64_t generation = 0;
  bool broken = false;               // a member failed: everybody bails out instead of waiting
  std::vector<const void *> send;    // published send buffers
  std::vector<int> device;
  void barrier() {
    std::unique_lock<std::mutex> lk(m);
    const uint64_t g = generation;
    if (++arrived == world) {
      arrived = 0;
      ++generation;
      cv.notify_all();
    } else {
      cv.wait(lk, [&] { return generation != g || broken; });
    }
  }
  void abort_all() {
    std::lock_guard<std::mutex> lk(m);
    broken = true;
    cv.notify_all();
  }
};

struct LocalExchange : Exchange {
  std::shared_ptr<LocalGroup> g;
  int device = 0;
  DevBuf<unsigned char> tmp;

  int allgather(const void *d_send, void *d_recv, size_t bytes, cudaStream_t s, std::string &err) override {
    cudaError_t e = cudaStreamSynchronize(s);  // my send buffer is complete
    if (e != cudaSuccess) {
      err = std::string("local exchange: ") + cudaGetErrorString(e);
      g->abort_all();
      return SMB_ERR_CUDA;
    }
    g->send[rank] = d_send;
    g->barrier();
    if (g->broken) {
      err = "local exchange: a group member failed";
      return SMB_ERR_STATE;
    }
    for (int r = 0; r < world && e == cudaSuccess; ++r)
      e = cudaMemcpyPeerAsync((unsigned char *)d_recv + (size_t)r * bytes, device, g->send[r], g->device[r], bytes, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
      err = std::string("local exchange: ") + cudaGetErrorString(e);
      g->abort_all();
      return SMB_ERR_CUDA;
    }
    g->barrier();  // nobody reuses its send buffer before every peer has read it
    if (g->broken) {
      err = "local exchange: a group member failed";
      return SMB_ERR_STATE;
    }
    return SMB_OK;
  }

  int broadcast(void *d_buf, size_t bytes, int root, cudaStream_t s, std::string &err) override {
    cudaError_t e = cudaStreamSynchronize(s);  // the root's buffer is complete
    if (e != cudaSuccess) {
      err = std::string("local exchange: ") + cudaGetErrorString(e);
      g->abort_all();
      return SMB_ERR_CUDA;
    }
    g->send[rank] = d_buf;
    g->barrier();
    if (g->broken) {
      err = "local exchange: a group member failed";
      return SMB_ERR_STATE;
    }
    if (rank != root && bytes) {
      e = cudaMemcpyPeerAsync(d_buf, device, g->send[root], g->device[root], bytes, s);
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);
      if (e != cudaSuccess) {
        err = std::string("local exchange: ") + cudaGetErrorString(e);
        g->abort_all();
        return SMB_ERR_CUDA;
      }
    }
    g->barrier();  // the root does not touch its buffer before every peer has read it
    if (g->broken) {
      err = "local exchange: a group member failed";
      return SMB_ERR_STATE;
    }
    return SMB_OK;
  }

  int allreduce(void *d_buf, size_t n, ExDType t, ExOp op, cudaStream_t s, std::string &err) override {
    const size_t es = t == EX_F64 ? 8 : 4;
    if (tmp.ensure(n * es * (size_t)world) != cudaSuccess) {
      err = "local exchange: out of device memory";
      g->abort_all();
      return SMB_ERR_CUDA;
    }
    int rc = allgather(d_buf, tmp.p, n * es, s, err);
    if (rc) return rc;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (t == EX_F32) k_ex_reduce<float><<<blocks, 256, 0, s>>>((float *)d_buf, (const float *)tmp.p, n, world, rank, op);
    else if (t == EX_F64) k_ex_reduce<double><<<blocks, 256, 0, s>>>((double *)d_buf, (const double *)tmp.p, n, world, rank, op);
    else k_ex_reduce<uint32_t><<<blocks, 256, 0, s>>>((uint32_t *)d_buf, (const uint32_t *)tmp.p, n, world, rank, op);
    if (cudaGetLastError() != cudaSuccess) {
      err = "local exchange: reduce kernel launch failed";
      return SMB_ERR_CUDA;
    }
    return SMB_OK;
  }
};

// ------------------------------------------------------------------ NCCL, bound at run time
struct NcclApi {
  typedef struct ncclComm *comm_t;
  struct unique_id { char internal[128]; };  // ncclUniqueId (NCCL_UNIQUE_ID_BYTES)
  int (*GetUniqueId)(unique_id *) = nullptr;
  int (*CommInitRank)(comm_t *, int, unique_id, int) = nullptr;
  int (*CommDestroy)(comm_t) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, comm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, comm_t, cudaStream_t) = nullptr;
  int (*Broadcast)(const void *, void *, size_t, int, int, comm_t, cudaStream_t) = nullptr;
  void *handle = nullptr;
  std::string error;
  bool load() {
    if (handle) return true;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *nm : names) {
      handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (handle) break;
    }
    if (!handle) {
      error = std::string("cannot load NCCL: ") + dlerror();
      return false;
    }
    auto sym = [&](const char *nm) -> void * {
      void *p = dlsym(handle, nm);
      if (!p) error = std::string("NCCL symbol missing: ") + nm;
      return p;
    };
    GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
    CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
    GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
    AllReduce = (decltype(AllReduce))sym("ncclAllReduce");
    AllGather = (decltype(AllGather))sym("ncclAllGather");
    Broadcast = (decltype(Broadcast))sym("ncclBroadcast");
    if (!GetUniqueId || !CommInitRank || !CommDestroy || !GetErrorString || !AllReduce || !AllGather || !Broadcast) {
      dlclose(handle);
      handle = nullptr;
      return false;
    }
    return true;
  }
  static NcclApi &get() {
    static NcclApi api;
    return api;
  }
};

struct NcclExchange : Exchange {
  NcclApi::comm_t comm = nullptr;
  ~NcclExchange() override {
    if (comm) NcclApi::get().CommDestroy(comm);
  }
  int check(int rc, const char *what, std::string &err) {
    if (rc == 0) return SMB_OK;
    err = std::string(what) + ": " + NcclApi::get().GetErrorString(rc);
    return SMB_ERR_CUDA;
  }
  int allreduce(void *d_buf, size_t n, ExDType t, ExOp op, cudaStream_t s, std::string &err) override {
    // nccl.h: ncclUint32 = 3, ncclFloat32 = 7, ncclFloat64 = 8; ncclSum = 0, ncclMax = 2
    const int dt = t == EX_F32 ? 7 : (t == EX_F64 ? 8 : 3);
    return check(NcclApi::get().AllReduce(d_buf, d_buf, n, dt, op == EX_MAX ? 2 : 0, comm, s), "ncclAllReduce", err);
  }
  int allgather(const void *d_send, void *d_recv, size_t bytes, cudaStream_t s, std::string &err) override {
    return check(NcclApi::get().AllGather(d_send, d_recv, bytes, /*ncclUint8*/ 1, comm, s), "ncclAllGather", err);
  }
  int broadcast(void *d_buf, size_t bytes, int root, cudaStream_t s, std::string &err) override {
    // in chunks below 2^31 bytes: one ncclBroadcast per GB keeps every count comfortably in range
    for (size_t at = 0; at < bytes; at += (size_t)1 << 30) {
      const size_t n = std::min<size_t>((size_t)1 << 30, bytes - at);
      int rc = check(NcclApi::get().Broadcast((const unsigned char *)d_buf + at, (unsigned char *)d_buf + at, n,
                                              /*ncclUint8*/ 1, root, comm, s), "ncclBroadcast", err);
      if (rc) return rc;
    }
    return SMB_OK;
  }
};

}  // namespace sb
#endif
