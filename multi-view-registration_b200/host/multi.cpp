// multi.cpp -- the multi-GPU form of the multi-view-register entry point, inside the C ABI.
//
// The reference is ONE process (its registration runs on a QtConcurrent pool thread, mvr/src/registrator.cpp:606, 696);
// what shards is the set of ring edges i -> (i + 1) % V it hands to LUM / computeError (mvr/src/registrator.cpp:482-487,
// 640-651).  mvr_register_turntable_multi keeps that shape: one caller, one call -- inside, one host thread per GPU
// aligns a contiguous block of the ring's pairs with its own Registrator (every view a rank needs is uploaded to that
// rank's GPU only, point data never crosses GPUs), the ranks exchange their fixed-size pair records (96 bytes per pair)
// with ONE ncclAllGather over NVLink, and the ring is closed on the host from the gathered records.
//
// NCCL is bound at run time (dlopen of libnccl.so.2: the system library, or the one the host process already loaded),
// so the library itself has no link-time dependency on it; a missing or failing NCCL surfaces as MVR_ERR_NCCL.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "registrator.h"

using namespace mvr;

namespace {

// the few NCCL entry points used, with the ABI of nccl.h (NCCL 2.x): ncclResult_t is an int enum (0 = success),
// ncclComm_t an opaque pointer, ncclChar = 0
typedef void* nccl_comm_t;
struct NcclApi {
  void* handle = nullptr;
  int (*CommInitAll)(nccl_comm_t*, int, const int*) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  std::string err;
  bool load() {
    if (handle) return true;
    const char* names[] = {std::getenv("MVR_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      if (!n || !*n) continue;
      handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (handle) break;
    }
    if (!handle) { err = "libnccl.so.2 not found (set MVR_NCCL_LIB)"; return false; }
    CommInitAll = (int (*)(nccl_comm_t*, int, const int*))dlsym(handle, "ncclCommInitAll");
    CommDestroy = (int (*)(nccl_comm_t))dlsym(handle, "ncclCommDestroy");
    AllGather = (int (*)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t))dlsym(handle, "ncclAllGather");
    GetErrorString = (const char* (*)(int))dlsym(handle, "ncclGetErrorString");
    if (!CommInitAll || !CommDestroy || !AllGather) { err = "libnccl lacks ncclCommInitAll / ncclAllGather"; handle = nullptr; return false; }
    return true;
  }
};

struct Rank {
  int device = 0;
  std::unique_ptr<Registrator> reg;
  cudaStream_t stream = nullptr;        // carries the exchange
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  void* d_send = nullptr;               // block * 96 bytes
  void* d_recv = nullptr;               // n_ranks * block * 96 bytes
  mvr_pair_record* h_recv = nullptr;    // pinned
  mvr_pair_record* h_send = nullptr;    // pinned
  size_t cap_pairs = 0;                 // block the exchange buffers are sized for
  std::vector<void*> resident;          // per view: device copy made by mvr_multi_upload (nullptr: none)
  std::vector<size_t> resident_n;
  int status = MVR_OK;
  std::string err;
  double ms = 0;
};

void pair_block(int rank, int world, int n_pairs, int* p0, int* p1) {
  *p0 = (int)(((long long)rank * n_pairs) / world);
  *p1 = (int)(((long long)(rank + 1) * n_pairs) / world);
}

}  // namespace

struct mvr_multi {
  std::vector<Rank> ranks;
  std::vector<nccl_comm_t> comms;
  NcclApi nccl;
  std::string err;
  int resident_views = 0;
};

namespace {

int fail(mvr_multi* m, int code, const std::string& msg) {
  if (m) m->err = msg;
  return code;
}

void free_resident(Rank& r) {
  cudaSetDevice(r.device);
  for (void* p : r.resident) if (p) cudaFree(p);
  r.resident.clear();
  r.resident_n.clear();
}

int ensure_exchange(Rank& r, int world, size_t block) {
  if (block <= r.cap_pairs) return MVR_OK;
  cudaSetDevice(r.device);
  if (r.d_send) cudaFree(r.d_send);
  if (r.d_recv) cudaFree(r.d_recv);
  if (r.h_recv) cudaFreeHost(r.h_recv);
  if (r.h_send) cudaFreeHost(r.h_send);
  r.d_send = r.d_recv = nullptr; r.h_recv = r.h_send = nullptr; r.cap_pairs = 0;
  const size_t rec = sizeof(mvr_pair_record);
  if (cudaMalloc(&r.d_send, block * rec) != cudaSuccess || cudaMalloc(&r.d_recv, (size_t)world * block * rec) != cudaSuccess ||
      cudaMallocHost((void**)&r.h_recv, (size_t)world * block * rec) != cudaSuccess || cudaMallocHost((void**)&r.h_send, block * rec) != cudaSuccess)
    return MVR_ERR_ALLOC;
  r.cap_pairs = block;
  return MVR_OK;
}

// What one rank does for one registration: its block of ring pairs, then the exchange.
void rank_work(mvr_multi* m, int k, const mvr_view* views, int V, const mvr_turntable_params* prm, bool use_resident) {
  Rank& r = m->ranks[(size_t)k];
  const int world = (int)m->ranks.size();
  r.status = MVR_OK; r.err.clear(); r.ms = 0;
  cudaSetDevice(r.device);
  int p0, p1;
  pair_block(k, world, V, &p0, &p1);
  size_t block = 0;
  for (int q = 0; q < world; ++q) { int a, b; pair_block(q, world, V, &a, &b); block = std::max(block, (size_t)(b - a)); }
  if ((r.status = ensure_exchange(r, world, std::max<size_t>(block, 1)))) { r.err = "exchange buffers"; return; }
  cudaEventRecord(r.ev0, r.stream);
  // this rank's views: the two ends of each of its pairs
  std::vector<View> v((size_t)V);
  for (int i = 0; i < V; ++i) {
    View& o = v[(size_t)i];
    o.view = i;
    if (views[i].init_pose) { std::memcpy(o.pose.m, views[i].init_pose, sizeof(o.pose.m)); o.pose_is_identity = false; }
    bool need = false;
    for (int p = p0; p < p1; ++p) if (i == p % V || i == (p + 1) % V) need = true;
    if (!need) continue;
    if (use_resident && (size_t)i < r.resident.size() && r.resident[(size_t)i]) {
      o.points = (const PointXYZ*)r.resident[(size_t)i]; o.size = r.resident_n[(size_t)i]; o.on_device = true;
    } else {
      o.points = (const PointXYZ*)views[i].xyzw; o.size = views[i].n; o.on_device = false;
    }
  }
  mvr_turntable_params mine = *prm;
  mine.mode = MVR_REGISTER_RING_PAIRS;
  mine.pair_begin = p0; mine.pair_end = p1;
  std::vector<mvr_pair_report> rep;
  if (p1 > p0) {
    r.status = r.reg->multiViewRegister(v, mine, rep);
    if (r.status) { r.err = r.reg->lastError(); }
  }
  // pack, exchange, unpack
  std::memset(r.h_send, 0, block * sizeof(mvr_pair_record));
  for (int p = p0; p < p1 && r.status == MVR_OK; ++p) {
    mvr_pair_record& o = r.h_send[p - p0];
    const mvr_pair_report& s = rep[(size_t)p];
    std::memcpy(o.pose, s.pose, sizeof(o.pose));
    o.n_correspondences = s.n_correspondences; o.iterations = s.iterations; o.status = s.status; o.reserved = 0;
    o.mse = s.mse; o.nn_queries = s.nn_queries;
  }
  if (world == 1) {
    std::memcpy(r.h_recv, r.h_send, block * sizeof(mvr_pair_record));
  } else {
    // every rank takes part in the collective even after a local failure (its records then carry status = -1)
    if (r.status != MVR_OK) for (size_t q = 0; q < block; ++q) r.h_send[q].status = -1;
    const size_t bytes = block * sizeof(mvr_pair_record);
    cudaMemcpyAsync(r.d_send, r.h_send, bytes, cudaMemcpyHostToDevice, r.stream);
    const int rc = m->nccl.AllGather(r.d_send, r.d_recv, bytes, /*ncclChar*/ 0, m->comms[(size_t)k], r.stream);
    if (rc != 0) {
      r.status = MVR_ERR_NCCL;
      r.err = std::string("ncclAllGather: ") + (m->nccl.GetErrorString ? m->nccl.GetErrorString(rc) : "error");
    }
    cudaMemcpyAsync(r.h_recv, r.d_recv, (size_t)world * bytes, cudaMemcpyDeviceToHost, r.stream);
  }
  cudaEventRecord(r.ev1, r.stream);
  if (cudaStreamSynchronize(r.stream) != cudaSuccess && r.status == MVR_OK) { r.status = MVR_ERR_CUDA; r.err = "exchange stream"; }
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, r.ev0, r.ev1) == cudaSuccess) r.ms = ms;
}

}  // namespace

extern "C" {

int mvr_multi_create(const int* devices, int n_devices, mvr_multi** out) {
  if (!out || n_devices < 1 || n_devices > 64) return MVR_ERR_BAD_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return MVR_ERR_CUDA;
  std::unique_ptr<mvr_multi> m(new mvr_multi());
  m->ranks.resize((size_t)n_devices);
  std::vector<int> devs((size_t)n_devices);
  for (int k = 0; k < n_devices; ++k) {
    const int d = devices ? devices[k] : k;
    if (d < 0 || d >= count) return MVR_ERR_BAD_ARG;
    for (int j = 0; j < k; ++j) if (devs[(size_t)j] == d) return MVR_ERR_BAD_ARG;   // one rank per GPU
    devs[(size_t)k] = d;
  }
  for (int k = 0; k < n_devices; ++k) {
    Rank& r = m->ranks[(size_t)k];
    r.device = devs[(size_t)k];
    r.reg.reset(new Registrator(r.device, 1));
    if (!r.reg->ok()) return MVR_ERR_CUDA;
    cudaSetDevice(r.device);
    if (cudaStreamCreateWithFlags(&r.stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&r.ev0) != cudaSuccess ||
        cudaEventCreate(&r.ev1) != cudaSuccess)
      return MVR_ERR_CUDA;
  }
  if (n_devices > 1) {
    if (!m->nccl.load()) { std::fprintf(stderr, "mvr_multi_create: %s\n", m->nccl.err.c_str()); return MVR_ERR_NCCL; }
    m->comms.assign((size_t)n_devices, nullptr);
    const int rc = m->nccl.CommInitAll(m->comms.data(), n_devices, devs.data());
    if (rc != 0) {
      std::fprintf(stderr, "mvr_multi_create: ncclCommInitAll: %s\n", m->nccl.GetErrorString ? m->nccl.GetErrorString(rc) : "error");
      m->comms.clear();
      return MVR_ERR_NCCL;
    }
  }
  *out = m.release();
  return MVR_OK;
}

int mvr_multi_destroy(mvr_multi* m) {
  if (!m) return MVR_OK;
  for (size_t k = 0; k < m->ranks.size(); ++k) {
    Rank& r = m->ranks[k];
    cudaSetDevice(r.device);
    if (r.stream) cudaStreamSynchronize(r.stream);
    if (k < m->comms.size() && m->comms[k]) m->nccl.CommDestroy(m->comms[k]);
    free_resident(r);
    if (r.d_send) cudaFree(r.d_send);
    if (r.d_recv) cudaFree(r.d_recv);
    if (r.h_recv) cudaFreeHost(r.h_recv);
    if (r.h_send) cudaFreeHost(r.h_send);
    if (r.ev0) cudaEventDestroy(r.ev0);
    if (r.ev1) cudaEventDestroy(r.ev1);
    if (r.stream) cudaStreamDestroy(r.stream);
    r.reg.reset();
  }
  delete m;
  return MVR_OK;
}

const char* mvr_multi_last_error(mvr_multi* m) { return m ? m->err.c_str() : "null handle"; }
int mvr_multi_devices(mvr_multi* m) { return m ? (int)m->ranks.size() : 0; }
mvr_ctx* mvr_multi_context(mvr_multi* m, int rank, int slot) {
  if (!m || rank < 0 || rank >= (int)m->ranks.size()) return nullptr;
  return m->ranks[(size_t)rank].reg->context(slot);
}
int mvr_multi_contexts(mvr_multi* m, int rank) {
  if (!m || rank < 0 || rank >= (int)m->ranks.size()) return 0;
  return m->ranks[(size_t)rank].reg->streams();
}

void mvr_multi_pair_range(int rank, int n_ranks, int n_pairs, int* pair_begin, int* pair_end) {
  int a = 0, b = 0;
  if (n_ranks > 0 && rank >= 0 && rank < n_ranks && n_pairs >= 0) pair_block(rank, n_ranks, n_pairs, &a, &b);
  if (pair_begin) *pair_begin = a;
  if (pair_end) *pair_end = b;
}

int mvr_multi_upload(mvr_multi* m, const mvr_view* views, int n_views) {
  if (!m || n_views < 0 || (n_views && !views)) return MVR_ERR_BAD_ARG;
  const int world = (int)m->ranks.size();
  for (int k = 0; k < world; ++k) {
    Rank& r = m->ranks[(size_t)k];
    free_resident(r);
    r.resident.assign((size_t)n_views, nullptr);
    r.resident_n.assign((size_t)n_views, 0);
    int p0, p1;
    pair_block(k, world, n_views, &p0, &p1);
    cudaSetDevice(r.device);
    for (int p = p0; p < p1; ++p)
      for (int e = 0; e < 2; ++e) {
        const int i = (p + e) % n_views;
        if (r.resident[(size_t)i] || views[i].n == 0) continue;
        if (views[i].on_device) return fail(m, MVR_ERR_BAD_ARG, "mvr_multi_upload takes host views");
        void* d = nullptr;
        if (cudaMalloc(&d, views[i].n * 16) != cudaSuccess) return fail(m, MVR_ERR_ALLOC, "resident view");
        if (cudaMemcpy(d, views[i].xyzw, views[i].n * 16, cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(d); return fail(m, MVR_ERR_CUDA, "resident view copy"); }
        r.resident[(size_t)i] = d;
        r.resident_n[(size_t)i] = views[i].n;
      }
  }
  m->resident_views = n_views;
  return MVR_OK;
}

int mvr_register_turntable_multi(mvr_multi* m, const mvr_view* views, int n_views, const mvr_turntable_params* prm, int use_resident,
                                 float* poses, mvr_pair_report* reports, mvr_pair_record* records, double* device_ms) {
  if (!m || !prm || n_views < 0 || (n_views && !views)) return MVR_ERR_BAD_ARG;
  if (prm->mode != MVR_REGISTER_RING_PAIRS) return fail(m, MVR_ERR_BAD_ARG, "only the ring-pair mode shards over GPUs (the accumulative modes grow one model)");
  if (use_resident && m->resident_views != n_views) return fail(m, MVR_ERR_NO_INPUT, "mvr_multi_upload has not been called for these views");
  const int V = n_views, world = (int)m->ranks.size();
  if (!use_resident)
    for (int i = 0; i < V; ++i) if (views[i].on_device) return fail(m, MVR_ERR_BAD_ARG, "views must be host buffers (each GPU uploads the ones it needs)");
  if (V < 2) {
    if (poses) for (int i = 0; i < V; ++i) for (int k = 0; k < 16; ++k) poses[16 * i + k] = (k % 5 == 0) ? 1.f : 0.f;
    return MVR_OK;
  }
  // one host thread per GPU (rank 0 runs on the calling thread)
  std::vector<std::thread> th;
  for (int k = 1; k < world; ++k) th.emplace_back(rank_work, m, k, views, V, prm, use_resident != 0);
  rank_work(m, 0, views, V, prm, use_resident != 0);
  for (std::thread& t : th) t.join();
  for (int k = 0; k < world; ++k) {
    if (device_ms) device_ms[k] = m->ranks[(size_t)k].ms;
    if (m->ranks[(size_t)k].status != MVR_OK) return fail(m, m->ranks[(size_t)k].status, "rank " + std::to_string(k) + ": " + m->ranks[(size_t)k].err);
  }
  // the gathered records, identical on every rank: take rank 0's copy
  size_t block = 0;
  for (int q = 0; q < world; ++q) { int a, b; pair_block(q, world, V, &a, &b); block = std::max(block, (size_t)(b - a)); }
  std::vector<mvr_pair_record> all((size_t)V);
  for (int q = 0; q < world; ++q) {
    int a, b;
    pair_block(q, world, V, &a, &b);
    for (int p = a; p < b; ++p) all[(size_t)p] = m->ranks[0].h_recv[(size_t)q * block + (size_t)(p - a)];
  }
  for (int p = 0; p < V; ++p) if (all[(size_t)p].status < 0) return fail(m, MVR_ERR_CUDA, "a rank failed before the exchange");
  if (records) std::memcpy(records, all.data(), (size_t)V * sizeof(mvr_pair_record));
  if (reports)
    for (int p = 0; p < V; ++p) {
      mvr_pair_report& o = reports[p];
      std::memset(&o, 0, sizeof(o));
      o.source_view = (p + 1) % V; o.target_view = p; o.status = all[(size_t)p].status; o.iterations = all[(size_t)p].iterations;
      o.n_correspondences = all[(size_t)p].n_correspondences; o.mse = all[(size_t)p].mse; o.fitness = -1; o.nn_queries = all[(size_t)p].nn_queries;
      std::memcpy(o.pose, all[(size_t)p].pose, sizeof(o.pose));
    }
  // host loop closure on the gathered records
  std::vector<Matrix4d> rel((size_t)V), X;
  std::vector<double> w((size_t)V);
  for (int p = 0; p < V; ++p) {
    Matrix4f f;
    std::memcpy(f.m, all[(size_t)p].pose, sizeof(f.m));
    rel[(size_t)p] = toDouble(f);
    w[(size_t)p] = all[(size_t)p].status == MVR_OK ? (double)all[(size_t)p].n_correspondences : 0.0;
  }
  const double radius = m->ranks[0].reg->lastTargetRadius();
  const int rc = ringClose(rel, w, prm->loop_closure != 0, prm->lum_iterations > 0 ? prm->lum_iterations : 16, prm->pivot, radius, X);
  if (rc) return fail(m, rc, "loop closure failed");
  Matrix4d base = identity4d();
  if (views[0].init_pose) std::memcpy(base.m, views[0].init_pose, sizeof(base.m));
  if (poses)
    for (int i = 0; i < V; ++i) {
      const Matrix4f f = toFloat(multiply(base, X[(size_t)i]));
      std::memcpy(poses + 16 * i, f.m, sizeof(f.m));
    }
  return MVR_OK;
}

int mvr_multi_set_angle_search(mvr_multi* m, const mvr_angle_search* s) {
  if (!m) return MVR_ERR_BAD_ARG;
  for (size_t k = 0; k < m->ranks.size(); ++k) {
    const int rc = m->ranks[k].reg->setAngleSearch(s);
    if (rc) return fail(m, rc, m->ranks[k].reg->lastError());
  }
  return MVR_OK;
}

int mvr_multi_get_angle_search(mvr_multi* m, mvr_angle_pick* out, int max_records, int* count) {
  if (!m || !count) return MVR_ERR_BAD_ARG;
  std::vector<mvr_angle_pick> all;   // rank k holds the records of its block of pairs: rank order is pair order
  for (const Rank& r : m->ranks) all.insert(all.end(), r.reg->angleLog().begin(), r.reg->angleLog().end());
  int n = (int)all.size();
  if (out) {
    n = std::min(n, std::max(max_records, 0));
    if (n) std::memcpy(out, all.data(), (size_t)n * sizeof(mvr_angle_pick));
  }
  *count = n;
  return MVR_OK;
}

}  // extern "C"
