// C ABI of the engine (include/afesp_gpu.h): argument checking, host<->device copies, status codes.
#include <dlfcn.h>

#include <cmath>
#include <cstring>
#include <functional>
#include <set>

#include "../../include/afesp_gpu.h"
#include "ccsd.cuh"

using namespace afesp;

namespace {

// ---- NCCL through dlopen: the library must load on hosts without NCCL and must share the copy a host process
//      (e.g. a torchrun launcher) has already loaded.
struct NcclId { char internal[128]; };
typedef void* NcclComm;
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(NcclComm*, int, NcclId, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
  int (*CommDestroy)(NcclComm) = nullptr;
  int (*Broadcast)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, NcclComm, cudaStream_t) = nullptr;
  int (*Send)(const void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool load(std::string& err) {
    if (lib) return true;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
    if (!lib) { err = "NCCL not found (dlopen libnccl.so.2)"; return false; }
    GetUniqueId = (int (*)(NcclId*))dlsym(lib, "ncclGetUniqueId");
    CommInitRank = (int (*)(NcclComm*, int, NcclId, int))dlsym(lib, "ncclCommInitRank");
    AllReduce = (int (*)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t))dlsym(lib, "ncclAllReduce");
    CommDestroy = (int (*)(NcclComm))dlsym(lib, "ncclCommDestroy");
    GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
    Broadcast = (int (*)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t))dlsym(lib, "ncclBroadcast");
    AllGather = (int (*)(const void*, void*, size_t, int, NcclComm, cudaStream_t))dlsym(lib, "ncclAllGather");
    Send = (int (*)(const void*, size_t, int, int, NcclComm, cudaStream_t))dlsym(lib, "ncclSend");
    Recv = (int (*)(void*, size_t, int, int, NcclComm, cudaStream_t))dlsym(lib, "ncclRecv");
    GroupStart = (int (*)())dlsym(lib, "ncclGroupStart");
    GroupEnd = (int (*)())dlsym(lib, "ncclGroupEnd");
    if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy || !Broadcast || !Send || !Recv || !GroupStart ||
        !GroupEnd) {
      err = "NCCL symbols missing";
      return false;
    }
    return true;
  }
};
NcclApi g_nccl;
constexpr int kNcclDouble = 8;  // ncclFloat64
constexpr int kNcclSum = 0;
// adapters installed into Engine::dist (tensor.cuh): doubles only
int dist_group_start() { return g_nccl.GroupStart(); }
int dist_group_end() { return g_nccl.GroupEnd(); }
int dist_bcast(const void* s, void* r, size_t n, int root, void* comm, cudaStream_t st) {
  return g_nccl.Broadcast(s, r, n, kNcclDouble, root, comm, st);
}
int dist_allgather(const void* s, void* r, size_t n, void* comm, cudaStream_t st) {
  return g_nccl.AllGather ? g_nccl.AllGather(s, r, n, kNcclDouble, comm, st) : -1;
}
int dist_send(const void* b, size_t n, int peer, void* comm, cudaStream_t st) {
  return g_nccl.Send(b, n, kNcclDouble, peer, comm, st);
}
int dist_recv(void* b, size_t n, int peer, void* comm, cudaStream_t st) {
  return g_nccl.Recv(b, n, kNcclDouble, peer, comm, st);
}

struct Handle {
  int device = 0;
  CCState s;
  DBuf eri_ao, coeff;
  int n_ao = 0;
  int frozen_core = 0;   // option "frozen_core": read by mp2_energy and ccsd_init (which copies it into the CC state)
  std::string err;
  int rank = 0, nranks = 1;
  NcclComm comm = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t tm0 = nullptr, tm1 = nullptr;  // afesp_gpu_timer
  double last_ms = 0.0;
  long long launches0 = 0;
  double flops0 = 0.0;
};

std::string g_open_error;
// One handle per device and process: the caching allocator and the GEMM workspace are per device and rely on
// stream-ordered reuse, i.e. on a single stream per device.
std::set<int>& g_open_devices = *new std::set<int>;

// Cached free blocks go back to the driver only when they add up to a sizeable part of the HBM (large shapes, where
// the next stage needs the room); small runs keep them so repeated init/finalize cycles never touch cudaMalloc.
void trim_if_large(size_t threshold = (size_t)48 << 30) {
  if (device_cached_bytes() > threshold) device_trim();
}

struct StageTimer {  // device time of one API stage, on the stream the kernels run on
  Handle* h;
  explicit StageTimer(Handle* hh) : h(hh) { cudaEventRecord(h->ev0, h->s.eng.stream); }
  void stop() {
    cudaEventRecord(h->ev1, h->s.eng.stream);
    cudaEventSynchronize(h->ev1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    h->last_ms = ms;
  }
};

template <class F>
int guarded(afesp_handle hv, F&& f) {
  Handle* h = static_cast<Handle*>(hv);
  if (!h) return 1;
  try {
    AFESP_CUDA_CHECK(cudaSetDevice(h->device));
    f(*h);
    return 0;
  } catch (const Error& e) {
    h->err = e.what();
    return e.code;
  } catch (const std::exception& e) {
    h->err = e.what();
    return 1;
  }
}

void assemble_finalize_checks(Handle& h) {
  AFESP_REQUIRE(h.s.t2.size() > 0, "CCSD state not initialised (call afesp_gpu_ccsd_init first)");
}

// Register-resident DMMA loop: every warp keeps 8 independent accumulator pairs in flight.
__global__ void k_dmma_peak(double* out, int iters) {
  double c[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) c[i] = 0.0;
  double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                   : "+d"(c[2 * i]), "+d"(c[2 * i + 1])
                   : "d"(a), "d"(b));
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += c[i];
  if (s == 12345.678) out[0] = s;  // keep the loop alive
}

}  // namespace

extern "C" {
#pragma GCC visibility push(default)

int afesp_gpu_open(int device, afesp_handle* out) {
  if (!out) return 1;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_open_error = std::string("afesp_gpu_open: no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback";
    return 2;
  }
  if (device < 0 || device >= ndev) { g_open_error = "afesp_gpu_open: device index out of range"; return 1; }
  cudaDeviceProp prop;
  cudaSetDevice(device);
  cudaGetDeviceProperties(&prop, device);
  if (prop.major < 10) {
    g_open_error = "afesp_gpu_open: kernels are built for sm_100a (Blackwell) only; found compute capability " +
                   std::to_string(prop.major) + "." + std::to_string(prop.minor);
    return 2;
  }
  if (g_open_devices.count(device)) {
    g_open_error = "afesp_gpu_open: device " + std::to_string(device) + " already has an open handle in this process (one "
                   "handle per device: close it first)";
    return 1;
  }
  Handle* h = new Handle();
  h->device = device;
  if (cudaStreamCreate(&h->s.eng.stream) != cudaSuccess || cudaEventCreate(&h->ev0) != cudaSuccess ||
      cudaEventCreate(&h->ev1) != cudaSuccess) {
    g_open_error = "afesp_gpu_open: stream/event creation failed";
    delete h;
    return 2;
  }
  if (gemm_tma_scope_get() > 0) {
    // once per process: the TMA-staged kernel must reproduce the cp.async kernel on this device, else it is switched off
    try {
      gemm_tma_selftest(h->s.eng.stream);
    } catch (const std::exception& e) {
      g_open_error = std::string("afesp_gpu_open: TMA self-test could not run: ") + e.what();
      cudaEventDestroy(h->ev0); cudaEventDestroy(h->ev1);
      cudaStream_t st = h->s.eng.stream;
      delete h;
      cudaStreamDestroy(st);
      return 2;
    }
  }
  h->launches0 = g_launch_count;
  h->flops0 = g_gemm_flops;
  g_open_devices.insert(device);
  *out = h;
  return 0;
}

int afesp_gpu_tma_status(afesp_handle hv, int* scope, int* selftest) {
  return guarded(hv, [&](Handle&) {
    if (scope) *scope = gemm_tma_scope_get();
    if (selftest) *selftest = gemm_tma_selftest_state();
  });
}

int afesp_gpu_close(afesp_handle hv) {
  Handle* h = static_cast<Handle*>(hv);
  if (!h) return 1;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->tm0) cudaEventDestroy(h->tm0);
  if (h->tm1) cudaEventDestroy(h->tm1);
  cudaStream_t st = h->s.eng.stream;
  g_open_devices.erase(h->device);
  delete h;
  if (st) cudaStreamDestroy(st);
  device_trim();
  return 0;
}

const char* afesp_gpu_last_error(afesp_handle hv) {
  Handle* h = static_cast<Handle*>(hv);
  return h ? h->err.c_str() : g_open_error.c_str();
}

int afesp_gpu_set_option(afesp_handle hv, const char* key, double value) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(key != nullptr, "set_option: null key");
    std::string k(key);
    Options& o = h.s.opt;
    if (k == "q1_transposed_foo") o.q1_transposed_foo = value != 0.0;
    else if (k == "q3a_truncated_e") o.q3a_truncated_e = value != 0.0;
    else if (k == "q3b_stale_intermediates") o.q3b_stale_intermediates = value != 0.0;
    else if (k == "triples_ijk_symmetry") o.triples_ijk_symmetry = value != 0.0;
    else if (k == "triples_batch_bytes") o.triples_batch_bytes = (long long)value;
    else if (k == "finalize_keep_ccsd") o.finalize_keep_ccsd = value != 0.0;
    else if (k == "spinorb_symmetry_tol") o.spinorb_symmetry_tol = value;
    else if (k == "frozen_core") {
      AFESP_REQUIRE(value >= 0.0 && value == std::floor(value) && value < 1e9,
                    "set_option: frozen_core must be a non-negative integer (number of frozen doubly occupied orbitals)");
      h.frozen_core = (int)value;
    }
    else if (k == "gemm_timing") gemm_timing_enable(value != 0.0);
    else if (k == "gemm_force_config") gemm_force_config((int)value);
    else if (k == "gemm_tma_edge") gemm_tma_edge((int)value);
    else if (k == "gemm_use_tma") {
      // 0 off, 1 the gathered (T) batches only, 2 every aligned GEMM the 64x64 tile is chosen for.  Switching it on runs
      // the consistency check against the cp.async kernel first (once per process); if that fails the path stays off.
      if ((int)value > 0) gemm_tma_selftest(h.s.eng.stream);
      gemm_tma_scope((int)value);
    }
    else if (k == "dist_allgather") h.s.eng.dist.use_allgather = value < 0.0 ? -1 : (value != 0.0 ? 1 : 0);
    else if (k == "dist_overlap_chunks") h.s.eng.dist.overlap_chunks = std::max(1, std::min(8, (int)value));
    else if (k == "dist_min_flops") h.s.eng.dist.min_flops = value;   // GEMMs below this stay replicated
    else if (k == "dist_ccsd") {   // 0: replicate CCSD / AO->MO, shard only (T)
      AFESP_REQUIRE(!(h.s.vpm_sharded && !h.s.finalized && value == 0.0),
                    "set_option: dist_ccsd cannot be switched off while the ladder integrals of the current CCSD state are "
                    "sharded (call afesp_gpu_ccsd_init again afterwards)");
      h.s.eng.dist.enabled = value != 0.0;
    }
    else throw Error(1, "set_option: unknown key " + k);
  });
}

int afesp_gpu_counters(afesp_handle hv, long long* launches, double* gemm_flops) {
  return guarded(hv, [&](Handle& h) {
    if (launches) *launches = g_launch_count - h.launches0;
    if (gemm_flops) *gemm_flops = g_gemm_flops - h.flops0;
  });
}

int afesp_gpu_ao2mo(afesp_handle hv, int n, const double* eri_ao, const double* coeff, double* eri_mo) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(n > 0, "ao2mo: nbasis must be positive");
    const long long np = npacked_of(n);
    cudaStream_t st = h.s.eng.stream;
    if (eri_ao || coeff) {
      AFESP_REQUIRE(eri_ao && coeff, "ao2mo: pass both eri_ao and coeff, or neither to reuse the resident copies");
      if ((long long)h.eri_ao.n != np) h.eri_ao.alloc((size_t)np);
      if ((long long)h.coeff.n != (long long)n * n) h.coeff.alloc((size_t)n * n);
      AFESP_CUDA_CHECK(cudaMemcpyAsync(h.eri_ao.p, eri_ao, np * 8, cudaMemcpyHostToDevice, st));
      AFESP_CUDA_CHECK(cudaMemcpyAsync(h.coeff.p, coeff, (size_t)n * n * 8, cudaMemcpyHostToDevice, st));
      h.n_ao = n;
    } else {
      AFESP_REQUIRE(h.n_ao == n && h.eri_ao.p, "ao2mo: no resident AO integrals for this nbasis");
    }
    if ((long long)h.s.eri_mo.n != np) h.s.eri_mo.alloc((size_t)np);
    h.s.n = n;
    StageTimer tm(&h);
    ao2mo_packed(h.s.eng, n, h.eri_ao.p, h.coeff.p, h.s.eri_mo.p);
    tm.stop();
    trim_if_large();  // the npair^2 half-transformed matrix goes back to the driver when it is big
    if (eri_mo) {
      AFESP_CUDA_CHECK(cudaMemcpyAsync(eri_mo, h.s.eri_mo.p, np * 8, cudaMemcpyDeviceToHost, st));
      AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
    }
  });
}

int afesp_gpu_synth_eri_ao(afesp_handle hv, int n, int naux, const double* factors, const double* coeff) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(n > 0 && naux > 0 && factors && coeff, "synth_eri_ao: bad arguments");
    const long long np = npacked_of(n), npair = npair_of(n);
    cudaStream_t st = h.s.eng.stream;
    DBuf B((size_t)npair * naux);
    AFESP_CUDA_CHECK(cudaMemcpyAsync(B.p, factors, (size_t)npair * naux * 8, cudaMemcpyHostToDevice, st));
    if ((long long)h.eri_ao.n != np) h.eri_ao.alloc((size_t)np);
    if ((long long)h.coeff.n != (long long)n * n) h.coeff.alloc((size_t)n * n);
    AFESP_CUDA_CHECK(cudaMemcpyAsync(h.coeff.p, coeff, (size_t)n * n * 8, cudaMemcpyHostToDevice, st));
    StageTimer tm(&h);
    synth_eri_from_factors(h.s.eng, n, naux, B.p, h.eri_ao.p);
    tm.stop();
    h.n_ao = n;
    trim_if_large();
  });
}

int afesp_gpu_get_eri_mo(afesp_handle hv, double* eri_mo) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(eri_mo && h.s.eri_mo.p, "get_eri_mo: no MO integrals on the device");
    AFESP_CUDA_CHECK(cudaMemcpy(eri_mo, h.s.eri_mo.p, h.s.eri_mo.n * 8, cudaMemcpyDeviceToHost));
  });
}

int afesp_gpu_release(afesp_handle hv, const char* what) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(what != nullptr, "release: null argument");
    std::string w(what);
    AFESP_CUDA_CHECK(cudaStreamSynchronize(h.s.eng.stream));
    if (w == "eri_ao") { h.eri_ao.release(); h.coeff.release(); h.n_ao = 0; }
    else if (w == "eri_mo") h.s.eri_mo.release();
    else if (w == "scratch") h.s.eng.pool.clear();
    else throw Error(1, "release: unknown object " + w);
  });
}

static void allreduce_sum(Handle& h, double* vals, int n);
int afesp_gpu_set_eri_mo(afesp_handle hv, int n, const double* eri_mo) {
  return guarded(hv, [&](Handle& h) {
    Dist& d = h.s.eng.dist;
    const bool collective = d.nranks > 1 && d.comm != nullptr;
    AFESP_REQUIRE(n > 0 && (eri_mo || collective), "set_eri_mo: bad arguments");
    const long long np = npacked_of(n);
    cudaStream_t st = h.s.eng.stream;
    if ((long long)h.s.eri_mo.n != np) h.s.eri_mo.alloc((size_t)np);
    if (!collective) {
      AFESP_CUDA_CHECK(cudaMemcpyAsync(h.s.eri_mo.p, eri_mo, np * 8, cudaMemcpyHostToDevice, st));
      AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
      h.s.n = n;
      return;
    }
    // Collective.  How many ranks hold the host array?  (one tiny allreduce)
    double have[1] = {eri_mo ? 1.0 : 0.0};
    allreduce_sum(h, have, 1);
    const int nhave = (int)(have[0] + 0.5);
    if (nhave == d.nranks) {
      // every rank can read the array (replicated host copies, or one copy in shared memory): each uploads 1/nranks of
      // it over ITS OWN PCIe link, then the shares are exchanged over NVLink
      std::vector<std::pair<long long, long long>> ranges(d.nranks);
      for (int r = 0; r < d.nranks; ++r) ranges[r] = {np * r / d.nranks, np * (r + 1) / d.nranks};
      const long long lo = ranges[d.rank].first, cnt = ranges[d.rank].second - lo;
      if (cnt > 0) AFESP_CUDA_CHECK(cudaMemcpyAsync(h.s.eri_mo.p + lo, eri_mo + lo, cnt * 8, cudaMemcpyHostToDevice, st));
      d.exchange(h.s.eri_mo.p, ranges, st);
    } else {
      // one host copy per node: rank 0 uploads, the other ranks receive it over NVLink
      AFESP_REQUIRE(nhave >= 1 && (d.rank != 0 || eri_mo), "set_eri_mo: rank 0 must pass the host array");
      if (d.rank == 0) AFESP_CUDA_CHECK(cudaMemcpyAsync(h.s.eri_mo.p, eri_mo, np * 8, cudaMemcpyHostToDevice, st));
      AFESP_REQUIRE(d.group_start() == 0, "ncclGroupStart failed");
      AFESP_REQUIRE(d.bcast(h.s.eri_mo.p, h.s.eri_mo.p, (size_t)np, 0, d.comm, st) == 0, "ncclBroadcast failed");
      AFESP_REQUIRE(d.group_end() == 0, "ncclGroupEnd failed");
    }
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
    h.s.n = n;
  });
}

static void upload_eps(Handle& h, const double* eps) {
  const int n = h.s.n;
  AFESP_REQUIRE(eps != nullptr, "eps must not be null");
  if ((int)h.s.eps.n != n) h.s.eps.alloc(n);
  h.s.eps_host.assign(eps, eps + n);
  AFESP_CUDA_CHECK(cudaMemcpyAsync(h.s.eps.p, eps, n * 8, cudaMemcpyHostToDevice, h.s.eng.stream));
  AFESP_CUDA_CHECK(cudaStreamSynchronize(h.s.eng.stream));
}

int afesp_gpu_mp2_energy(afesp_handle hv, int nocc, const double* eps, double* e_mp2) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(h.s.n > 0 && h.s.eri_mo.p, "mp2_energy: no MO integrals on the device");
    AFESP_REQUIRE(nocc > 0 && nocc < h.s.n && e_mp2, "mp2_energy: bad arguments");
    AFESP_REQUIRE(h.frozen_core < nocc, "mp2_energy: frozen_core (" + std::to_string(h.frozen_core) +
                                            ") must be smaller than nocc (" + std::to_string(nocc) + ")");
    upload_eps(h, eps);
    if (h.s.red_out.n < 16) h.s.red_out.alloc(16);
    StageTimer tm(&h);
    mp2_energy(h.s.eng, h.s.n, nocc, h.frozen_core, h.s.eri_mo.p, h.s.eps.p, h.s.red_out.p);
    tm.stop();
    AFESP_CUDA_CHECK(cudaMemcpy(e_mp2, h.s.red_out.p, 8, cudaMemcpyDeviceToHost));
  });
}

int afesp_gpu_ccsd_init(afesp_handle hv, int nocc, int restricted, const double* eps, int diis_n, double* e_mp1,
                        double* rmst2) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(h.s.n > 0 && h.s.eri_mo.p, "ccsd_init: no MO integrals on the device");
    AFESP_REQUIRE(nocc > 0 && nocc < h.s.n, "ccsd_init: bad nocc");
    AFESP_REQUIRE(h.frozen_core < nocc, "ccsd_init: frozen_core (" + std::to_string(h.frozen_core) +
                                            ") must be smaller than nocc (" + std::to_string(nocc) + ")");
    upload_eps(h, eps);
    h.s.nocc_spatial = nocc;
    h.s.nfrozen = h.frozen_core;
    {
      Trace tr(h.s.eng.stream);
      h.s.T.clear();
      tr.lap(0);
      const char* names[] = {"init free old"};
      tr.report(names, 1);
    }
    StageTimer tm(&h);
    if (restricted) ccsd_spatial_init(h.s, diis_n);
    else ccsd_spinorb_init(h.s, diis_n);
    cc_update_energy(h.s);  // the "MP1" line (src/ccsd.f90:325-331)
    tm.stop();
    if (e_mp1) *e_mp1 = h.s.energy;
    if (rmst2) *rmst2 = h.s.rms;
  });
}

int afesp_gpu_ccsd_init_info(afesp_handle hv, double info[4]) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(info != nullptr, "ccsd_init_info: null output");
    info[0] = h.s.sym_err; info[1] = h.s.ms_slices * 1e-3; info[2] = h.s.ms_symcheck * 1e-3; info[3] = 0.0;
  });
}

int afesp_gpu_ccsd_iterate(afesp_handle hv, double* e_cc, double* rmst2) {
  return guarded(hv, [&](Handle& h) {
    assemble_finalize_checks(h);
    AFESP_REQUIRE(!h.s.finalized, "ccsd_iterate: state already finalised");
    StageTimer tm(&h);
    cc_diis_stash(h.s);
    if (h.s.restricted) ccsd_spatial_iterate(h.s);
    else ccsd_spinorb_iterate(h.s);
    cc_update_energy(h.s);
    tm.stop();
    if (e_cc) *e_cc = h.s.energy;
    if (rmst2) *rmst2 = h.s.rms;
  });
}

int afesp_gpu_ccsd_diis(afesp_handle hv) {
  return guarded(hv, [&](Handle& h) {
    assemble_finalize_checks(h);
    AFESP_REQUIRE(!h.s.finalized, "ccsd_diis: state already finalised");
    StageTimer tm(&h);
    cc_diis_update(h.s);
    tm.stop();
  });
}

int afesp_gpu_ccsd_finalize(afesp_handle hv, int want_cr, double* t1_diag, double* t1, double* t2) {
  return guarded(hv, [&](Handle& h) {
    assemble_finalize_checks(h);
    CCState& s = h.s;
    StageTimer tm(&h);
    if (t1_diag) {
      // sqrt(sum t1^2)/sqrt(nel), nel = number of correlated electrons (src/ccsd.f90:372)
      *t1_diag = std::sqrt(cc_t1_norm2(s)) / std::sqrt((double)(2 * (s.nocc_spatial - s.nfrozen)));
    }
    if (want_cr && !s.have_cr) {
      AFESP_REQUIRE(s.restricted, "CR intermediates exist only in the spin-free formulation");
      ccsd_spatial_cr_intermediates(s);
    }
    // release what the (T) stage does not need (the reference's cc_int goes out of scope, src/ccsd.f90:386-392)
    if (s.opt.finalize_keep_ccsd && !(want_cr && s.have_cr)) {
      // benchmark loops: keep the DIIS history and the intermediates so that ccsd_iterate can be called again.  (Not after
      // the CR intermediates were built: that step consumes V+/-, I_oooo, ... -- the state is then finalised as usual.)
      tm.stop();
      if (t1) AFESP_CUDA_CHECK(cudaMemcpy(t1, s.t1.p(), s.t1.size() * 8, cudaMemcpyDeviceToHost));
      if (t2) AFESP_CUDA_CHECK(cudaMemcpy(t2, s.t2.p(), s.t2.size() * 8, cudaMemcpyDeviceToHost));
      return;
    }
    s.diis = CCDiis();
    for (const char* nm : {"v_vvvv", "V_plus", "V_minus", "W_efab", "vvvv", "ovvv", "I_oooo", "I_ovov", "I_voov", "I_ooov_p",
                           "x_voov", "c_oovv", "A_oovv", "W_ijmn", "W_ovvo", "tau", "tau_tilde"})
      s.drop(nm);
    s.t1n.free(); s.t2n.free(); s.t2_old.free();
    trim_if_large();
    s.finalized = true;
    tm.stop();
    if (t1) AFESP_CUDA_CHECK(cudaMemcpy(t1, s.t1.p(), s.t1.size() * 8, cudaMemcpyDeviceToHost));
    if (t2) AFESP_CUDA_CHECK(cudaMemcpy(t2, s.t2.p(), s.t2.size() * 8, cudaMemcpyDeviceToHost));
  });
}

static void allreduce_sum(Handle& h, double* vals, int n) {
  if (!h.comm || h.nranks == 1) return;
  if (h.s.red_out.n < 16) h.s.red_out.alloc(16);
  AFESP_REQUIRE(n <= 16, "allreduce: too many values");
  cudaStream_t st = h.s.eng.stream;
  AFESP_CUDA_CHECK(cudaMemcpyAsync(h.s.red_out.p, vals, n * 8, cudaMemcpyHostToDevice, st));
  int rc = g_nccl.AllReduce(h.s.red_out.p, h.s.red_out.p, (size_t)n, kNcclDouble, kNcclSum, h.comm, st);
  if (rc != 0) throw Error(4, std::string("ncclAllReduce failed: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"));
  AFESP_CUDA_CHECK(cudaMemcpyAsync(vals, h.s.red_out.p, n * 8, cudaMemcpyDeviceToHost, st));
  AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
}

int afesp_gpu_ccsd_t_spatial(afesp_handle hv, int paren, int renorm, int comp_renorm, double sums[6],
                             double* denominator_constant) {
  return guarded(hv, [&](Handle& h) {
    assemble_finalize_checks(h);
    AFESP_REQUIRE(sums != nullptr, "ccsd_t: sums must not be null");
    StageTimer tm(&h);
    triples_spatial(h.s, paren != 0, renorm != 0, comp_renorm != 0, h.rank, h.nranks, sums);
    allreduce_sum(h, sums, 6);
    double c = 0.0;
    if (renorm || comp_renorm) c = triples_denominator_constant(h.s);
    tm.stop();
    if (denominator_constant) *denominator_constant = c;
  });
}

int afesp_gpu_ccsd_t_spinorb(afesp_handle hv, double* e_T) {
  return guarded(hv, [&](Handle& h) {
    assemble_finalize_checks(h);
    AFESP_REQUIRE(e_T != nullptr, "ccsd_t: e_T must not be null");
    StageTimer tm(&h);
    triples_spinorb(h.s, h.rank, h.nranks, e_T);
    allreduce_sum(h, e_T, 1);
    tm.stop();
  });
}

int afesp_gpu_comm_unique_id(char id[128]) {
  std::string err;
  if (!id || !g_nccl.load(err)) { g_open_error = err; return 4; }
  NcclId nid;
  if (g_nccl.GetUniqueId(&nid) != 0) { g_open_error = "ncclGetUniqueId failed"; return 4; }
  std::memcpy(id, nid.internal, 128);
  return 0;
}

int afesp_gpu_comm_init(afesp_handle hv, int rank, int nranks, const char id[128]) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks && id, "comm_init: bad arguments");
    std::string err;
    if (!g_nccl.load(err)) throw Error(4, err);
    NcclId nid;
    std::memcpy(nid.internal, id, 128);
    int rc = g_nccl.CommInitRank(&h.comm, nranks, nid, rank);
    if (rc != 0) throw Error(4, std::string("ncclCommInitRank failed: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"));
    h.rank = rank; h.nranks = nranks;
    Dist& d = h.s.eng.dist;
    d.rank = rank; d.nranks = nranks; d.comm = h.comm;
    d.group_start = dist_group_start; d.group_end = dist_group_end;
    d.bcast = dist_bcast; d.send = dist_send; d.recv = dist_recv;
    d.allgather = g_nccl.AllGather ? dist_allgather : nullptr;
  });
}

int afesp_gpu_host_register(void* ptr, long long bytes) {
  if (!ptr || bytes <= 0) return 1;
  const cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault);
  if (e != cudaSuccess) { cudaGetLastError(); return 2; }   // not sticky: the caller falls back to pageable transfers
  return 0;
}

int afesp_gpu_host_unregister(void* ptr) {
  if (!ptr) return 1;
  const cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess) { cudaGetLastError(); return 2; }
  return 0;
}

int afesp_gpu_set_partition(afesp_handle hv, int rank, int nranks) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "set_partition: bad arguments");
    AFESP_REQUIRE(h.comm == nullptr, "set_partition: a communicator is attached");
    h.rank = rank; h.nranks = nranks;
  });
}

int afesp_gpu_triples_partition(int nocc_active, int symmetric, int strict, int nranks, long long* counts) {
  if (nocc_active < 0 || nranks < 1 || !counts) return 1;
  triples_partition_counts(nocc_active, symmetric != 0, strict != 0, nranks, counts);
  return 0;
}

int afesp_gpu_column_partition(long long ncols, int nranks, int granularity, long long* lo, long long* hi) {
  if (ncols < 0 || nranks < 1 || granularity < 1 || !lo || !hi) return 1;
  Dist d;
  d.nranks = nranks;
  for (int r = 0; r < nranks; ++r) d.col_range(ncols, r, &lo[r], &hi[r], granularity);
  return 0;
}

int afesp_gpu_dgemm_wrapper(afesp_handle hv, char ta, char tb, int M, int N, int K, const double* A, const double* B,
                            double* C, double alpha, double beta) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(M >= 0 && N >= 0 && K >= 0 && C, "dgemm_wrapper: bad arguments");
    const bool tA = (ta == 'T' || ta == 't'), tB = (tb == 'T' || tb == 't');
    const long long lda = tA ? K : M, ldb = tB ? N : K;  // src/linalg.fpp:69-79
    const size_t na = (size_t)M * K, nb = (size_t)K * N, nc = (size_t)M * N;
    cudaStream_t st = h.s.eng.stream;
    DBuf dA(std::max<size_t>(na, 1)), dB(std::max<size_t>(nb, 1)), dC(std::max<size_t>(nc, 1));
    if (na) AFESP_CUDA_CHECK(cudaMemcpyAsync(dA.p, A, na * 8, cudaMemcpyHostToDevice, st));
    if (nb) AFESP_CUDA_CHECK(cudaMemcpyAsync(dB.p, B, nb * 8, cudaMemcpyHostToDevice, st));
    if (nc && beta != 0.0) AFESP_CUDA_CHECK(cudaMemcpyAsync(dC.p, C, nc * 8, cudaMemcpyHostToDevice, st));
    StageTimer tm(&h);
    dgemm(st, ta, tb, M, N, K, alpha, dA.p, std::max<long long>(lda, 1), dB.p, std::max<long long>(ldb, 1), beta, dC.p,
          std::max(M, 1));
    tm.stop();
    if (nc) AFESP_CUDA_CHECK(cudaMemcpyAsync(C, dC.p, nc * 8, cudaMemcpyDeviceToHost, st));
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
  });
}

int afesp_gpu_omp_reshape(afesp_handle hv, double* out_arr, const double* in_arr, const int in_dims[4],
                          const char arr_order[4], int has_beta, double beta) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(out_arr && in_arr && in_dims && arr_order, "omp_reshape: null argument");
    int perm[4], dims[4];
    size_t total = 1;
    for (int d = 0; d < 4; ++d) {
      AFESP_REQUIRE(arr_order[d] >= '1' && arr_order[d] <= '4', "omp_reshape: arr_order must be a permutation of 1234");
      perm[d] = arr_order[d] - '1';  // out axis d takes in axis perm[d]  (src/linalg.fpp:133-147)
      dims[d] = in_dims[d];
      AFESP_REQUIRE(dims[d] >= 0, "omp_reshape: negative extent");
      total *= (size_t)dims[d];
    }
    if (total == 0) return;
    cudaStream_t st = h.s.eng.stream;
    DBuf din(total), dout(total);
    AFESP_CUDA_CHECK(cudaMemcpyAsync(din.p, in_arr, total * 8, cudaMemcpyHostToDevice, st));
    const double b = has_beta ? beta : 0.0;
    if (b != 0.0) AFESP_CUDA_CHECK(cudaMemcpyAsync(dout.p, out_arr, total * 8, cudaMemcpyHostToDevice, st));
    StageTimer tm(&h);
    permute(st, 4, dims, perm, 1.0, din.p, b, dout.p);
    tm.stop();
    AFESP_CUDA_CHECK(cudaMemcpyAsync(out_arr, dout.p, total * 8, cudaMemcpyDeviceToHost, st));
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
  });
}

int afesp_gpu_bench_dgemm(afesp_handle hv, char ta, char tb, int M, int N, int K, double beta, int reps, double* ms) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(M > 0 && N > 0 && K > 0 && reps > 0 && ms, "bench_dgemm: bad arguments");
    const bool tA = (ta == 'T' || ta == 't'), tB = (tb == 'T' || tb == 't');
    const long long lda = tA ? K : M, ldb = tB ? N : K;
    cudaStream_t st = h.s.eng.stream;
    DBuf dA((size_t)M * K), dB((size_t)K * N), dC((size_t)M * N);
    fill(st, (long long)M * K, 1.0 / 3.0, dA.p);
    fill(st, (long long)K * N, 3.0 / 7.0, dB.p);
    dgemm(st, ta, tb, M, N, K, 1.0, dA.p, lda, dB.p, ldb, 0.0, dC.p, M);  // warm-up
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
    StageTimer tm(&h);
    for (int r = 0; r < reps; ++r) dgemm(st, ta, tb, M, N, K, 1.0, dA.p, lda, dB.p, ldb, beta, dC.p, M);
    tm.stop();
    AFESP_CUDA_CHECK(cudaGetLastError());
    *ms = h.last_ms / reps;
  });
}

// HBM-bound kernels at the shape of an (o,o,v,v) amplitude array, device resident, `reps` launches:
//   what = "permute:<order>"  out = permute(in), 4-index order as in omp_reshape, e.g. "permute:3412"   16 B/element
//          "permute_acc:<order>"  out = permute(in) + out                                                24 B/element
//          "divide"   t2 = x / D_ijab, denominators from eps on the fly (src/ccsd.f90:1727)               16 B/element
//          "energy"   E_CC + sum dT2^2 in one pass (src/ccsd.f90:1767-1786)                               24 B/element
//          "axpby"    y = a x + b y                                                                        24 B/element
// Returns milliseconds per launch and the algorithmic bytes per launch.
int afesp_gpu_bench_hbm(afesp_handle hv, const char* what, int o, int v, int reps, double* ms, double* bytes) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(what && o > 0 && v > 0 && reps > 0 && ms && bytes, "bench_hbm: bad arguments");
    const std::string w(what);
    cudaStream_t st = h.s.eng.stream;
    const long long n = (long long)o * o * v * v;
    DBuf a((size_t)n), b((size_t)n), c((size_t)n), eo(o), ev(v), t1((size_t)o * v);
    fill(st, n, 1.0 / 3.0, a.p); fill(st, n, 0.25, b.p); fill(st, n, 0.5, c.p);
    fill(st, o, -1.0, eo.p); fill(st, v, 1.0, ev.p); fill(st, (long long)o * v, 0.01, t1.p);
    if (h.s.red_out.n < 16) h.s.red_out.alloc(16);
    std::function<void()> run;
    double per = 16.0;
    if (w.rfind("permute", 0) == 0) {
      const bool acc = w.rfind("permute_acc", 0) == 0;
      const size_t colon = w.find(':');
      AFESP_REQUIRE(colon != std::string::npos && w.size() == colon + 5, "bench_hbm: permute:<4-digit order>");
      static int perm[4];
      static int dims[4];
      const int in_dims[4] = {o, o, v, v};
      for (int d = 0; d < 4; ++d) {
        perm[d] = w[colon + 1 + d] - '1';
        AFESP_REQUIRE(perm[d] >= 0 && perm[d] < 4, "bench_hbm: bad order");
        dims[d] = in_dims[d];
      }
      per = acc ? 24.0 : 16.0;
      run = [=, &a, &b] { permute(st, 4, dims, perm, 1.0, a.p, acc ? 1.0 : 0.0, b.p); };
    } else if (w == "divide") {
      run = [=, &a, &b, &eo, &ev] { divide_d2(st, b.p, a.p, eo.p, ev.p, o, v); };
    } else if (w == "divide_probe") {
      run = [=, &a, &b, &eo, &ev] { divide_d2_probe(st, b.p, a.p, eo.p, ev.p, o, v); };
    } else if (w == "energy") {
      per = 24.0;
      run = [=, &a, &b, &c, &t1, &h] { cc_energy_restricted(h.s.eng, a.p, b.p, t1.p, c.p, o, v, h.s.red_out.p); };
    } else if (w == "axpby") {
      per = 24.0;
      run = [=, &a, &b] { axpby(st, n, 0.5, a.p, 0.5, b.p); };
    } else {
      throw Error(1, "bench_hbm: unknown kernel " + w);
    }
    run();
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
    StageTimer tm(&h);
    for (int r = 0; r < reps; ++r) run();
    tm.stop();
    AFESP_CUDA_CHECK(cudaGetLastError());
    *ms = h.last_ms / reps;
    *bytes = per * (double)n;
  });
}

int afesp_gpu_gemm_crosscheck(afesp_handle hv, char ta, char tb, int M, int N, int K, int nbatch, double beta, int reps,
                              long long* mismatches, double* ms_tma, double* ms_cpasync) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(mismatches != nullptr, "gemm_crosscheck: null output");
    unsigned long long bad = 0;
    gemm_crosscheck(h.s.eng.stream, ta, tb, M, N, K, nbatch, beta, reps, &bad, ms_tma, ms_cpasync);
    *mismatches = (long long)bad;
  });
}

int afesp_gpu_dmma_peak(afesp_handle hv, double* tflops) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(tflops != nullptr, "dmma_peak: null output");
    int sms = 0;
    AFESP_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h.device));
    cudaStream_t st = h.s.eng.stream;
    DBuf out(8);
    const int iters = 20000, threads = 256, blocks = sms * 4;
    k_dmma_peak<<<blocks, threads, 0, st>>>(out.p, 100);
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
    StageTimer tm(&h);
    k_dmma_peak<<<blocks, threads, 0, st>>>(out.p, iters);
    count_launch(2);
    tm.stop();
    AFESP_CUDA_CHECK(cudaGetLastError());
    const double flops = 2.0 * 256.0 * 8.0 * iters * (threads / 32.0) * blocks;
    *tflops = flops / (h.last_ms * 1e-3) / 1e12;
  });
}

int afesp_gpu_gemm_time(afesp_handle hv, double* ms, double* flops) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(ms && flops, "gemm_time: null output");
    AFESP_CUDA_CHECK(cudaStreamSynchronize(h.s.eng.stream));
    *ms = gemm_timing_collect(flops);
  });
}

int afesp_gpu_gemm_stats(afesp_handle hv, double* ms, double* flops, long long* launches) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(ms && flops && launches, "gemm_stats: null output");
    AFESP_CUDA_CHECK(cudaStreamSynchronize(h.s.eng.stream));
    *ms = gemm_timing_collect(flops, launches);
  });
}

int afesp_gpu_timer(afesp_handle hv, int stop, double* ms) {
  return guarded(hv, [&](Handle& h) {
    if (!h.tm0) { AFESP_CUDA_CHECK(cudaEventCreate(&h.tm0)); AFESP_CUDA_CHECK(cudaEventCreate(&h.tm1)); }
    cudaStream_t st = h.s.eng.stream;
    if (!stop) {
      AFESP_CUDA_CHECK(cudaEventRecord(h.tm0, st));
      return;
    }
    AFESP_REQUIRE(ms != nullptr, "timer: null output");
    AFESP_CUDA_CHECK(cudaEventRecord(h.tm1, st));
    AFESP_CUDA_CHECK(cudaEventSynchronize(h.tm1));
    float t = 0.f;
    AFESP_CUDA_CHECK(cudaEventElapsedTime(&t, h.tm0, h.tm1));
    *ms = t;
  });
}

int afesp_gpu_last_stage_ms(afesp_handle hv, double* ms) {
  return guarded(hv, [&](Handle& h) {
    AFESP_REQUIRE(ms != nullptr, "last_stage_ms: null output");
    *ms = h.last_ms;
  });
}

#pragma GCC visibility pop
}  // extern "C"
