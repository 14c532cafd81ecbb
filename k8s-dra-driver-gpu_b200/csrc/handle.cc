// handle.cc — the probe handle behind the C ABI (include/cdprobe.h).
//
// Who calls this: the compute-domain-daemon's `run()` owns one handle for the
// life of the pod (reference: cmd/compute-domain-daemon/main.go:212-347; the
// cliqueID == "" branch main.go:244-250 is the single-node HGX B200 case) and
// re-runs the probe on every daemon-set change; `check()` (main.go:435-459)
// only reads the cached verdict.  bench.py drives the same ABI with one process
// per GPU (world_size > 1).
//
// Threading: cdprobe_run launches one persistent kernel per local GPU from the
// calling thread (a launch is ~4 us; the first device barrier absorbs the
// skew) and then polls the pinned result rows the kernels write.  No thread
// survives a call.
#include <cuda.h>
#include <cuda_runtime.h>
#include <errno.h>
#include <fcntl.h>
#include <sched.h>
#include <stddef.h>
#include <stdio.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include <new>
#include <string>
#include <vector>

#include "../../include/cdprobe.h"
#include "plan.h"
#include "probe_launch.h"
#include "probe_types.h"
#include "rendezvous.h"
#include "schedule.h"
#include "vmm.h"

namespace cdp {

thread_local std::string g_last_error;

static void set_err(const std::string& s) { g_last_error = s; }

static double now_ms() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e3 + ts.tv_nsec / 1e6;
}

constexpr int32_t kStatusUnmapped = CDPROBE_ERR_STATE;  // fault-injected / torn-down mapping

struct LocalRank {
  uint32_t grank = 0;
  int ordinal = -1;
  int sm_count = 0;
  uint32_t ctas = 0;
  bool coop = false;
  bool mig = false;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int max_ctas = 0;
  CUmemGenericAllocationHandle own = 0;
  bool has_own = false;
  int own_fd = -1;
  CUdeviceptr va[kMaxRanks] = {};
  bool mapped[kMaxRanks] = {};
  ResultRow* row = nullptr;
  char uuid[48] = {};
  Phase phases[kMaxPhases];
  uint32_t n_phases = 0;
  uint32_t peer_mask = 0;
};

}  // namespace cdp

using namespace cdp;

struct cdprobe {
  cdprobe_config_t cfg;
  Plan plan;
  Driver drv;
  Rendezvous rdv;
  uint32_t n_total = 0, n_local = 0, first = 0;
  uint32_t handle_type = 0;  // 0 none, 1 posix fd, 8 fabric
  LocalRank lr[kMaxRanks];
  CUmemGenericAllocationHandle imported[kMaxRanks] = {};
  bool has_import[kMaxRanks] = {};
  int32_t status[kMaxRanks][kMaxRanks];  // [issuer][owner] mapping status, all ranks
  uint64_t launch_seq = 0;
  uint64_t seed = 0;
  uint64_t src_sum[kMaxRanks][kMaxRanks] = {};
  uint64_t src_xor[kMaxRanks][kMaxRanks] = {};
  bool sticky = false;
  bool event_timing = false;
  uint32_t path = 0;          // 0 TMA bulk, 1 ld/st 128-bit, 2 ld/st 256-bit
  uint32_t warm_mode = 1;     // 0 never, 1 auto (after an idle gap), 2 always
  uint64_t warm_bytes = 8ull << 20;   // measured: the wake-up costs a fixed ~115 us whatever the byte count
  double warm_idle_ms = 5.0;  // auto: no penalty after 10 ms idle, full penalty after 50 ms (profiles/r01_cold_start_n2.jsonl)
  double last_run_end_ms = -1.0;
  bool warm_now = false;
  uint32_t debug_skip_rank = 0;  // 1-based local rank whose kernel is NOT launched (fault injection)
  uint32_t solo_rank = 0;        // 1-based local rank that runs alone, no cross-GPU barrier (ncu captures)
  uint32_t damage_write = 0;     // CDPROBE_OPT_DEBUG_DAMAGE_WRITE value (fault injection; 0 = off)
  double last_probe_ms = 0.0;    // host wall clock of the previous run (wait_rows: how long to spin hot)
  uint32_t verify_ctas = 32;  // CTAs that verify landing slots under CDPROBE_FLAG_OVERLAP_VERIFY
  double open_ms = 0, fill_ms = 0;
};

namespace cdp {

static int fail_cuda(const char* what, cudaError_t e) {
  set_err(std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
  if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInitializationError ||
      e == cudaErrorSystemDriverMismatch || e == cudaErrorSystemNotReady || e == cudaErrorNotSupported)
    return CDPROBE_ERR_NO_DEVICE;
  if (e == cudaErrorNoKernelImageForDevice || e == cudaErrorInvalidDeviceFunction ||
      e == cudaErrorCooperativeLaunchTooLarge)
    return CDPROBE_ERR_UNSUPPORTED;
  if (e == cudaErrorMemoryAllocation) return CDPROBE_ERR_NOMEM;
  return CDPROBE_ERR_CUDA;
}

static int fail_drv(const cdprobe* h, const char* what, CUresult r) {
  set_err(std::string(what) + ": " + h->drv.error_name(r));
  if (r == CUDA_ERROR_OUT_OF_MEMORY) return CDPROBE_ERR_NOMEM;
  if (r == CUDA_ERROR_NOT_SUPPORTED) return CDPROBE_ERR_UNSUPPORTED;
  return CDPROBE_ERR_CUDA;
}

#define CDP_RT(call)                                       \
  do {                                                     \
    cudaError_t e_ = (call);                               \
    if (e_ != cudaSuccess) return cdp::fail_cuda(#call, e_);    \
  } while (0)

static void format_uuid(const cudaUUID_t& u, bool mig, char out[48]) {
  const unsigned char* b = reinterpret_cast<const unsigned char*>(u.bytes);
  snprintf(out, 48, "%s-%02x%02x%02x%02x-%02x%02x-%02x%02x-%02x%02x-%02x%02x%02x%02x%02x%02x", mig ? "MIG" : "GPU",
           b[0], b[1], b[2], b[3], b[4], b[5], b[6], b[7], b[8], b[9], b[10], b[11], b[12], b[13], b[14], b[15]);
}

static bool imex_channel0_present() {
  int fd = ::open("/dev/nvidia-caps-imex-channels/channel0", O_RDONLY | O_CLOEXEC);
  if (fd < 0) return false;
  ::close(fd);
  return true;
}

// Map rank j's allocation into local rank i's address space.
static int32_t map_peer(cdprobe* h, uint32_t li, uint32_t j) {
  LocalRank& L = h->lr[li];
  if (L.mapped[j]) return 0;
  CUmemGenericAllocationHandle hnd;
  if (j >= h->first && j < h->first + h->n_local) {
    hnd = h->lr[j - h->first].own;
  } else if (h->has_import[j]) {
    hnd = h->imported[j];
  } else {
    return CDPROBE_ERR_RENDEZVOUS;
  }
  if (cudaSetDevice(L.ordinal) != cudaSuccess) return CDPROBE_ERR_CUDA;
  CUdeviceptr va = 0;
  const size_t sz = h->plan.alloc_bytes;
  CUresult r = h->drv.MemAddressReserve(&va, sz, kVmmGranule, 0, 0);
  if (r != CUDA_SUCCESS) return (int32_t)r;
  r = h->drv.MemMap(va, sz, 0, hnd, 0);
  if (r != CUDA_SUCCESS) {
    h->drv.MemAddressFree(va, sz);
    return (int32_t)r;
  }
  CUmemAccessDesc ad;
  memset(&ad, 0, sizeof(ad));
  ad.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  ad.location.id = L.ordinal;
  ad.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  r = h->drv.MemSetAccess(va, sz, &ad, 1);
  if (r != CUDA_SUCCESS) {
    h->drv.MemUnmap(va, sz);
    h->drv.MemAddressFree(va, sz);
    return (int32_t)r;
  }
  L.va[j] = va;
  L.mapped[j] = true;
  return 0;
}

static void unmap_peer(cdprobe* h, uint32_t li, uint32_t j) {
  LocalRank& L = h->lr[li];
  if (!L.mapped[j]) return;
  cudaSetDevice(L.ordinal);
  h->drv.MemUnmap(L.va[j], h->plan.alloc_bytes);
  h->drv.MemAddressFree(L.va[j], h->plan.alloc_bytes);
  L.va[j] = 0;
  L.mapped[j] = false;
}

// Phase table of local rank li: see schedule.cc.
static int build_phases(cdprobe* h, uint32_t li) {
  LocalRank& L = h->lr[li];
  ScheduleInput in;
  in.plan = &h->plan;
  in.rank = L.grank;
  in.ops = h->cfg.ops;
  in.flags = h->cfg.flags;
  in.ctas = L.ctas;
  in.verify_ctas = h->verify_ctas;
  in.status = h->status;
  const int rc = make_phases(in, L.phases, &L.n_phases, &L.peer_mask);
  if (rc != CDPROBE_OK) set_err("schedule needs more than CDPROBE_MAX_PHASES phases (use overlap-verify or fewer ops)");
  return rc;
}

static int rebuild_all(cdprobe* h) {
  for (uint32_t li = 0; li < h->n_local; ++li) {
    const int rc = build_phases(h, li);
    if (rc != CDPROBE_OK) return rc;
  }
  return CDPROBE_OK;
}

static void fill_params(const cdprobe* h, uint32_t li, const Phase* phases, uint32_t n_phases, uint32_t peer_mask,
                        ProbeParams* P) {
  const LocalRank& L = h->lr[li];
  memset(P, 0, sizeof(*P));
  for (uint32_t j = 0; j < h->n_total; ++j) P->base_peer[j] = L.mapped[j] ? reinterpret_cast<uint8_t*>(L.va[j]) : nullptr;
  P->row = L.row;
  P->run_seq = h->launch_seq;
  P->seq_base = h->launch_seq * (uint64_t)(kMaxPhases + 2);
  P->timeout_ns = (uint64_t)h->cfg.timeout_ms * 1000000ull;
  P->bpp = h->plan.bpp;
  P->src_off = h->plan.src_off;
  P->land_off = h->plan.land_off;
  P->rank = L.grank;
  P->n_ranks = h->n_total;
  P->n_phases = n_phases;
  P->peer_mask = peer_mask;
  P->use_ldst = h->path;
  P->full_mode = h->plan.full ? 1u : 0u;
  for (uint32_t p = 0; p < n_phases; ++p) {
    P->phase[p] = phases[p];
    for (int jb = 0; jb < 2; ++jb) {
      Job& job = P->phase[p].job[jb];
      if (job.kind == kJobWrite) job.salt = write_salt(h->seed, L.grank, (uint32_t)job.peer, h->launch_seq);
      // fault injection: the writer byte is unused on write jobs; nonzero = damage code the barrier applies
      if (job.kind == kJobWrite && h->damage_write != 0 && (h->damage_write >> 16) == li + 1 &&
          ((h->damage_write >> 8) & 0xffu) == (uint32_t)job.peer)
        job.writer = (uint8_t)(h->damage_write & 0xffu);
      if (job.kind == kJobWarm) job.salt = h->warm_now ? h->warm_bytes : 0ull;
    }
  }
}

// Waits until every local row carries `token`; returns false on host timeout or a kernel error.
// The rows are pinned host words the kernels write themselves.  A healthy probe is over in 0.5-3.3 ms,
// so the wait spins hot for as long as a healthy run can plausibly take (twice the previous run, at
// least 2 ms, at most 50 ms) and then backs off to a 100 us sleep between polls: a hung peer costs the
// daemon pod a sleeping thread for timeout_ms, not a core burnt inside its CPU limit.
static bool wait_rows(cdprobe* h, uint64_t token) {
  const double t_begin = now_ms();
  const double t_end = t_begin + h->cfg.timeout_ms + 2000.0;
  double hot_ms = 2.0 * h->last_probe_ms;
  if (hot_ms < 2.0) hot_ms = 2.0;
  if (hot_ms > 50.0) hot_ms = 50.0;
  const double t_hot = t_begin + hot_ms;
  bool hot = true;
  uint32_t spins = 0;
  for (;;) {
    bool all = true;
    for (uint32_t li = 0; li < h->n_local; ++li) {
      if (h->lr[li].row->done != token) {
        all = false;
        break;
      }
    }
    if (all) {
      __sync_synchronize();
      return true;
    }
    if (!hot) {
      timespec ts = {0, 100000};
      nanosleep(&ts, nullptr);
    }
    if (!hot || (++spins & 0x3ffu) == 0) {
      const double t = now_ms();
      if (t > t_end) return false;
      if (hot && t > t_hot) hot = false;
      if (hot || (++spins & 0x3fu) == 0) {
        // surface asynchronous launch/kernel errors instead of waiting on them
        for (uint32_t li = 0; li < h->n_local; ++li) {
          if (h->solo_rank && h->solo_rank != li + 1) continue;
          cudaSetDevice(h->lr[li].ordinal);
          cudaError_t q = cudaStreamQuery(h->lr[li].stream);
          if (q != cudaSuccess && q != cudaErrorNotReady) {
            set_err(std::string("kernel failed: ") + cudaGetErrorName(q));
            return false;
          }
        }
      }
    }
  }
}

static int reset_ctrl_local(cdprobe* h, uint32_t li) {
  LocalRank& L = h->lr[li];
  CDP_RT(cudaSetDevice(L.ordinal));
  uint8_t* base = reinterpret_cast<uint8_t*>(L.va[L.grank]);
  const size_t off = offsetof(Ctrl, grid_arrive);
  CDP_RT(cudaMemsetAsync(base + off, 0, sizeof(Ctrl) - off, L.stream));
  CDP_RT(cudaStreamSynchronize(L.stream));
  return CDPROBE_OK;
}

static int launch_one(cdprobe* h, uint32_t li, const ProbeParams& P) {
  LocalRank& L = h->lr[li];
  CDP_RT(cudaSetDevice(L.ordinal));
  const bool coop = L.coop && !(h->cfg.flags & CDPROBE_FLAG_NO_COOPERATIVE);
  cudaError_t e = (cudaError_t)probe_kernel_launch(&P, L.ctas, coop, L.stream);
  if (e != cudaSuccess) return fail_cuda("launch cdprobe_kernel", e);
  return CDPROBE_OK;
}

// Open-time: fill the source pattern and let the probe kernel itself compute the
// slice checksums that readers will compare against (published in Ctrl).
static int fill_and_publish(cdprobe* h) {
  const Plan& pl = h->plan;
  h->launch_seq++;
  for (uint32_t li = 0; li < h->n_local; ++li) {
    LocalRank& L = h->lr[li];
    CDP_RT(cudaSetDevice(L.ordinal));
    uint8_t* base = reinterpret_cast<uint8_t*>(L.va[L.grank]);
    CDP_RT(cudaMemsetAsync(base, 0, kCtrlBytes, L.stream));
    CDP_RT(cudaMemsetAsync(base + pl.land_off, 0, pl.land_bytes, L.stream));
    cudaError_t e = (cudaError_t)probe_fill_launch(base + pl.src_off, pl.src_bytes, h->seed, L.grank,
                                                   (unsigned)L.sm_count * 8u, L.stream);
    if (e != cudaSuccess) return fail_cuda("launch fill kernel", e);
    Phase ph[kMaxPhases];
    memset(ph, 0, sizeof(ph));
    for (uint32_t s = 0; s < pl.n_slices; ++s) {
      ph[s].job[0].kind = kJobRead;
      ph[s].job[0].peer = (int8_t)L.grank;
      ph[s].job[0].slot = (uint8_t)s;
      ph[s].job[0].cta0 = 0;
      ph[s].job[0].nctas = (uint16_t)L.ctas;
      ph[s].sync_mask = 0;
      ph[s].post_mask = 0;
    }
    ProbeParams P;
    fill_params(h, li, ph, pl.n_slices, 0u, &P);
    L.row->done = 0;
    const int rc = launch_one(h, li, P);
    if (rc != CDPROBE_OK) return rc;
  }
  if (!wait_rows(h, h->launch_seq)) {
    h->sticky = true;
    if (g_last_error.empty()) set_err("timeout computing source checksums");
    return CDPROBE_ERR_TIMEOUT;
  }
  for (uint32_t li = 0; li < h->n_local; ++li) {
    LocalRank& L = h->lr[li];
    CDP_RT(cudaSetDevice(L.ordinal));
    if (L.row->aborted) {
      set_err("device watchdog fired while computing source checksums");
      return CDPROBE_ERR_TIMEOUT;
    }
    uint64_t pub[2][kMaxRanks];
    memset(pub, 0, sizeof(pub));
    for (uint32_t s = 0; s < pl.n_slices; ++s) {
      pub[0][s] = h->src_sum[li][s] = L.row->ph[s].sum[0];
      pub[1][s] = h->src_xor[li][s] = L.row->ph[s].xr[0];
    }
    uint8_t* base = reinterpret_cast<uint8_t*>(L.va[L.grank]);
    CDP_RT(cudaMemcpyAsync(base + offsetof(Ctrl, src_sum), pub[0], sizeof(pub[0]), cudaMemcpyHostToDevice, L.stream));
    CDP_RT(cudaMemcpyAsync(base + offsetof(Ctrl, src_xor), pub[1], sizeof(pub[1]), cudaMemcpyHostToDevice, L.stream));
    CDP_RT(cudaStreamSynchronize(L.stream));
  }
  return CDPROBE_OK;
}

static void destroy(cdprobe* h) {
  if (h == nullptr) return;
  for (uint32_t li = 0; li < h->n_local; ++li) {
    LocalRank& L = h->lr[li];
    if (L.ordinal < 0) continue;
    cudaSetDevice(L.ordinal);
    if (L.stream) cudaStreamSynchronize(L.stream);
    for (uint32_t j = 0; j < (uint32_t)kMaxRanks; ++j) unmap_peer(h, li, j);
  }
  for (uint32_t j = 0; j < (uint32_t)kMaxRanks; ++j)
    if (h->has_import[j]) {
      h->drv.MemRelease(h->imported[j]);
      h->has_import[j] = false;
    }
  for (uint32_t li = 0; li < h->n_local; ++li) {
    LocalRank& L = h->lr[li];
    if (L.ordinal < 0) continue;
    cudaSetDevice(L.ordinal);
    if (L.has_own) h->drv.MemRelease(L.own);
    if (L.own_fd >= 0) ::close(L.own_fd);
    if (L.row) cudaFreeHost(L.row);
    if (L.ev0) cudaEventDestroy(L.ev0);
    if (L.ev1) cudaEventDestroy(L.ev1);
    if (L.stream) cudaStreamDestroy(L.stream);
  }
  h->rdv.close();
  delete h;
}

static int open_impl(const cdprobe_config_t* cfg, cdprobe* h) {
  const double t0 = now_ms();
  h->cfg = *cfg;
  cdprobe_config_t& c = h->cfg;
  if (c.ops == 0) c.ops = CDPROBE_OP_READ | CDPROBE_OP_WRITE;
  if (c.ops & ~(CDPROBE_OP_READ | CDPROBE_OP_WRITE)) return CDPROBE_ERR_ARG;
  if (c.timeout_ms == 0) c.timeout_ms = 5000;
  // gate: see gate_gbps(); 0 in either field selects the default at verdict time
  if (c.link_peak_gbps < 0.f || c.min_fraction < 0.f) return CDPROBE_ERR_ARG;
  if (c.world_size == 0) c.world_size = 1;
  if (c.rank >= c.world_size) return CDPROBE_ERR_ARG;
  h->path = (c.flags & CDPROBE_FLAG_PATH_LDST) ? 1u : 0u;
  if (!(c.flags & CDPROBE_FLAG_SERIAL_VERIFY)) c.flags |= CDPROBE_FLAG_OVERLAP_VERIFY;  // overlapped verify is the default
  h->seed = c.seed ? c.seed : kDefaultSeed;
  c.session[sizeof(c.session) - 1] = '\0';
  memset(h->status, 0, sizeof(h->status));

  std::string err;
  cudaError_t e = h->drv.load(&err);
  if (e != cudaSuccess) {
    set_err(err);
    return CDPROBE_ERR_NO_DEVICE;
  }
  int ndev = 0;
  e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess) return fail_cuda("cudaGetDeviceCount", e);
  if (ndev <= 0) {
    set_err("no CUDA device visible");
    return CDPROBE_ERR_NO_DEVICE;
  }
  if (c.n_gpus == 0) {
    c.n_gpus = ndev > kMaxRanks ? kMaxRanks : (uint32_t)ndev;
    for (uint32_t i = 0; i < c.n_gpus; ++i) c.ordinals[i] = (int32_t)i;
  }
  if (c.n_gpus > (uint32_t)kMaxRanks) return CDPROBE_ERR_ARG;
  for (uint32_t i = 0; i < c.n_gpus; ++i) {
    if (c.ordinals[i] < 0 || c.ordinals[i] >= ndev) {
      set_err("ordinal out of range");
      return CDPROBE_ERR_ARG;
    }
    if (!(c.flags & CDPROBE_FLAG_ALLOW_SAME_DEVICE))
      for (uint32_t k = 0; k < i; ++k)
        if (c.ordinals[k] == c.ordinals[i]) {
          set_err("duplicate ordinal (set CDPROBE_FLAG_ALLOW_SAME_DEVICE for tests)");
          return CDPROBE_ERR_ARG;
        }
  }
  h->n_local = c.n_gpus;
  h->n_total = c.n_gpus * c.world_size;
  h->first = c.rank * c.n_gpus;
  if (h->n_total > (uint32_t)kMaxRanks) {
    set_err("more than CDPROBE_MAX_GPUS ranks");
    return CDPROBE_ERR_ARG;
  }
  int rc = make_plan(h->n_total, c.bytes, c.mode, c.flags, &h->plan);
  if (rc != CDPROBE_OK) {
    set_err("invalid bytes/mode for this domain size");
    return rc;
  }

  if (c.world_size > 1) {
    if (h->rdv.connect(c.session, c.rank, c.world_size, c.timeout_ms + 20000, &err) != 0) {
      set_err(err);
      return CDPROBE_ERR_RENDEZVOUS;
    }
    uint32_t mine = c.n_gpus, all[kMaxRanks * 4];
    if (c.world_size > (uint32_t)kMaxRanks || h->rdv.allgather(&mine, sizeof(mine), all, &err) != 0) {
      set_err(err);
      return CDPROBE_ERR_RENDEZVOUS;
    }
    for (uint32_t r = 0; r < c.world_size; ++r)
      if (all[r] != c.n_gpus) {
        set_err("every process must drive the same number of GPUs");
        return CDPROBE_ERR_ARG;
      }
  }

  const bool want_fabric = (c.flags & CDPROBE_FLAG_FABRIC_HANDLES) && imex_channel0_present();
  h->handle_type = want_fabric ? 8u : (c.world_size > 1 ? 1u : 0u);
  if (c.world_size > 1 && h->rdv.is_tcp() && !want_fabric) {
    set_err("a tcp: rendezvous spans nodes: it needs CDPROBE_FLAG_FABRIC_HANDLES and /dev/nvidia-caps-imex-channels/channel0");
    return CDPROBE_ERR_UNSUPPORTED;
  }

  // ---- per local rank: device, stream, allocation, result row -------------
  for (uint32_t li = 0; li < h->n_local; ++li) {
    LocalRank& L = h->lr[li];
    L.grank = h->first + li;
    L.ordinal = c.ordinals[li];
    CDP_RT(cudaSetDevice(L.ordinal));
    CDP_RT(cudaFree(0));
    cudaDeviceProp prop;
    CDP_RT(cudaGetDeviceProperties(&prop, L.ordinal));
    if (prop.major != 10) {
      set_err(std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
              "; libcdprobe carries sm_100a code only");
      return CDPROBE_ERR_UNSUPPORTED;
    }
    L.sm_count = prop.multiProcessorCount;
    L.mig = strstr(prop.name, "MIG") != nullptr || (c.flags & CDPROBE_FLAG_SIMULATE_MIG);
    format_uuid(prop.uuid, L.mig, L.uuid);
    int coop = 0;
    CDP_RT(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, L.ordinal));
    L.coop = coop != 0;
    int per_sm = 0;
    e = (cudaError_t)probe_kernel_prepare(&per_sm);
    if (e != cudaSuccess) return fail_cuda("prepare cdprobe_kernel", e);
    if (per_sm < 1) {
      set_err("persistent kernel does not fit an SM");
      return CDPROBE_ERR_UNSUPPORTED;
    }
    uint32_t ctas = c.ctas ? c.ctas : (uint32_t)L.sm_count;
    const uint32_t cap = (uint32_t)L.sm_count * (uint32_t)per_sm;
    if (ctas > cap) ctas = cap;
    if (ctas > 65535u) ctas = 65535u;
    L.ctas = ctas;
    L.max_ctas = (int)(cap > 65535u ? 65535u : cap);
    CDP_RT(cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
    CDP_RT(cudaEventCreate(&L.ev0));
    CDP_RT(cudaEventCreate(&L.ev1));

    CUmemAllocationProp ap;
    memset(&ap, 0, sizeof(ap));
    ap.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    ap.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    ap.location.id = L.ordinal;
    ap.requestedHandleTypes = h->handle_type == 8u   ? CU_MEM_HANDLE_TYPE_FABRIC
                              : h->handle_type == 1u ? CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR
                                                     : CU_MEM_HANDLE_TYPE_NONE;
    size_t gran = 0;
    CUresult r = h->drv.MemGetAllocationGranularity(&gran, &ap, CU_MEM_ALLOC_GRANULARITY_MINIMUM);
    if (r != CUDA_SUCCESS) return fail_drv(h, "cuMemGetAllocationGranularity", r);
    if (gran == 0 || kVmmGranule % gran != 0) {
      set_err("unexpected VMM granularity " + std::to_string(gran));
      return CDPROBE_ERR_UNSUPPORTED;
    }
    r = h->drv.MemCreate(&L.own, h->plan.alloc_bytes, &ap, 0);
    if (r != CUDA_SUCCESS) return fail_drv(h, "cuMemCreate", r);
    L.has_own = true;
    if (h->handle_type == 1u) {
      int fd = -1;
      r = h->drv.MemExportToShareableHandle(&fd, L.own, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0);
      if (r != CUDA_SUCCESS) return fail_drv(h, "cuMemExportToShareableHandle(fd)", r);
      L.own_fd = fd;
    }
    void* row = nullptr;
    CDP_RT(cudaHostAlloc(&row, sizeof(ResultRow), cudaHostAllocPortable | cudaHostAllocMapped));
    memset(row, 0, sizeof(ResultRow));
    L.row = static_cast<ResultRow*>(row);
  }

  // ---- exchange handles between processes ---------------------------------
  if (c.world_size > 1) {
    if (h->handle_type == 1u) {
      int mine[kMaxRanks];
      for (uint32_t li = 0; li < h->n_local; ++li) mine[li] = h->lr[li].own_fd;
      std::vector<int> all;
      if (h->rdv.allgather_fds(mine, h->n_local, &all, &err) != 0) {
        set_err(err);
        return CDPROBE_ERR_RENDEZVOUS;
      }
      for (uint32_t j = 0; j < h->n_total; ++j) {
        const bool local = j >= h->first && j < h->first + h->n_local;
        if (!local) {
          CUresult r = h->drv.MemImportFromShareableHandle(&h->imported[j], (void*)(uintptr_t)all[j],
                                                           CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR);
          if (r == CUDA_SUCCESS) h->has_import[j] = true;
          else
            for (uint32_t li = 0; li < h->n_local; ++li) h->status[h->first + li][j] = (int32_t)r;
        }
        ::close(all[j]);
      }
    } else {
      CUmemFabricHandle mine[kMaxRanks], all[kMaxRanks];
      memset(mine, 0, sizeof(mine));
      for (uint32_t li = 0; li < h->n_local; ++li) {
        CUresult r = h->drv.MemExportToShareableHandle(&mine[li], h->lr[li].own, CU_MEM_HANDLE_TYPE_FABRIC, 0);
        if (r != CUDA_SUCCESS) return fail_drv(h, "cuMemExportToShareableHandle(fabric)", r);
      }
      if (h->rdv.allgather(mine, sizeof(CUmemFabricHandle) * h->n_local, all, &err) != 0) {
        set_err(err);
        return CDPROBE_ERR_RENDEZVOUS;
      }
      for (uint32_t j = 0; j < h->n_total; ++j) {
        const bool local = j >= h->first && j < h->first + h->n_local;
        if (local) continue;
        CUresult r = h->drv.MemImportFromShareableHandle(&h->imported[j], &all[j], CU_MEM_HANDLE_TYPE_FABRIC);
        if (r == CUDA_SUCCESS) h->has_import[j] = true;
        else
          for (uint32_t li = 0; li < h->n_local; ++li) h->status[h->first + li][j] = (int32_t)r;
      }
    }
  }

  // ---- map every rank's allocation into every local rank's address space --
  for (uint32_t li = 0; li < h->n_local; ++li) {
    LocalRank& L = h->lr[li];
    for (uint32_t j = 0; j < h->n_total; ++j) {
      int32_t st = h->status[L.grank][j];
      if (st == 0) {
        if (j != L.grank && L.mig && (c.flags & (CDPROBE_FLAG_MIG_AWARE | CDPROBE_FLAG_SIMULATE_MIG)))
          st = CDPROBE_ERR_UNSUPPORTED;  // no P2P under MIG (SURVEY H8): identity matrix, "not applicable"
        else st = map_peer(h, li, j);
      }
      h->status[L.grank][j] = st;
    }
    if (h->status[L.grank][L.grank] != 0) {
      set_err("cannot map own allocation: " + h->drv.error_name((CUresult)h->status[L.grank][L.grank]));
      return CDPROBE_ERR_CUDA;
    }
  }
  if (c.world_size > 1) {
    int32_t mine[kMaxRanks][kMaxRanks], all[kMaxRanks][kMaxRanks][kMaxRanks];
    memset(mine, 0, sizeof(mine));
    for (uint32_t li = 0; li < h->n_local; ++li) memcpy(mine[li], h->status[h->first + li], sizeof(mine[li]));
    if (h->rdv.allgather(mine, sizeof(int32_t) * kMaxRanks * h->n_local, all, &err) != 0) {
      set_err(err);
      return CDPROBE_ERR_RENDEZVOUS;
    }
    const int32_t* flat = &all[0][0][0];
    for (uint32_t g = 0; g < h->n_total; ++g) memcpy(h->status[g], flat + (size_t)g * kMaxRanks, sizeof(h->status[g]));
  }
  rc = rebuild_all(h);
  if (rc != CDPROBE_OK) return rc;
  h->open_ms = now_ms() - t0;

  const double t1 = now_ms();
  rc = fill_and_publish(h);
  if (rc != CDPROBE_OK) return rc;
  h->fill_ms = now_ms() - t1;
  // nobody may start probing before every rank has published its checksums
  if (c.world_size > 1 && h->rdv.barrier(&err) != 0) {
    set_err(err);
    return CDPROBE_ERR_RENDEZVOUS;
  }
  return CDPROBE_OK;
}

// The GB/s an ordered pair must reach for a passing verdict (0: bandwidth is not judged).
//   link_peak_gbps > 0 : absolute, min_fraction x link_peak_gbps (default fraction 0.65: the round-1 gate
//                        against nominal 900).
//   link_peak_gbps == 0: calibrated.  What a healthy B200 port delivers to SM-issued traffic, measured on
//                        the same box next to the copy engine (tools/linkbench.cu ->
//                        profiles/r02_linkbench_n2.jsonl), de-rated for the ~8 us a phase spends ramping and
//                        draining; default fraction 0.90.  Run-to-run spread of a pair is 0.2-0.7 %, spread
//                        across pairs and boxes ~3 %: 0.90 leaves healthy hardware a 7 % margin, while a
//                        port that lost 2 of its 18 links (-11 %) fails.
struct HealthyRates {  // GB/s per direction per GPU, 1 GiB transfers
  double read_bidi = 672.0, write_bidi = 703.0, read_uni = 785.0, write_uni = 714.7;
  double phase_overhead_ns = 8000.0;
};
static float gate_gbps_for(const cdprobe_config_t& cfg, uint32_t n_total, uint64_t bpp, bool is_read) {
  if (cfg.mode == CDPROBE_MODE_REACH_ONLY || n_total <= 1) return 0.f;
  if (cfg.link_peak_gbps > 0.f) return (cfg.min_fraction > 0.f ? cfg.min_fraction : 0.65f) * cfg.link_peak_gbps;
  const HealthyRates hr;
  const bool uni = (cfg.flags & CDPROBE_FLAG_UNIDIRECTIONAL) != 0;
  const double rate = is_read ? (uni ? hr.read_uni : hr.read_bidi) : (uni ? hr.write_uni : hr.write_bidi);
  const double b = (double)bpp;
  const double expected = b / (b / rate + hr.phase_overhead_ns);  // bytes per ns == GB/s
  return (float)((cfg.min_fraction > 0.f ? cfg.min_fraction : 0.90f) * expected);
}
static float gate_gbps(const cdprobe* h, bool is_read) { return gate_gbps_for(h->cfg, h->n_total, h->plan.bpp, is_read); }

static void assemble(const cdprobe* h, cdprobe_result_t* out) {
  const Plan& pl = h->plan;
  const float gate_r = gate_gbps(h, true), gate_w = gate_gbps(h, false);
  out->gate_gbps_read = gate_r;
  out->gate_gbps_write = gate_w;
  bool verdict = true;
  float min_r = 0.f, min_w = 0.f;
  bool have_r = false, have_w = false;
  for (uint32_t li = 0; li < h->n_local; ++li) {
    const LocalRank& L = h->lr[li];
    const ResultRow* row = L.row;
    const uint32_t g = L.grank;
    out->row_mask |= 1u << g;
    for (uint32_t j = 0; j < h->n_total; ++j) out->status[g * CDPROBE_MAX_GPUS + j] = h->status[g][j];
    if (!pl.diag) {
      out->reach_read[g * CDPROBE_MAX_GPUS + g] = 1;  // frozen oracle: reach[i][i] = 1 (SURVEY.md §8c)
      out->reach_write[g * CDPROBE_MAX_GPUS + g] = 1;
    }
    if (row->aborted) out->aborted = 1;
    out->device_ms[li] = row->t_last > row->t_first ? (double)(row->t_last - row->t_first) / 1e6 : 0.0;
    out->kernel_ms[li] = row->t_exit > row->t_enter ? (double)(row->t_exit - row->t_enter) / 1e6 : 0.0;
    double bar_ns = 0.0;
    bool slow[kMaxRanks] = {};
    for (uint32_t p = 0; p < L.n_phases; ++p) {
      const PhaseOut& o = row->ph[p];
      if (p + 1 < L.n_phases) {
        const PhaseOut& nx = row->ph[p + 1];
        if (nx.t_start > o.t_arrive) bar_ns += (double)(nx.t_start - o.t_arrive);
      }
      const Job& job = L.phases[p].job[0];
      if (job.kind != kJobRead && job.kind != kJobWrite) continue;
      const uint32_t idx = g * CDPROBE_MAX_GPUS + (uint32_t)job.peer;
      const bool done = o.code[0] == kCodeOk && o.t_end[0] > o.t_start;
      const float gbps = done ? (float)((double)pl.bpp / (double)(o.t_end[0] - o.t_start)) : 0.f;
      const bool offdiag = (uint32_t)job.peer != g || h->n_total == 1;
      if (job.kind == kJobRead) {
        const bool ok = done && o.sum[0] == o.exp_sum[0] && o.xr[0] == o.exp_xr[0];
        out->reach_read[idx] = ok ? 1 : 0;
        out->gbps_read[idx] = gbps;
        out->sum_read[idx] = o.sum[0];
        out->xor_read[idx] = o.xr[0];
        if (offdiag) {
          if (!have_r || gbps < min_r) min_r = gbps;
          have_r = true;
          if (ok && (uint32_t)job.peer != g && gbps < gate_r) slow[job.peer] = true;
        }
      } else {
        const bool ok = done && o.verdict[0] == h->launch_seq * 4ull + kVerdictOk;
        out->reach_write[idx] = ok ? 1 : 0;
        out->gbps_write[idx] = gbps;
        out->sum_write[idx] = o.sum[0];
        out->xor_write[idx] = o.xr[0];
        if (offdiag) {
          if (!have_w || gbps < min_w) min_w = gbps;
          have_w = true;
          if (ok && (uint32_t)job.peer != g && gbps < gate_w) slow[job.peer] = true;
        }
      }
    }
    out->barrier_us[li] = bar_ns / 1e3;
    // every off-diagonal cell of this row must have been probed, reachable and at speed
    for (uint32_t j = 0; j < h->n_total; ++j) {
      if (j == g) continue;
      // P2P is not applicable between MIG instances: the cell stays 0 but must not turn a MIG-only
      // domain NotReady (SURVEY H8)
      if (h->status[g][j] == CDPROBE_ERR_UNSUPPORTED || h->status[j][g] == CDPROBE_ERR_UNSUPPORTED) continue;
      const uint32_t idx = g * CDPROBE_MAX_GPUS + j;
      const bool unreachable = ((h->cfg.ops & CDPROBE_OP_READ) && !out->reach_read[idx]) ||
                               ((h->cfg.ops & CDPROBE_OP_WRITE) && !out->reach_write[idx]);
      if (unreachable) out->unreachable_pairs++;
      else if (slow[j]) out->slow_pairs++;
      if (unreachable || slow[j]) verdict = false;
    }
    if (h->n_total == 1 && pl.diag) {  // loop-back: reachability only (HBM speed is not a fabric property)
      const uint32_t idx = g * CDPROBE_MAX_GPUS + g;
      if (((h->cfg.ops & CDPROBE_OP_READ) && !out->reach_read[idx]) || ((h->cfg.ops & CDPROBE_OP_WRITE) && !out->reach_write[idx]))
        verdict = false;
    }
  }
  out->min_gbps_read = min_r;
  out->min_gbps_write = min_w;
  out->verdict = (verdict && !out->aborted) ? 1u : 0u;
}

}  // namespace cdp

// ------------------------------------------------------------------ C ABI ----
extern "C" {

uint32_t cdprobe_abi_version(void) { return CDPROBE_ABI_VERSION; }

const char* cdprobe_strerror(int code) {
  switch (code) {
    case CDPROBE_OK: return "ok";
    case CDPROBE_ERR_ABI: return "ABI version mismatch";
    case CDPROBE_ERR_ARG: return "invalid argument";
    case CDPROBE_ERR_NO_DEVICE: return "no CUDA driver or device (there is no CPU fallback)";
    case CDPROBE_ERR_CUDA: return "CUDA call failed";
    case CDPROBE_ERR_TIMEOUT: return "probe timed out";
    case CDPROBE_ERR_RENDEZVOUS: return "multi-process rendezvous failed";
    case CDPROBE_ERR_NOMEM: return "out of memory";
    case CDPROBE_ERR_UNSUPPORTED: return "device or driver lacks a required feature";
    case CDPROBE_ERR_STATE: return "handle is in an unusable state";
    case CDPROBE_ERR_INTEGRITY: return "integrity self-check failed";
    default: return "unknown cdprobe error";
  }
}

const char* cdprobe_last_error(void) { return cdp::g_last_error.c_str(); }

int cdprobe_open(const cdprobe_config_t* cfg, cdprobe_t** out) {
  cdp::g_last_error.clear();
  if (cfg == nullptr || out == nullptr) return CDPROBE_ERR_ARG;
  *out = nullptr;
  if (cfg->abi != CDPROBE_ABI_VERSION) return CDPROBE_ERR_ABI;
  cdprobe* h = new (std::nothrow) cdprobe();
  if (h == nullptr) return CDPROBE_ERR_NOMEM;
  const int rc = cdp::open_impl(cfg, h);
  if (rc != CDPROBE_OK) {
    const std::string keep = cdp::g_last_error;
    cdp::destroy(h);
    cdp::g_last_error = keep;
    return rc;
  }
  *out = h;
  return CDPROBE_OK;
}

int cdprobe_run(cdprobe_t* h, cdprobe_result_t* out) {
  cdp::g_last_error.clear();
  if (h == nullptr || out == nullptr) return CDPROBE_ERR_ARG;
  // The caller reads *out whatever the return code (the daemon writes a verdict from it): never leave it
  // as it came in.
  memset(out, 0, sizeof(*out));
  out->abi = CDPROBE_ABI_VERSION;
  out->n = h->n_total;
  out->bytes_per_pair = h->plan.bpp;
  out->rounds = h->plan.rounds;
  if (h->sticky) {
    cdp::set_err("handle is unusable after an earlier timeout or CUDA error: close it and open a new one");
    return CDPROBE_ERR_STATE;
  }
  const double t0 = cdp::now_ms();
  h->launch_seq++;
  out->run_seq = h->launch_seq;
  h->warm_now = h->warm_mode == 2 ||
                (h->warm_mode == 1 && (h->last_run_end_ms < 0 || t0 - h->last_run_end_ms > h->warm_idle_ms));
  cdp::ProbeParams P;
  for (uint32_t li = 0; li < h->n_local; ++li) {
    cdp::LocalRank& L = h->lr[li];
    const bool skipped = h->debug_skip_rank == li + 1 || (h->solo_rank != 0 && h->solo_rank != li + 1);
    if (skipped) {  // fault injection / solo profiling: this rank never shows up at the barriers
      memset(L.row->ph, 0, sizeof(L.row->ph));
      L.row->aborted = h->solo_rank ? 0u : 1u;
      L.row->n_phases = L.n_phases;
      L.row->t_first = L.row->t_last = 0;
      L.row->t_enter = L.row->t_exit = 0;
      L.row->done = h->launch_seq;
      continue;
    }
    if (h->solo_rank == li + 1) {
      // only this rank's own transfers; nobody to wait for, nobody verifies (reach_write stays 0)
      cdp::Phase solo[cdp::kMaxPhases];
      for (uint32_t p = 0; p < L.n_phases; ++p) {
        solo[p] = L.phases[p];
        solo[p].sync_mask = 0;
        solo[p].post_mask = 0;
        for (int jb = 0; jb < 2; ++jb)
          if (solo[p].job[jb].kind == cdp::kJobVerify) solo[p].job[jb].kind = cdp::kJobNone;
      }
      cdp::fill_params(h, li, solo, L.n_phases, 0u, &P);
    } else {
      cdp::fill_params(h, li, L.phases, L.n_phases, L.peer_mask, &P);
    }
    if (h->event_timing) {
      cudaSetDevice(L.ordinal);
      cudaEventRecord(L.ev0, L.stream);
    }
    const int rc = cdp::launch_one(h, li, P);
    if (rc != CDPROBE_OK) {
      h->sticky = true;
      return rc;
    }
    if (h->event_timing) cudaEventRecord(L.ev1, L.stream);
    out->launches++;
    out->phases = L.n_phases;
  }
  if (!cdp::wait_rows(h, h->launch_seq)) {
    h->sticky = true;
    if (cdp::g_last_error.empty()) cdp::set_err("host watchdog: kernels did not report within timeout_ms + 2 s");
    out->probe_ms = cdp::now_ms() - t0;
    return CDPROBE_ERR_TIMEOUT;
  }
  cdp::assemble(h, out);
  h->last_run_end_ms = cdp::now_ms();
  out->probe_ms = h->last_run_end_ms - t0;
  h->last_probe_ms = out->probe_ms;
  out->warmed = (h->warm_now && h->plan.rounds > 0) ? 1u : 0u;  // N = 1 has no link to wake
  if (h->event_timing) {  // after probe_ms: the event round trip is not part of the probe
    for (uint32_t li = 0; li < h->n_local; ++li) {
      cdp::LocalRank& L = h->lr[li];
      if (h->debug_skip_rank == li + 1 || (h->solo_rank != 0 && h->solo_rank != li + 1)) continue;
      float ms = 0.f;
      cudaSetDevice(L.ordinal);
      if (cudaEventSynchronize(L.ev1) == cudaSuccess && cudaEventElapsedTime(&ms, L.ev0, L.ev1) == cudaSuccess)
        out->event_ms[li] = ms;
    }
  }
  if (out->aborted) {
    for (uint32_t li = 0; li < h->n_local; ++li) {
      const int rc = cdp::reset_ctrl_local(h, li);
      if (rc != CDPROBE_OK) {
        h->sticky = true;
        return rc;
      }
    }
    cdp::set_err("device watchdog fired (a peer did not reach a barrier within timeout_ms)");
    // In one process all ranks share the run counter and the handle stays usable.  Across processes
    // the peers' counters may have diverged: the handle must be reopened.
    if (h->cfg.world_size > 1) h->sticky = true;
    return CDPROBE_ERR_TIMEOUT;
  }
  return CDPROBE_OK;
}

int cdprobe_gather(cdprobe_t* h, cdprobe_result_t* inout) {
  if (h == nullptr || inout == nullptr) return CDPROBE_ERR_ARG;
  if (h->cfg.world_size <= 1) return CDPROBE_OK;
  std::vector<cdprobe_result_t> all(h->cfg.world_size);
  std::string err;
  if (h->rdv.allgather(inout, sizeof(cdprobe_result_t), all.data(), &err) != 0) {
    cdp::set_err(err);
    return CDPROBE_ERR_RENDEZVOUS;
  }
  for (uint32_t r = 0; r < h->cfg.world_size; ++r) {
    if (r == h->cfg.rank) continue;
    const cdprobe_result_t& o = all[r];
    for (uint32_t g = 0; g < h->n_total; ++g) {
      if (!((o.row_mask >> g) & 1u) || ((inout->row_mask >> g) & 1u)) continue;
      const size_t a = (size_t)g * CDPROBE_MAX_GPUS;
      memcpy(inout->reach_read + a, o.reach_read + a, CDPROBE_MAX_GPUS);
      memcpy(inout->reach_write + a, o.reach_write + a, CDPROBE_MAX_GPUS);
      memcpy(inout->gbps_read + a, o.gbps_read + a, CDPROBE_MAX_GPUS * sizeof(float));
      memcpy(inout->gbps_write + a, o.gbps_write + a, CDPROBE_MAX_GPUS * sizeof(float));
      memcpy(inout->status + a, o.status + a, CDPROBE_MAX_GPUS * sizeof(int32_t));
      memcpy(inout->sum_read + a, o.sum_read + a, CDPROBE_MAX_GPUS * sizeof(uint64_t));
      memcpy(inout->xor_read + a, o.xor_read + a, CDPROBE_MAX_GPUS * sizeof(uint64_t));
      memcpy(inout->sum_write + a, o.sum_write + a, CDPROBE_MAX_GPUS * sizeof(uint64_t));
      memcpy(inout->xor_write + a, o.xor_write + a, CDPROBE_MAX_GPUS * sizeof(uint64_t));
      inout->row_mask |= 1u << g;
    }
    if (!o.verdict) inout->verdict = 0;
    if (o.aborted) inout->aborted = 1;
    inout->unreachable_pairs += o.unreachable_pairs;
    inout->slow_pairs += o.slow_pairs;
    if (o.min_gbps_read > 0.f && (inout->min_gbps_read == 0.f || o.min_gbps_read < inout->min_gbps_read))
      inout->min_gbps_read = o.min_gbps_read;
    if (o.min_gbps_write > 0.f && (inout->min_gbps_write == 0.f || o.min_gbps_write < inout->min_gbps_write))
      inout->min_gbps_write = o.min_gbps_write;
    if (o.probe_ms > inout->probe_ms) inout->probe_ms = o.probe_ms;
  }
  return CDPROBE_OK;
}

int cdprobe_info(cdprobe_t* h, cdprobe_info_t* out) {
  if (h == nullptr || out == nullptr) return CDPROBE_ERR_ARG;
  memset(out, 0, sizeof(*out));
  out->abi = CDPROBE_ABI_VERSION;
  out->n = h->n_total;
  out->n_local = h->n_local;
  out->first_local_rank = h->first;
  for (uint32_t li = 0; li < h->n_local; ++li) {
    const cdp::LocalRank& L = h->lr[li];
    out->ordinal[li] = L.ordinal;
    out->sm_count[li] = (uint32_t)L.sm_count;
    out->ctas[li] = L.ctas;
    out->mig[li] = L.mig ? 1u : 0u;
    memcpy(out->uuid[li], L.uuid, sizeof(out->uuid[li]));
    for (uint32_t s = 0; s < h->plan.n_slices; ++s) {
      out->src_sum[li][s] = h->src_sum[li][s];
      out->src_xor[li][s] = h->src_xor[li][s];
    }
  }
  out->handle_type = h->handle_type;
  out->path = h->path;
  out->bytes_per_pair = h->plan.bpp;
  out->alloc_bytes = h->plan.alloc_bytes;
  out->n_slices = h->plan.n_slices;
  out->smem_bytes = cdp::kSmemBytes;
  out->open_ms = h->open_ms;
  out->fill_ms = h->fill_ms;
  return CDPROBE_OK;
}

int cdprobe_trace(cdprobe_t* h, uint32_t local, cdprobe_trace_t* out) {
  if (h == nullptr || out == nullptr || local >= h->n_local) return CDPROBE_ERR_ARG;
  memset(out, 0, sizeof(*out));
  out->abi = CDPROBE_ABI_VERSION;
  const cdp::LocalRank& L = h->lr[local];
  const cdp::ResultRow* row = L.row;
  out->n_phases = L.n_phases;
  const uint64_t t0 = row->t_first;
  auto rel = [&](uint64_t t) { return t > t0 ? t - t0 : 0ull; };
  for (uint32_t p = 0; p < L.n_phases; ++p) {
    const cdp::PhaseOut& o = row->ph[p];
    out->kind0[p] = L.phases[p].job[0].kind;
    out->kind1[p] = L.phases[p].job[1].kind;
    out->peer0[p] = L.phases[p].job[0].peer;
    out->peer1[p] = L.phases[p].job[1].peer;
    out->sync_mask[p] = (uint16_t)(L.phases[p].sync_mask & L.peer_mask);
    out->post_mask[p] = (uint16_t)(L.phases[p].post_mask & L.peer_mask);
    out->sync_all[p] = (uint8_t)(L.peer_mask != 0 && (L.phases[p].sync_mask & L.peer_mask) == L.peer_mask);
    out->t_start[p] = rel(o.t_start);
    out->t_end0[p] = rel(o.t_end[0]);
    out->t_end1[p] = rel(o.t_end[1]);
    out->t_arrive[p] = rel(o.t_arrive);
  }
  return CDPROBE_OK;
}

int cdprobe_set_option(cdprobe_t* h, uint32_t option, uint64_t value) {
  if (h == nullptr) return CDPROBE_ERR_ARG;
  switch (option) {
    case CDPROBE_OPT_EVENT_TIMING:
      h->event_timing = value != 0;
      return CDPROBE_OK;
    case CDPROBE_OPT_CTAS:
      for (uint32_t li = 0; li < h->n_local; ++li) {
        cdp::LocalRank& L = h->lr[li];
        uint32_t c = value ? (uint32_t)value : (uint32_t)L.sm_count;
        if (c > (uint32_t)L.max_ctas) c = (uint32_t)L.max_ctas;
        L.ctas = c;
      }
      return cdp::rebuild_all(h);
    case CDPROBE_OPT_PATH:
      if (value > 2) return CDPROBE_ERR_ARG;
      h->path = (uint32_t)value;
      return CDPROBE_OK;
    case CDPROBE_OPT_TIMEOUT_MS:
      if (value == 0 || value > 600000) return CDPROBE_ERR_ARG;
      h->cfg.timeout_ms = (uint32_t)value;
      return CDPROBE_OK;
    case CDPROBE_OPT_OVERLAP_VERIFY:
    {
      const uint32_t old = h->cfg.flags;
      h->cfg.flags = (h->cfg.flags & ~CDPROBE_FLAG_OVERLAP_VERIFY) | (value ? CDPROBE_FLAG_OVERLAP_VERIFY : 0u);
      const int rc = cdp::rebuild_all(h);
      if (rc != CDPROBE_OK) {
        h->cfg.flags = old;
        cdp::rebuild_all(h);
      }
      return rc;
    }
    case CDPROBE_OPT_UNIDIRECTIONAL:
    {
      const uint32_t old = h->cfg.flags;
      h->cfg.flags = (h->cfg.flags & ~CDPROBE_FLAG_UNIDIRECTIONAL) | (value ? CDPROBE_FLAG_UNIDIRECTIONAL : 0u);
      const int rc = cdp::rebuild_all(h);
      if (rc != CDPROBE_OK) {
        h->cfg.flags = old;
        cdp::rebuild_all(h);
      }
      return rc;
    }
    case CDPROBE_OPT_ALL_RANK_BARRIERS:
    {
      const uint32_t old = h->cfg.flags;
      h->cfg.flags = (h->cfg.flags & ~CDPROBE_FLAG_ALL_RANK_BARRIERS) | (value ? CDPROBE_FLAG_ALL_RANK_BARRIERS : 0u);
      const int rc = cdp::rebuild_all(h);
      if (rc != CDPROBE_OK) {
        h->cfg.flags = old;
        cdp::rebuild_all(h);
      }
      return rc;
    }
    case CDPROBE_OPT_PAIR_BARRIERS:
    {
      const uint32_t old = h->cfg.flags;
      h->cfg.flags = (h->cfg.flags & ~CDPROBE_FLAG_PAIR_BARRIERS) | (value ? CDPROBE_FLAG_PAIR_BARRIERS : 0u);
      const int rc = cdp::rebuild_all(h);
      if (rc != CDPROBE_OK) {
        h->cfg.flags = old;
        cdp::rebuild_all(h);
      }
      return rc;
    }
    case CDPROBE_OPT_CTAS_RANK:
    {
      const uint32_t li = (uint32_t)(value >> 16), c = (uint32_t)(value & 0xffffu);
      if (li == 0 || li > h->n_local || c == 0) return CDPROBE_ERR_ARG;
      cdp::LocalRank& L = h->lr[li - 1];
      L.ctas = c > (uint32_t)L.max_ctas ? (uint32_t)L.max_ctas : c;
      return cdp::rebuild_all(h);
    }
    case CDPROBE_OPT_MIN_FRACTION_PPM:
      if (value > 100000000ull) return CDPROBE_ERR_ARG;
      h->cfg.min_fraction = (float)((double)value / 1e6);
      return CDPROBE_OK;
    case CDPROBE_OPT_LINK_PEAK_MBPS:
      if (value > 100000000000ull) return CDPROBE_ERR_ARG;
      h->cfg.link_peak_gbps = (float)((double)value / 1e3);
      return CDPROBE_OK;
    case CDPROBE_OPT_SOLO_RANK:
      if (value > h->n_local || h->cfg.world_size > 1) return CDPROBE_ERR_ARG;
      h->solo_rank = (uint32_t)value;
      return CDPROBE_OK;
    case CDPROBE_OPT_DEBUG_SKIP_RANK:
      if (value > h->n_local) return CDPROBE_ERR_ARG;
      h->debug_skip_rank = (uint32_t)value;
      return CDPROBE_OK;
    case CDPROBE_OPT_WARMUP:
      if (value > 2) return CDPROBE_ERR_ARG;
      h->warm_mode = (uint32_t)value;
      return CDPROBE_OK;
    case CDPROBE_OPT_WARMUP_BYTES:
      h->warm_bytes = value / 128 * 128;
      return CDPROBE_OK;
    case CDPROBE_OPT_DEBUG_DAMAGE_WRITE:
    {
      if (value == 0) {
        h->damage_write = 0;
        return CDPROBE_OK;
      }
      const uint64_t li = value >> 16, target = (value >> 8) & 0xffu, code = value & 0xffu;
      if (li == 0 || li > h->n_local || target >= h->n_total || code < 1 || code > 4) return CDPROBE_ERR_ARG;
      if (target == h->lr[li - 1].grank && !h->plan.diag) return CDPROBE_ERR_ARG;  // no write job into itself
      h->damage_write = (uint32_t)value;
      return CDPROBE_OK;
    }
    case CDPROBE_OPT_VERIFY_CTAS:
      if (value == 0 || value > 65535) return CDPROBE_ERR_ARG;
      h->verify_ctas = (uint32_t)value;
      return cdp::rebuild_all(h);
    default:
      return CDPROBE_ERR_ARG;
  }
}

int cdprobe_unmap_peer(cdprobe_t* h, uint32_t local, uint32_t peer) {
  if (h == nullptr || local >= h->n_local || peer >= h->n_total) return CDPROBE_ERR_ARG;
  if (h->cfg.world_size > 1) return CDPROBE_ERR_UNSUPPORTED;  // peers would not learn about it
  const uint32_t g = h->lr[local].grank;
  if (peer == g) return CDPROBE_ERR_ARG;
  cdp::unmap_peer(h, local, peer);
  h->status[g][peer] = cdp::kStatusUnmapped;
  return cdp::rebuild_all(h);
}

int cdprobe_remap_peer(cdprobe_t* h, uint32_t local, uint32_t peer) {
  if (h == nullptr || local >= h->n_local || peer >= h->n_total) return CDPROBE_ERR_ARG;
  const uint32_t g = h->lr[local].grank;
  if (peer == g) return CDPROBE_ERR_ARG;
  if (h->sticky) return CDPROBE_ERR_STATE;
  cdp::unmap_peer(h, local, peer);
  const int32_t st = cdp::map_peer(h, local, peer);
  if (st != 0 && h->cfg.world_size > 1) {
    // the other processes build their phase tables from the mapping status exchanged at open and would
    // not learn that this pair is gone: the domain has to be reopened
    h->sticky = true;
    cdp::set_err("re-mapping a peer failed in a multi-process domain: " + h->drv.error_name((CUresult)st));
    return CDPROBE_ERR_CUDA;
  }
  h->status[g][peer] = st;
  const int rc = cdp::rebuild_all(h);
  if (rc != CDPROBE_OK) return rc;
  return st == 0 ? CDPROBE_OK : CDPROBE_ERR_CUDA;
}

int cdprobe_corrupt(cdprobe_t* h, uint32_t local, uint64_t byte_offset, uint64_t xor_mask) {
  if (h == nullptr || local >= h->n_local) return CDPROBE_ERR_ARG;
  if (byte_offset % 8 != 0 || byte_offset + 8 > h->plan.src_bytes) return CDPROBE_ERR_ARG;
  cdp::LocalRank& L = h->lr[local];
  CDP_RT(cudaSetDevice(L.ordinal));
  uint8_t* p = reinterpret_cast<uint8_t*>(L.va[L.grank]) + h->plan.src_off + byte_offset;
  uint64_t w = 0;
  CDP_RT(cudaMemcpyAsync(&w, p, 8, cudaMemcpyDeviceToHost, L.stream));
  CDP_RT(cudaStreamSynchronize(L.stream));
  w ^= xor_mask;
  CDP_RT(cudaMemcpyAsync(p, &w, 8, cudaMemcpyHostToDevice, L.stream));
  CDP_RT(cudaStreamSynchronize(L.stream));
  return CDPROBE_OK;
}

int cdprobe_peek(cdprobe_t* h, uint32_t local, uint64_t byte_offset, uint64_t bytes, void* out) {
  if (h == nullptr || out == nullptr || local >= h->n_local || bytes == 0) return CDPROBE_ERR_ARG;
  const uint64_t alloc = h->plan.alloc_bytes;
  if (byte_offset > alloc || bytes > alloc - byte_offset) return CDPROBE_ERR_ARG;  // no overflow in offset + bytes
  if (h->sticky) return CDPROBE_ERR_STATE;
  cdp::LocalRank& L = h->lr[local];
  CDP_RT(cudaSetDevice(L.ordinal));
  const uint8_t* p = reinterpret_cast<const uint8_t*>(L.va[L.grank]) + byte_offset;
  CDP_RT(cudaMemcpyAsync(out, p, bytes, cudaMemcpyDeviceToHost, L.stream));
  CDP_RT(cudaStreamSynchronize(L.stream));
  return CDPROBE_OK;
}

int cdprobe_ce_copy(cdprobe_t* h, uint32_t n_copies, const uint32_t* local, const uint32_t* peer, uint32_t push,
                    uint64_t bytes, uint32_t reps, double* ms_out) {
  cdp::g_last_error.clear();
  if (h == nullptr || local == nullptr || peer == nullptr || ms_out == nullptr || n_copies == 0 ||
      n_copies > h->n_local || reps == 0 || reps > 1024)
    return CDPROBE_ERR_ARG;
  if (h->sticky) return CDPROBE_ERR_STATE;
  const cdp::Plan& pl = h->plan;
  uint64_t nb = bytes;
  if (nb == 0 || nb > pl.src_bytes) nb = pl.src_bytes;
  if (nb > pl.land_bytes) nb = pl.land_bytes;
  for (uint32_t k = 0; k < n_copies; ++k) {
    if (local[k] >= h->n_local || peer[k] >= h->n_total) return CDPROBE_ERR_ARG;
    for (uint32_t q = 0; q < k; ++q)
      if (local[q] == local[k]) return CDPROBE_ERR_ARG;  // one copy per local rank: each has one stream and event pair
    const cdp::LocalRank& L = h->lr[local[k]];
    if (!L.mapped[peer[k]]) {
      cdp::set_err("peer is not mapped into this rank's address space");
      return CDPROBE_ERR_STATE;
    }
  }
  for (uint32_t k = 0; k < n_copies; ++k) {
    cdp::LocalRank& L = h->lr[local[k]];
    CDP_RT(cudaSetDevice(L.ordinal));
    const uint8_t* mine = reinterpret_cast<const uint8_t*>(L.va[L.grank]);
    const uint8_t* theirs = reinterpret_cast<const uint8_t*>(L.va[peer[k]]);
    const void* src = push ? mine + pl.src_off : theirs + pl.src_off;
    void* dst = const_cast<uint8_t*>(push ? theirs : mine) + pl.land_off;
    CDP_RT(cudaEventRecord(L.ev0, L.stream));
    for (uint32_t r = 0; r < reps; ++r) CDP_RT(cudaMemcpyAsync(dst, src, nb, cudaMemcpyDeviceToDevice, L.stream));
    CDP_RT(cudaEventRecord(L.ev1, L.stream));
  }
  for (uint32_t k = 0; k < n_copies; ++k) {
    cdp::LocalRank& L = h->lr[local[k]];
    CDP_RT(cudaSetDevice(L.ordinal));
    CDP_RT(cudaEventSynchronize(L.ev1));
    float ms = 0.f;
    CDP_RT(cudaEventElapsedTime(&ms, L.ev0, L.ev1));
    ms_out[k] = ms;
  }
  return CDPROBE_OK;
}

int cdprobe_gate(const cdprobe_config_t* cfg, uint32_t n_total, float* gate_read_gbps, float* gate_write_gbps) {
  if (cfg == nullptr || gate_read_gbps == nullptr || gate_write_gbps == nullptr) return CDPROBE_ERR_ARG;
  if (cfg->abi != CDPROBE_ABI_VERSION) return CDPROBE_ERR_ABI;
  if (cfg->link_peak_gbps < 0.f || cfg->min_fraction < 0.f) return CDPROBE_ERR_ARG;
  cdp::Plan pl;
  const int rc = cdp::make_plan(n_total, cfg->bytes, cfg->mode, cfg->flags, &pl);
  if (rc != CDPROBE_OK) return rc;
  *gate_read_gbps = cdp::gate_gbps_for(*cfg, n_total, pl.bpp, true);
  *gate_write_gbps = cdp::gate_gbps_for(*cfg, n_total, pl.bpp, false);
  return CDPROBE_OK;
}

void cdprobe_close(cdprobe_t* h) { cdp::destroy(h); }

}  // extern "C"
