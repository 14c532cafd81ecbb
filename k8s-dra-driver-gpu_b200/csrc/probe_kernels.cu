// probe_kernels.cu — sm_100a kernels of the ComputeDomain fabric probe.
//
// K1 read probe   : every warp streams 8 KiB units of a peer's source slice
//                   into shared memory with 1-D TMA bulk copies
//                   (cp.async.bulk.shared::cluster.global + mbarrier complete_tx,
//                   3 stages in flight per warp) or with 128-/256-bit
//                   ld.global loads, and folds them into the (S, X) checksum.
// K2 write probe  : every warp generates the write pattern into shared memory
//                   and pushes it into the peer's landing slot with TMA bulk
//                   stores (cp.async.bulk.global.shared::cta) or st.global.v4/.v8.
// K3 barrier      : grid barrier (atomic arrive / release word) whose last
//                   arriver runs the cross-GPU flag exchange with the ranks the
//                   phase table names (at most four between rounds, nobody between
//                   the write and the read of a round, everybody at open/close):
//                   publish, one fence.sys only if something was published,
//                   pipelined st.relaxed.sys epochs into those peers' Ctrl,
//                   ld.acquire.sys on the local copy.
// K4 verify/local : the read probe pointed at local HBM (landing slots, source
//                   slices at open, the N = 1 loop-back).
//
// One persistent cooperative kernel per GPU runs every phase of a probe
// (wake-up, tournament rounds x {write, read + overlapped verify}) so a run
// costs one launch per GPU; phases are timed with %globaltimer on the issuing
// GPU (SURVEY.md H7).  The phase table comes from schedule.cc.
//
// The reference has no kernel for this path (SURVEY.md F1/F3); the gate it
// implements is cmd/compute-domain-daemon/main.go:435-459.
#include <cuda_runtime.h>
#include <stdint.h>

#include "probe_launch.h"
#include "probe_types.h"

namespace cdp {
namespace {

// ------------------------------------------------------------------ PTX ----
__device__ __forceinline__ uint64_t gtimer() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void st_release_sys(uint64_t* p, uint64_t v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_acquire_sys(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint64_t ld_relaxed_sys(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// 1-D TMA bulk load: global (local HBM or NVLink peer) -> this CTA's shared memory.
__device__ __forceinline__ void bulk_load(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
// 1-D TMA bulk store: shared memory -> global (local HBM or NVLink peer).
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_smem), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 128-bit streaming load (coherent at L2; L1 is not polluted). Not .nc: the
// verify job reads data a peer wrote earlier in the same kernel.
__device__ __forceinline__ uint4 ldg_stream_v4(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p)
               : "memory");
  return r;
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void stg_v4(uint4* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}
struct U8 {
  uint32_t r[8];
};
// 256-bit global accesses (sm_100+: LDG.E.256 / STG.E.256) — 1 KiB contiguous per warp instruction.
__device__ __forceinline__ U8 ldg_v8(const void* p) {
  U8 v;
  asm volatile("ld.global.L1::no_allocate.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v.r[0]), "=r"(v.r[1]), "=r"(v.r[2]), "=r"(v.r[3]), "=r"(v.r[4]), "=r"(v.r[5]), "=r"(v.r[6]),
                 "=r"(v.r[7])
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ void stg_v8(void* p, const U8& v) {
  asm volatile("st.global.L1::no_allocate.v8.u32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v.r[0]),
               "r"(v.r[1]), "r"(v.r[2]), "r"(v.r[3]), "r"(v.r[4]), "r"(v.r[5]), "r"(v.r[6]), "r"(v.r[7])
               : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ uint64_t pack64(uint32_t lo, uint32_t hi) { return (uint64_t)lo | ((uint64_t)hi << 32); }

// ------------------------------------------------------------- context -----
struct Ctx {
  Ctrl* ctrl;
  uint64_t deadline;
  uint32_t stage_smem;   // shared address of this warp's stage 0
  uint32_t bar_smem;     // shared address of this warp's mbarrier 0
  uint32_t parity_bits;  // bit s: parity to wait for on stage s
  int warp, lane;
};

__device__ __forceinline__ bool aborted(const Ctx& c) {
  return *reinterpret_cast<volatile unsigned int*>(&c.ctrl->abort_flag) != 0u;
}
// Slow-path check used inside spin loops: watchdog + abort propagation.
__device__ __noinline__ bool check_abort(const Ctx& c) {
  if (aborted(c)) return true;
  if (gtimer() > c.deadline) {
    atomicExch(&c.ctrl->abort_flag, 1u);
    return true;
  }
  return false;
}

// Waits for the bulk load armed on `stage`.  Returns false when the run was aborted while waiting —
// the load is then STILL IN FLIGHT towards this CTA's shared memory and the caller must drain it
// (mbar_drain) before the CTA may exit or reuse the stage.
__device__ __forceinline__ bool mbar_wait(Ctx& c, int stage) {
  const uint32_t bar = c.bar_smem + 8u * stage;
  const uint32_t parity = (c.parity_bits >> stage) & 1u;
  uint32_t spins = 0;
  bool ok = true;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 255u) == 0u && check_abort(c)) {
      ok = false;
      break;
    }
  }
  // warp-uniform outcome: a lane that saw the phase complete while another saw the abort must not
  // flip its parity alone (mbar_drain re-waits the same phase; a completed one passes at once)
  if (!__all_sync(0xffffffffu, ok)) return false;
  c.parity_bits ^= (1u << stage);
  return true;
}
// After an abort: wait, without the watchdog, for a load that was already issued.  An abort means a PEER
// missed a barrier; the memory this load targets is mapped and the copy completes in microseconds.  If
// it has not after kDrainNs the fabric itself is gone: trap (sticky error on the context, reported by
// the host as a kernel failure) rather than let a bulk copy land in the shared memory of an exited CTA.
constexpr uint64_t kDrainNs = 200ull * 1000 * 1000;
__device__ __noinline__ void mbar_drain(Ctx& c, int stage) {
  const uint32_t bar = c.bar_smem + 8u * stage;
  const uint32_t parity = (c.parity_bits >> stage) & 1u;
  const uint64_t t_give_up = gtimer() + kDrainNs;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 1023u) == 0u && gtimer() > t_give_up) __trap();
  }
  c.parity_bits ^= (1u << stage);
}

// ------------------------------------------------------------ checksum -----
struct Sum {
  uint64_t s0, s1;  // two partial sums (ILP), folded at the end
  uint64_t x;       // position-folded xor
};

__device__ __forceinline__ void fold_unit(Sum& a, uint64_t unit_xor, uint64_t unit) {
  const uint32_t g = static_cast<uint32_t>(unit / (kGranuleBytes / kUnitBytes));
  a.x ^= rotl64(unit_xor, fold6(g));
}

// ------------------------------------------------------- K1/K4: reading ----
__device__ __forceinline__ void issue_load(const Ctx& c, const uint8_t* base, uint64_t bytes, uint64_t u, int stage) {
  const uint64_t off = u * kUnitBytes;
  const uint64_t left = bytes - off;
  const uint32_t n = left < kUnitBytes ? static_cast<uint32_t>(left) : kUnitBytes;
  const uint32_t bar = c.bar_smem + 8u * stage;
  mbar_arrive_expect_tx(bar, n);
  bulk_load(c.stage_smem + stage * kUnitBytes, base + off, n, bar);
}

__device__ void job_read_tma(Ctx& c, const uint8_t* base, uint64_t bytes, uint32_t gwarp, uint32_t nwarps, Sum& a) {
  const uint64_t n_units = (bytes + kUnitBytes - 1) / kUnitBytes;
  uint64_t u_issue = gwarp;
  uint32_t in_flight = 0;  // loads issued and not yet waited for (warp-uniform)
  if (c.lane == 0) fence_proxy_async_global();  // data may have been written through the generic proxy
#pragma unroll
  for (int s = 0; s < kStages; ++s) {
    if (u_issue < n_units) {
      if (c.lane == 0) issue_load(c, base, bytes, u_issue, s);
      u_issue += nwarps;
      ++in_flight;
    }
  }
  int s = 0;
  for (uint64_t u = gwarp; u < n_units; u += nwarps) {
    if (!mbar_wait(c, s)) {
      // aborted: stop issuing, but every load already in flight must land before this CTA can exit
      for (; in_flight > 0; --in_flight) {
        mbar_drain(c, s);
        s = (s + 1 == kStages) ? 0 : s + 1;
      }
      return;
    }
    --in_flight;
    const uint64_t left = bytes - u * kUnitBytes;
    const uint32_t nvec = (left < kUnitBytes ? static_cast<uint32_t>(left) : kUnitBytes) >> 4;
    const uint32_t sbase = c.stage_smem + s * kUnitBytes + c.lane * 16u;
    uint64_t ux = 0;
    if (nvec == kUnitBytes / 16) {
#pragma unroll
      for (int k = 0; k < (int)(kUnitBytes / 16 / 32); ++k) {
        const uint4 v = lds_v4(sbase + k * 512u);
        const uint64_t w0 = pack64(v.x, v.y), w1 = pack64(v.z, v.w);
        a.s0 += w0;
        a.s1 += w1;
        ux ^= w0 ^ w1;
      }
    } else {
      for (uint32_t i = c.lane; i < nvec; i += 32) {
        const uint4 v = lds_v4(c.stage_smem + s * kUnitBytes + i * 16u);
        const uint64_t w0 = pack64(v.x, v.y), w1 = pack64(v.z, v.w);
        a.s0 += w0;
        a.s1 += w1;
        ux ^= w0 ^ w1;
      }
    }
    fold_unit(a, ux, u);
    __syncwarp();
    if (u_issue < n_units) {
      if (c.lane == 0) {
        fence_proxy_async_smem();
        issue_load(c, base, bytes, u_issue, s);
      }
      u_issue += nwarps;
      ++in_flight;
    }
    s = (s + 1 == kStages) ? 0 : s + 1;
  }
}

__device__ void job_read_ldg(Ctx& c, const uint8_t* base, uint64_t bytes, uint32_t gwarp, uint32_t nwarps, Sum& a) {
  const uint64_t n_units = (bytes + kUnitBytes - 1) / kUnitBytes;
  for (uint64_t u = gwarp; u < n_units; u += nwarps) {
    const uint64_t left = bytes - u * kUnitBytes;
    const uint32_t nvec = (left < kUnitBytes ? static_cast<uint32_t>(left) : kUnitBytes) >> 4;
    const uint4* gp = reinterpret_cast<const uint4*>(base + u * kUnitBytes) + c.lane;
    uint4 v[kLdstVecs];
    if (nvec == kUnitBytes / 16) {
#pragma unroll
      for (int k = 0; k < (int)kLdstVecs; ++k) v[k] = ldg_stream_v4(gp + k * 32);
    } else {
#pragma unroll
      for (int k = 0; k < (int)kLdstVecs; ++k) {
        v[k] = make_uint4(0u, 0u, 0u, 0u);
        if (c.lane + k * 32u < nvec) v[k] = ldg_stream_v4(gp + k * 32);
      }
    }
    uint64_t ux = 0;
#pragma unroll
    for (int k = 0; k < (int)kLdstVecs; ++k) {
      const uint64_t w0 = pack64(v[k].x, v[k].y), w1 = pack64(v[k].z, v[k].w);
      a.s0 += w0;
      a.s1 += w1;
      ux ^= w0 ^ w1;
    }
    fold_unit(a, ux, u);
  }
}

__device__ void job_read_ldg256(Ctx& c, const uint8_t* base, uint64_t bytes, uint32_t gwarp, uint32_t nwarps, Sum& a) {
  const uint64_t n_units = (bytes + kUnitBytes - 1) / kUnitBytes;
  constexpr int kV = kUnitBytes / 32 / 32;  // 32-byte vectors per lane per full unit
  for (uint64_t u = gwarp; u < n_units; u += nwarps) {
    const uint64_t left = bytes - u * kUnitBytes;
    const uint32_t nvec = (left < kUnitBytes ? static_cast<uint32_t>(left) : kUnitBytes) >> 5;
    const uint8_t* gp = base + u * kUnitBytes + c.lane * 32u;
    U8 v[kV];
    if (nvec == kUnitBytes / 32) {
#pragma unroll
      for (int k = 0; k < kV; ++k) v[k] = ldg_v8(gp + k * 1024);
    } else {
#pragma unroll
      for (int k = 0; k < kV; ++k) {
#pragma unroll
        for (int q = 0; q < 8; ++q) v[k].r[q] = 0u;
        if (c.lane + k * 32u < nvec) v[k] = ldg_v8(gp + k * 1024);
      }
    }
    uint64_t ux = 0;
#pragma unroll
    for (int k = 0; k < kV; ++k) {
      const uint64_t w0 = pack64(v[k].r[0], v[k].r[1]), w1 = pack64(v[k].r[2], v[k].r[3]);
      const uint64_t w2 = pack64(v[k].r[4], v[k].r[5]), w3 = pack64(v[k].r[6], v[k].r[7]);
      a.s0 += w0 + w2;
      a.s1 += w1 + w3;
      ux ^= w0 ^ w1 ^ w2 ^ w3;
    }
    fold_unit(a, ux, u);
  }
}

// ---------------------------------------------------------- K2: writing ----
__device__ void job_write_tma(Ctx& c, uint8_t* base, uint64_t bytes, uint32_t gwarp, uint32_t nwarps, uint64_t salt,
                              Sum& a) {
  const uint64_t n_units = (bytes + kUnitBytes - 1) / kUnitBytes;
  uint32_t it = 0;
  int s = 0;
  for (uint64_t u = gwarp; u < n_units; u += nwarps, ++it) {
    if (it >= (uint32_t)kStages) {
      if (c.lane == 0) bulk_wait_read<kStages - 1>();  // the store that used stage s has drained it
    }
    __syncwarp();
    const uint64_t left = bytes - u * kUnitBytes;
    const uint32_t nb = left < kUnitBytes ? static_cast<uint32_t>(left) : kUnitBytes;
    const uint32_t nvec = nb >> 4;
    const uint32_t sbase = c.stage_smem + s * kUnitBytes;
    uint64_t z = (salt + u * (kUnitBytes / 8) + 2ull * c.lane) * kGolden;
    uint64_t ux = 0;
    for (uint32_t i = c.lane; i < nvec; i += 32) {
      const uint64_t z1 = z + kGolden;
      const uint64_t w0 = z ^ (z >> 32), w1 = z1 ^ (z1 >> 32);
      z += 64ull * kGolden;
      sts_v4(sbase + i * 16u, make_uint4((uint32_t)w0, (uint32_t)(w0 >> 32), (uint32_t)w1, (uint32_t)(w1 >> 32)));
      a.s0 += w0;
      a.s1 += w1;
      ux ^= w0 ^ w1;
    }
    fold_unit(a, ux, u);
    fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the async proxy
    __syncwarp();
    if (c.lane == 0) {
      bulk_store(base + u * kUnitBytes, sbase, nb);
      bulk_commit();
    }
    s = (s + 1 == kStages) ? 0 : s + 1;
  }
  if (c.lane == 0) bulk_wait_all();  // stores complete (not just smem drained)
  __syncwarp();
}

__device__ void job_write_stg(Ctx& c, uint8_t* base, uint64_t bytes, uint32_t gwarp, uint32_t nwarps, uint64_t salt,
                              Sum& a) {
  const uint64_t n_units = (bytes + kUnitBytes - 1) / kUnitBytes;
  for (uint64_t u = gwarp; u < n_units; u += nwarps) {
    const uint64_t left = bytes - u * kUnitBytes;
    const uint32_t nvec = (left < kUnitBytes ? static_cast<uint32_t>(left) : kUnitBytes) >> 4;
    uint4* gp = reinterpret_cast<uint4*>(base + u * kUnitBytes);
    uint64_t z = (salt + u * (kUnitBytes / 8) + 2ull * c.lane) * kGolden;
    uint64_t ux = 0;
#pragma unroll 4
    for (uint32_t i = c.lane; i < nvec; i += 32) {
      const uint64_t z1 = z + kGolden;
      const uint64_t w0 = z ^ (z >> 32), w1 = z1 ^ (z1 >> 32);
      z += 64ull * kGolden;
      stg_v4(gp + i, make_uint4((uint32_t)w0, (uint32_t)(w0 >> 32), (uint32_t)w1, (uint32_t)(w1 >> 32)));
      a.s0 += w0;
      a.s1 += w1;
      ux ^= w0 ^ w1;
    }
    fold_unit(a, ux, u);
  }
}

__device__ void job_write_stg256(Ctx& c, uint8_t* base, uint64_t bytes, uint32_t gwarp, uint32_t nwarps, uint64_t salt,
                                 Sum& a) {
  const uint64_t n_units = (bytes + kUnitBytes - 1) / kUnitBytes;
  for (uint64_t u = gwarp; u < n_units; u += nwarps) {
    const uint64_t left = bytes - u * kUnitBytes;
    const uint32_t nvec = (left < kUnitBytes ? static_cast<uint32_t>(left) : kUnitBytes) >> 5;
    uint8_t* gp = base + u * kUnitBytes;
    uint64_t z = (salt + u * (kUnitBytes / 8) + 4ull * c.lane) * kGolden;
    uint64_t ux = 0;
#pragma unroll 4
    for (uint32_t i = c.lane; i < nvec; i += 32) {
      U8 v;
      uint64_t zz = z;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint64_t w = zz ^ (zz >> 32);
        zz += kGolden;
        v.r[2 * q] = (uint32_t)w;
        v.r[2 * q + 1] = (uint32_t)(w >> 32);
        if (q & 1) a.s1 += w;
        else a.s0 += w;
        ux ^= w;
      }
      z += 128ull * kGolden;
      stg_v8(gp + (uint64_t)i * 32u, v);
    }
    fold_unit(a, ux, u);
  }
}

// ---------------------------------------------------------- K3: barrier ----
// Leader-only publications once every local CTA has finished a phase.
//  * a write job: (S, X, run_seq) of what was stored, into the owner's Ctrl, so that the owner can verify the
//    landing slot — must be visible before the flag that tells the owner "phase done";
//  * verify jobs: the verdict goes back to the writer.  Writers read it only when they assemble their result row,
//    after the last barrier of the run, so ALL verdicts are published by the last barrier's leader in one go (one
//    thread, one fence: no cross-thread ordering argument needed).
__device__ bool publish_writes(const ProbeParams& P, Ctrl* ctrl, int ph) {
  bool any = false;
#pragma unroll
  for (int jb = 0; jb < 2; ++jb) {
    const Job job = P.phase[ph].job[jb];
    if (job.kind != kJobWrite) continue;
    const volatile Acc* acc = &ctrl->acc[ph][jb];
    Ctrl* pc = reinterpret_cast<Ctrl*>(P.base_peer[job.peer]);
    st_relaxed_sys(&pc->wr[job.slot].sum, acc->sum);
    st_relaxed_sys(&pc->wr[job.slot].xr, acc->xr);
    st_relaxed_sys(&pc->wr[job.slot].seq, P.run_seq);
    any = true;
  }
  return any;
}
__device__ void publish_verdicts(const ProbeParams& P, Ctrl* ctrl) {
  for (uint32_t ph = 0; ph < P.n_phases; ++ph) {
#pragma unroll
    for (int jb = 0; jb < 2; ++jb) {
      const Job job = P.phase[ph].job[jb];
      if (job.kind != kJobVerify) continue;
      const volatile Acc* acc = &ctrl->acc[ph][jb];
      const uint64_t wsum = ld_relaxed_sys(&ctrl->wr[job.slot].sum);
      const uint64_t wxr = ld_relaxed_sys(&ctrl->wr[job.slot].xr);
      const uint64_t wseq = ld_relaxed_sys(&ctrl->wr[job.slot].seq);
      uint64_t code = kVerdictNotWritten;
      if (wseq == P.run_seq) code = (wsum == acc->sum && wxr == acc->xr) ? kVerdictOk : kVerdictMismatch;
      uint8_t* wb = P.base_peer[job.writer];
      if (wb != nullptr) st_relaxed_sys(&reinterpret_cast<Ctrl*>(wb)->verdict[P.rank], P.run_seq * 4ull + code);
    }
  }
}

// Fault injection (CDPROBE_OPT_DEBUG_DAMAGE_WRITE): the host put a damage code into the `writer` byte of a write
// job (unused on write jobs).  The barrier leader that closes the job's phase applies it to the landing slot after
// every local CTA has arrived and before anything is published, released or signalled: the loop-back's diagonal
// verify starts as soon as the grid is released, a remote verify once this rank signals.  The writer's own (S, X)
// stays that of the clean pattern.
__device__ __noinline__ void damage_slot(const ProbeParams& P, const Job& job) {
  uint8_t* pb = P.base_peer[job.peer];
  if (pb == nullptr) return;
  // TMA-path stores came through the async proxy: order them before this thread's generic accesses
  fence_proxy_async_global();
  uint64_t* w = reinterpret_cast<uint64_t*>(pb + P.land_off + (uint64_t)job.slot * P.bpp);
  uint64_t* last = w + (P.bpp / 8 - 1);
  switch (job.writer) {
    case 1: st_relaxed_sys(w, ld_relaxed_sys(w) ^ 1ull); break;
    case 2: st_relaxed_sys(last, ld_relaxed_sys(last) ^ (1ull << 63)); break;
    case 3:
      st_relaxed_sys(w, ld_relaxed_sys(w) + kGolden);
      st_relaxed_sys(last, ld_relaxed_sys(last) - kGolden);
      break;
    case 4: {
      const uint64_t w0 = ld_relaxed_sys(w), w1 = ld_relaxed_sys(w + 1);
      st_relaxed_sys(w, w1);
      st_relaxed_sys(w + 1, w0);
      break;
    }
    default: break;
  }
  __threadfence_system();
}

__device__ __forceinline__ void signal_ranks(const ProbeParams& P, uint32_t mask, uint64_t target) {
  for (uint32_t j = 0; j < P.n_ranks; ++j) {
    if (j == P.rank || !((mask >> j) & 1u)) continue;
    st_relaxed_sys(&reinterpret_cast<Ctrl*>(P.base_peer[j])->flags[P.rank].v, target);
  }
}

// Barrier b: b == 0 opens the run, barrier b >= 1 closes phase b - 1.
//   sync = ranks to exchange flags with (signal, then wait): the ranks whose traffic touches the same NVLink ports
//          as this rank's in the phases either side of the barrier (schedule.cc: current partner, next partner and
//          their partners; every rank at open and close).  Symmetric: whoever is waited for also signals.
//   post = ranks that are only signalled, AFTER this rank's own CTAs have been released: the write -> read step
//          inside a round — nobody waits there; the verify job that needs the partner's data polls for it itself.
// A system-scope fence precedes the flag stores only when this rank published something the receiver acts on at
// this barrier (write checksums; the verdicts at the last barrier): reads leave nothing in flight, and each CTA
// already fenced its own remote stores before it arrived.
__device__ void barrier(const ProbeParams& P, Ctx& c, int b, uint32_t sync, uint32_t post, bool last) {
  __syncthreads();
  if (threadIdx.x == 0) {
    Ctrl* ctrl = c.ctrl;
    const bool ab = aborted(c);
    if (!ab) {
      const unsigned long long target = P.seq_base + (unsigned long long)b + 1ull;
      // This CTA's accumulator atomics precede the arrive.  Remote stores of a write job were already
      // fenced at system scope by this thread (see the job epilogue), so gpu scope is enough here.
      __threadfence();
      const unsigned int prev = atomicAdd(&ctrl->grid_arrive, 1u);
      if (prev == gridDim.x - 1) {
        // last arriver: every local CTA is done with the phase
        *reinterpret_cast<volatile unsigned int*>(&ctrl->grid_arrive) = 0u;
        __threadfence();
        const uint64_t t_arr = gtimer();
        if (b >= 1) {
#pragma unroll
          for (int jb = 0; jb < 2; ++jb) {
            const Job& job = P.phase[b - 1].job[jb];
            if (job.kind == kJobWrite && job.writer != 0) damage_slot(P, job);
          }
        }
        bool published = false, wrote_done = false;
        if (sync) {
          if (b >= 1) {
            published = publish_writes(P, ctrl, b - 1);
            wrote_done = true;
          }
          if (last) {
            publish_verdicts(P, ctrl);
            published = true;
          }
          if (published) __threadfence_system();  // one fence, then relaxed flag stores that pipeline over NVLink
          signal_ranks(P, sync, target);
          bool timed_out = false;
          for (uint32_t j = 0; j < P.n_ranks && !timed_out; ++j) {
            if (j == P.rank || !((sync >> j) & 1u)) continue;
            uint32_t spins = 0;
            while (ld_acquire_sys(&ctrl->flags[j].v) < target) {
              if ((++spins & 63u) == 0u && check_abort(c)) {
                timed_out = true;
                break;
              }
            }
          }
        } else if (last) {
          publish_verdicts(P, ctrl);  // single-rank domains: the verdict word is local
          __threadfence_system();
        }
        const uint64_t t_rel = gtimer();
        ctrl->t_arr[b] = t_arr;
        ctrl->t_rel[b] = t_rel;
        st_release_gpu(&ctrl->grid_release, target);
        // off the critical path: the local CTAs are already running the next phase
        if (post && !aborted(c)) {
          if (b >= 1 && !wrote_done) publish_writes(P, ctrl, b - 1);
          __threadfence_system();
          signal_ranks(P, post, target);
        } else if (b >= 1 && !wrote_done && !aborted(c)) {
          if (publish_writes(P, ctrl, b - 1)) __threadfence_system();  // loop-back write: the owner is this GPU
        }
      } else {
        uint32_t spins = 0;
        while (ld_acquire_gpu(&ctrl->grid_release) < target) {
          if ((++spins & 63u) == 0u && check_abort(c)) break;
        }
      }
    }
  }
  __syncthreads();
}

__device__ __forceinline__ uint64_t warp_sum64(uint64_t v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}
__device__ __forceinline__ uint64_t warp_xor64(uint64_t v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v ^= __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

}  // namespace

// ------------------------------------------------- the persistent kernel ----
__global__ void __launch_bounds__(kThreads, 1) cdprobe_kernel(const __grid_constant__ ProbeParams P) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWarpsPerCta * kStages * kUnitBytes);
  uint64_t* red = bars + kWarpsPerCta * kStages;  // [kWarpsPerCta][2]
  __shared__ uint64_t s_deadline;

  Ctx c;
  c.ctrl = reinterpret_cast<Ctrl*>(P.base_peer[P.rank]);
  c.warp = threadIdx.x >> 5;
  c.lane = threadIdx.x & 31;
  c.stage_smem = smem_u32(smem) + c.warp * kStages * kUnitBytes;
  c.bar_smem = smem_u32(bars) + c.warp * kStages * 8u;
  c.parity_bits = 0u;
  __shared__ uint64_t s_enter;
  if (threadIdx.x == 0) {
    s_enter = gtimer();
    s_deadline = s_enter + P.timeout_ns;
  }
  if (c.lane == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) mbar_init(c.bar_smem + 8u * s, 1u);
    fence_mbar_init();
  }
  __syncthreads();
  c.deadline = s_deadline;

  barrier(P, c, 0, P.peer_mask, 0u, false);

  for (uint32_t ph = 0; ph < P.n_phases; ++ph) {
    const Phase& phd = P.phase[ph];
#pragma unroll
    for (int jb = 0; jb < 2; ++jb) {
      const Job job = phd.job[jb];
      if (job.kind == kJobNone) continue;
      if (blockIdx.x < job.cta0 || blockIdx.x >= (uint32_t)job.cta0 + job.nctas) continue;
      Sum a{0ull, 0ull, 0ull};
      if (!aborted(c)) {
        const uint32_t gwarp = (blockIdx.x - job.cta0) * kWarpsPerCta + c.warp;
        const uint32_t nwarps = (uint32_t)job.nctas * kWarpsPerCta;
        uint8_t* pb = P.base_peer[job.peer];
        if (job.kind == kJobWarm) {
          // untimed link wake-up: stream a prefix of the partner's slice (result ignored)
          const uint8_t* src = pb + P.src_off + (P.full_mode ? 0ull : (uint64_t)job.slot * P.bpp);
          const uint64_t nb = job.salt < P.bpp ? job.salt : P.bpp;
          if (nb) {
            if (P.use_ldst == 2u) job_read_ldg256(c, src, nb, gwarp, nwarps, a);
            else if (P.use_ldst == 1u) job_read_ldg(c, src, nb, gwarp, nwarps, a);
            else job_read_tma(c, src, nb, gwarp, nwarps, a);
          }
        } else if (job.kind == kJobRead) {
          const uint8_t* src = pb + P.src_off + (P.full_mode ? 0ull : (uint64_t)job.slot * P.bpp);
          if (P.use_ldst == 2u) job_read_ldg256(c, src, P.bpp, gwarp, nwarps, a);
          else if (P.use_ldst == 1u) job_read_ldg(c, src, P.bpp, gwarp, nwarps, a);
          else job_read_tma(c, src, P.bpp, gwarp, nwarps, a);
        } else if (job.kind == kJobVerify) {
          // the slot's writer signals when its write phase is over (and its checksums are published); where the
          // schedule put no wait between that phase and this one (post_mask), this job does the waiting
          bool go = true;
          if (job.salt != 0 && job.writer != P.rank && P.base_peer[job.writer] != nullptr) {
            if (threadIdx.x == 0) {
              const uint64_t need = P.seq_base + job.salt + 1ull;
              uint32_t spins = 0;
              while (ld_acquire_sys(&c.ctrl->flags[job.writer].v) < need) {
                if ((++spins & 63u) == 0u && check_abort(c)) break;
              }
            }
            __syncthreads();
            go = !aborted(c);
          }
          if (go) {
            const uint8_t* src = pb + P.land_off + (uint64_t)job.slot * P.bpp;
            if (P.use_ldst == 2u) job_read_ldg256(c, src, P.bpp, gwarp, nwarps, a);
            else if (P.use_ldst == 1u) job_read_ldg(c, src, P.bpp, gwarp, nwarps, a);
            else job_read_tma(c, src, P.bpp, gwarp, nwarps, a);
          }
        } else {
          uint8_t* dst = pb + P.land_off + (uint64_t)job.slot * P.bpp;
          if (P.use_ldst == 2u) job_write_stg256(c, dst, P.bpp, gwarp, nwarps, job.salt, a);
          else if (P.use_ldst == 1u) job_write_stg(c, dst, P.bpp, gwarp, nwarps, job.salt, a);
          else job_write_tma(c, dst, P.bpp, gwarp, nwarps, job.salt, a);
        }
      }
      // CTA reduce -> one atomic per CTA into the phase accumulator
      const uint64_t ws = warp_sum64(a.s0 + a.s1);
      const uint64_t wx = warp_xor64(a.x);
      if (c.lane == 0) {
        red[c.warp * 2 + 0] = ws;
        red[c.warp * 2 + 1] = wx;
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        uint64_t ts = 0, tx = 0;
#pragma unroll
        for (int w = 0; w < kWarpsPerCta; ++w) {
          ts += red[w * 2 + 0];
          tx ^= red[w * 2 + 1];
        }
        Acc* acc = &c.ctrl->acc[ph][jb];
        atomicAdd(&acc->sum, (unsigned long long)ts);
        atomicXor(&acc->xr, (unsigned long long)tx);
        if (job.kind == kJobWrite) __threadfence_system();  // stores have reached the peer
        atomicMax(&acc->t_end, (unsigned long long)gtimer());
      }
    }
    barrier(P, c, (int)ph + 1, phd.sync_mask & P.peer_mask, phd.post_mask & P.peer_mask, ph + 1 == P.n_phases);
  }

  // ---- output: CTA 0 writes the result row into pinned host memory ----------
  if (blockIdx.x == 0) {
    Ctrl* ctrl = c.ctrl;
    ResultRow* row = P.row;
    const bool ab = aborted(c);
    const uint32_t t = threadIdx.x;
    if (t < P.n_phases) {
      PhaseOut o;
      o.t_start = *reinterpret_cast<volatile uint64_t*>(&ctrl->t_rel[t]);
      o.t_arrive = *reinterpret_cast<volatile uint64_t*>(&ctrl->t_arr[t + 1]);
#pragma unroll
      for (int jb = 0; jb < 2; ++jb) {
        const Job job = P.phase[t].job[jb];
        const volatile Acc* acc = &ctrl->acc[t][jb];
        o.t_end[jb] = acc->t_end;
        o.sum[jb] = acc->sum;
        o.xr[jb] = acc->xr;
        o.exp_sum[jb] = 0;
        o.exp_xr[jb] = 0;
        o.verdict[jb] = 0;
        o.code[jb] = job.kind == kJobNone ? kCodeSkipped : (ab ? kCodeAborted : kCodeOk);
        if (!ab) {
          if (job.kind == kJobRead) {
            const Ctrl* pc = reinterpret_cast<const Ctrl*>(P.base_peer[job.peer]);
            const uint32_t slice = P.full_mode ? 0u : job.slot;
            o.exp_sum[jb] = ld_relaxed_sys(&pc->src_sum[slice]);
            o.exp_xr[jb] = ld_relaxed_sys(&pc->src_xor[slice]);
          } else if (job.kind == kJobVerify) {
            o.exp_sum[jb] = ld_relaxed_sys(&ctrl->wr[job.slot].sum);
            o.exp_xr[jb] = ld_relaxed_sys(&ctrl->wr[job.slot].xr);
            o.verdict[jb] = ld_relaxed_sys(&ctrl->wr[job.slot].seq);
          } else if (job.kind == kJobWrite) {
            o.verdict[jb] = ld_relaxed_sys(&ctrl->verdict[job.peer]);
          }
        }
      }
      row->ph[t] = o;
    }
    __syncthreads();
    // reset the accumulators for the next run
    if (t < P.n_phases) {
#pragma unroll
      for (int jb = 0; jb < 2; ++jb) {
        Acc* acc = &ctrl->acc[t][jb];
        acc->sum = 0ull;
        acc->xr = 0ull;
        acc->t_end = 0ull;
      }
    }
    // The row lives in pinned host memory.  One release at system scope by thread 0 publishes it: the other
    // threads' stores are ordered before it through the CTA barrier (cumulativity), so no per-thread
    // fence.sys — each one is a round trip over PCIe (round 1 had three of them here: ~5 us per run, 512 -> 507 us at N = 1).
    __syncthreads();
    if (t == 0) {
      row->t_first = *reinterpret_cast<volatile uint64_t*>(&ctrl->t_rel[0]);
      row->t_last = *reinterpret_cast<volatile uint64_t*>(&ctrl->t_arr[P.n_phases]);
      row->aborted = ab ? 1u : 0u;
      row->n_phases = P.n_phases;
      row->t_enter = s_enter;
      row->t_exit = gtimer();
      st_release_sys(const_cast<uint64_t*>(&row->done), P.run_seq);
    }
  }
}

// ------------------------------------------------------- source pattern ----
__global__ void __launch_bounds__(256) cdprobe_fill_src_kernel(uint4* dst, uint64_t nvec, uint64_t seed, uint32_t rank) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += stride) {
    const uint64_t w0 = src_word(seed, rank, 2 * v), w1 = src_word(seed, rank, 2 * v + 1);
    dst[v] = make_uint4((uint32_t)w0, (uint32_t)(w0 >> 32), (uint32_t)w1, (uint32_t)(w1 >> 32));
  }
}

// ----------------------------------------------------------- launchers -----
int probe_kernel_prepare(int* max_ctas_per_sm) {
  cudaError_t e = cudaFuncSetAttribute(cdprobe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
  if (e != cudaSuccess) return (int)e;
  int nb = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, cdprobe_kernel, kThreads, kSmemBytes);
  if (e != cudaSuccess) return (int)e;
  if (max_ctas_per_sm) *max_ctas_per_sm = nb;
  return 0;
}

int probe_kernel_launch(const ProbeParams* p, unsigned grid, bool cooperative, cudaStream_t stream) {
  void* args[] = {const_cast<ProbeParams*>(p)};
  cudaError_t e;
  if (cooperative) {
    e = cudaLaunchCooperativeKernel((const void*)cdprobe_kernel, dim3(grid), dim3(kThreads), args, kSmemBytes, stream);
  } else {
    e = cudaLaunchKernel((const void*)cdprobe_kernel, dim3(grid), dim3(kThreads), args, kSmemBytes, stream);
  }
  return (int)e;
}

int probe_fill_launch(void* dst, uint64_t bytes, uint64_t seed, uint32_t rank, unsigned grid, cudaStream_t stream) {
  cdprobe_fill_src_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<uint4*>(dst), bytes / 16, seed, rank);
  return (int)cudaGetLastError();
}

}  // namespace cdp
