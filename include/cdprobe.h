/*
 * cdprobe.h — C ABI of libcdprobe.so: the ComputeDomain fabric-validation probe.
 *
 * This is the drop-in boundary for the compute-domain-daemon's domain-ready
 * gate.  The reference's gate is `check()` in
 *   cmd/compute-domain-daemon/main.go:435-459
 * (exec `nvidia-imex-ctl -q`, compare stdout with "READY\n"; a no-op when
 * CLIQUE_ID is empty, main.go:436-439).  The reference has no NVLink probe
 * (SURVEY.md F1); the functions below are what a Go shim `pkg/fabricprobe`
 * binds over cgo (see INTEGRATION.md) so that `run()` (main.go:212-347) can
 * execute an all-pairs NVLink reachability + bandwidth probe on the GPUs the
 * daemon owns and `check()` can consult its verdict.
 *
 * Rules of the ABI (SURVEY.md §8b):
 *   - plain C, fixed-width integers, caller-allocated outputs, no pointers
 *     cross back except the opaque handle;
 *   - 0 = ok, <0 = cdprobe error enum (below); the CUDA/driver status that
 *     caused a CDPROBE_ERR_CUDA is available from cdprobe_last_error();
 *   - the library never prints and never aborts (klog owns stdout/stderr in
 *     the daemon: cmd/compute-domain-daemon/process.go:92-96);
 *   - a handle is not thread-safe; distinct handles are independent;
 *   - there is NO CPU fallback: without a CUDA driver + sm_100 device
 *     cdprobe_open() fails with CDPROBE_ERR_NO_DEVICE / _UNSUPPORTED.
 *
 * All integer results (reachability bits, checksums, schedule) are exact;
 * GB/s values are measurements (run-to-run tolerance +-2 %, north_star).
 */
#ifndef CDPROBE_H_
#define CDPROBE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CDPROBE_API __attribute__((visibility("default")))
#else
#define CDPROBE_API
#endif

#define CDPROBE_ABI_VERSION 2u         /* 2: neighbourhood barriers (sync_mask), calibrated gate, ce_copy */
#define CDPROBE_MAX_GPUS 16          /* ranks in one probe domain (8 on HGX B200) */
#define CDPROBE_MAX_PHASES 64
#define CDPROBE_NVLINK_MAX_LINKS 18  /* == NVML_NVLINK_MAX_LINKS (nvml.h:389) */

/* Error enum (return values). */
#define CDPROBE_OK 0
#define CDPROBE_ERR_ABI (-1)         /* abi field mismatch */
#define CDPROBE_ERR_ARG (-2)         /* invalid argument / config */
#define CDPROBE_ERR_NO_DEVICE (-3)   /* no CUDA driver, or no usable GPU */
#define CDPROBE_ERR_CUDA (-4)        /* a CUDA call failed; see cdprobe_last_error */
#define CDPROBE_ERR_TIMEOUT (-5)     /* timeout_ms expired (device or host watchdog) */
#define CDPROBE_ERR_RENDEZVOUS (-6)  /* multi-process handle exchange failed */
#define CDPROBE_ERR_NOMEM (-7)
#define CDPROBE_ERR_UNSUPPORTED (-8) /* device lacks VMM / cooperative launch / sm_100 */
#define CDPROBE_ERR_STATE (-9)       /* handle unusable after a sticky CUDA error */
#define CDPROBE_ERR_INTEGRITY (-10)  /* self-check of published checksums failed */

/* cdprobe_config_t.mode — SURVEY.md §8(d) "Modes & algorithmic bytes". */
#define CDPROBE_MODE_REACH_ONLY 0u   /* 64 KiB per ordered pair: latency floor */
#define CDPROBE_MODE_SLICED 1u       /* bytes_per_pair = floor(B/(N-1)/128)*128 */
#define CDPROBE_MODE_FULL 2u         /* bytes_per_pair = B */

/* cdprobe_config_t.ops */
#define CDPROBE_OP_READ 1u           /* rank i loads peer j's slice, checksums it */
#define CDPROBE_OP_WRITE 2u          /* rank i stores a pattern into peer j; j verifies */

/* cdprobe_config_t.flags */
#define CDPROBE_FLAG_FABRIC_HANDLES 0x01u  /* CU_MEM_HANDLE_TYPE_FABRIC when /dev/nvidia-caps-imex-channels/channel0 opens */
#define CDPROBE_FLAG_MIG_AWARE 0x02u       /* MIG devices: skip peer mapping, identity matrix (SURVEY H8) */
#define CDPROBE_FLAG_LOCAL_DIAG 0x04u      /* also measure the diagonal (loop-back into local HBM; always on when n == 1) */
#define CDPROBE_FLAG_PATH_LDST 0x08u       /* 128-bit ld/st.global instead of TMA bulk copies */
#define CDPROBE_FLAG_NO_COOPERATIVE 0x10u  /* plain launch (tests that put 2 ranks on one device) */
#define CDPROBE_FLAG_OVERLAP_VERIFY 0x20u  /* verify landing slots on spare CTAs while the next round runs (default) */
#define CDPROBE_FLAG_SIMULATE_MIG 0x200u   /* treat every local GPU as a MIG instance (BASELINE config 4 without MIG hardware) */
#define CDPROBE_FLAG_SERIAL_VERIFY 0x100u  /* opt out of the overlapped verify: verify every slot after the rounds */
#define CDPROBE_FLAG_ALLOW_SAME_DEVICE 0x40u /* several ranks may name the same CUDA ordinal (testing) */
#define CDPROBE_FLAG_ALL_RANK_BARRIERS 0x400u /* every tournament phase closes with an all-rank flag exchange (round-1
                                              behaviour); default: only the ranks whose traffic shares an NVLink
                                              port with this rank's in the two phases either side of the barrier */
#define CDPROBE_FLAG_PAIR_BARRIERS 0x800u  /* keep the pair's flag exchange between the write and the read phase of a round
                                              (default: no wait there — the rank only signals its partner and the
                                              verify job waits for that signal itself) */
#define CDPROBE_FLAG_UNIDIRECTIONAL 0x80u  /* each round in two halves: one rank of a pair issues at a time, so a
                                              port carries payload one way only (per-link figure; 2x the phases) */

typedef struct cdprobe cdprobe_t;

typedef struct {
  uint32_t abi;                         /* CDPROBE_ABI_VERSION */
  uint32_t n_gpus;                      /* GPUs driven by THIS process; 0 = all visible */
  int32_t ordinals[CDPROBE_MAX_GPUS];   /* CUDA ordinals; ignored when n_gpus == 0 */
  uint64_t bytes;                       /* B: per-GPU probe buffer (1 GiB for the headline config) */
  uint32_t mode;                        /* CDPROBE_MODE_* */
  uint32_t ops;                         /* CDPROBE_OP_* bits; 0 = read|write */
  uint32_t timeout_ms;                  /* device + host watchdog; 0 = 5000 */
  uint32_t flags;                       /* CDPROBE_FLAG_* */
  uint64_t seed;                        /* 0 = 0xCD5EED0000000001 */
  float min_fraction;                   /* verdict threshold on pair GB/s, as a fraction of the reference figure below;
                                           0 = default (0.90 with the calibrated reference, see link_peak_gbps) */
  float link_peak_gbps;                 /* reference figure of the gate.
                                           0 (default) = CALIBRATED: what a healthy B200 NVLink-5 port delivers to
                                           SM-issued traffic of that op and schedule, measured next to the copy engine
                                           on the same box (profiles/r02_linkbench_n2.jsonl: both directions loaded,
                                           reads 672 / writes 703 GB/s; one way, reads 785 / writes 714.7 — SM stores
                                           cap there on every store shape and CTA count; the copy engine moves
                                           773-778), de-rated for the ~8 us a phase spends ramping and draining:
                                               expected(bytes_per_pair) = bytes_per_pair / (bytes_per_pair / rate + 8 us)
                                           >0 = absolute: threshold = min_fraction x link_peak_gbps (900 = nominal
                                           NVLink 5 per direction; the north_star's "0.85 x 900 = 765" is above what
                                           any SM write and any bidirectional transfer reaches on healthy hardware) */
  uint32_t ctas;                        /* CTAs of the persistent kernel; 0 = one per SM */
  uint32_t world_size;                  /* processes in the probe domain; 0/1 = single process */
  uint32_t rank;                        /* this process's index in [0, world_size) */
  uint32_t reserved0;
  char session[64];                     /* rendezvous name shared by all processes (world_size > 1) */
} cdprobe_config_t;

/* Matrices are row-major [issuer * CDPROBE_MAX_GPUS + target], issuer = the
 * rank whose SMs issue the loads (read) or stores (write).  A process fills
 * the rows of its local ranks (row_mask); cdprobe_gather() completes them. */
typedef struct {
  uint32_t abi;
  uint32_t n;                           /* total ranks in the domain */
  uint32_t row_mask;                    /* bit r set: row r is filled in */
  uint32_t verdict;                     /* 1: every filled off-diagonal cell reachable and >= min_fraction */
  uint8_t reach_read[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS];
  uint8_t reach_write[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS];
  float gbps_read[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS];
  float gbps_write[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS];
  int32_t status[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS]; /* 0 ok; <0 CDPROBE_ERR_*; >0 CUresult of the mapping */
  uint64_t sum_read[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS];  /* checksum S the issuer computed (parity tests) */
  uint64_t xor_read[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS];  /* checksum X */
  uint64_t sum_write[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS]; /* checksum of the pattern the issuer generated */
  uint64_t xor_write[CDPROBE_MAX_GPUS * CDPROBE_MAX_GPUS];
  uint64_t bytes_per_pair;
  uint64_t run_seq;                     /* 1-based count of cdprobe_run on this handle */
  uint32_t rounds;                      /* tournament rounds (N-1 for even N) */
  uint32_t phases;                      /* device phases executed */
  uint32_t launches;                    /* kernels launched by this call (one per local rank) */
  uint32_t aborted;                     /* 1: a device watchdog fired */
  uint32_t warmed;                      /* 1: this run streamed the link wake-up prefix (phase 0) */
  uint32_t reserved1;
  double probe_ms;                      /* host wall clock of this cdprobe_run call */
  double device_ms[CDPROBE_MAX_GPUS];   /* per local rank: first barrier release -> last arrive (%globaltimer) */
  double barrier_us[CDPROBE_MAX_GPUS];  /* per local rank: sum of (release - arrive) over all barriers */
  double event_ms[CDPROBE_MAX_GPUS];    /* per local rank: kernel duration by CUDA events on the launch stream
                                           (only with CDPROBE_OPT_EVENT_TIMING; 0 otherwise) */
  float min_gbps_read;                  /* over filled off-diagonal cells (diagonal when n == 1) */
  float min_gbps_write;
  float gate_gbps_read;                 /* the GB/s threshold this run's verdict applied to reads (0: bandwidth not judged) */
  float gate_gbps_write;
  double kernel_ms[CDPROBE_MAX_GPUS];   /* per local rank: CTA 0 entering the kernel -> result row published (%globaltimer);
                                           event_ms - kernel_ms = launch and completion latency outside the kernel,
                                           kernel_ms - device_ms = residency barrier before the first phase + row output */
  uint32_t unreachable_pairs;           /* filled off-diagonal cells with reach_read & reach_write == 0 (MIG-excluded cells not counted) */
  uint32_t slow_pairs;                  /* filled off-diagonal cells that are reachable but under the gate */
} cdprobe_result_t;

typedef struct {
  uint32_t abi;
  uint32_t n;                           /* total ranks */
  uint32_t n_local;
  uint32_t first_local_rank;
  int32_t ordinal[CDPROBE_MAX_GPUS];    /* per local rank */
  uint32_t sm_count[CDPROBE_MAX_GPUS];
  uint32_t ctas[CDPROBE_MAX_GPUS];
  uint32_t mig[CDPROBE_MAX_GPUS];
  char uuid[CDPROBE_MAX_GPUS][48];      /* "GPU-xxxxxxxx-xxxx-xxxx-xxxx-xxxxxxxxxxxx" per local rank */
  uint32_t handle_type;                 /* 0 none (in-process), 1 POSIX fd, 8 fabric */
  uint32_t path;                        /* 0 TMA bulk, 1 ld/st */
  uint64_t bytes_per_pair;
  uint64_t alloc_bytes;                 /* HBM per rank */
  uint64_t src_sum[CDPROBE_MAX_GPUS][CDPROBE_MAX_GPUS]; /* [local rank][slice]: device-computed checksum S of the source slices */
  uint64_t src_xor[CDPROBE_MAX_GPUS][CDPROBE_MAX_GPUS];
  uint32_t n_slices;
  uint32_t smem_bytes;
  double open_ms;                       /* contexts + VMM + mapping */
  double fill_ms;                       /* pattern fill + slice checksums */
} cdprobe_info_t;

/* Plan (host-only arithmetic; usable without a GPU). */
typedef struct {
  uint32_t abi;
  uint32_t n;
  uint32_t rounds;
  uint32_t n_slots;                     /* landing slots per rank */
  uint32_t n_slices;                    /* source slices per rank */
  uint32_t reserved;
  uint64_t bytes_per_pair;
  uint64_t src_bytes;
  uint64_t land_bytes;
  int8_t partner[CDPROBE_MAX_GPUS][CDPROBE_MAX_GPUS]; /* [round][rank], -1 = idle */
} cdprobe_plan_t;

/* Per-phase timeline of the last run of one local rank (ns, relative to the first barrier release). */
typedef struct {
  uint32_t abi;
  uint32_t n_phases;
  uint8_t kind0[CDPROBE_MAX_PHASES], kind1[CDPROBE_MAX_PHASES];  /* 0 none, 1 read, 2 write, 3 verify, 4 warm-up */
  int8_t peer0[CDPROBE_MAX_PHASES], peer1[CDPROBE_MAX_PHASES];
  uint8_t sync_all[CDPROBE_MAX_PHASES];                          /* closing barrier spans all ranks */
  uint16_t sync_mask[CDPROBE_MAX_PHASES];                        /* ranks of the closing barrier's flag exchange */
  uint16_t post_mask[CDPROBE_MAX_PHASES];                        /* ranks only signalled at the closing barrier (no wait) */
  uint64_t t_start[CDPROBE_MAX_PHASES];                          /* opening barrier released */
  uint64_t t_end0[CDPROBE_MAX_PHASES], t_end1[CDPROBE_MAX_PHASES]; /* last CTA of job 0 / job 1 done */
  uint64_t t_arrive[CDPROBE_MAX_PHASES];                         /* every local CTA reached the closing barrier */
} cdprobe_trace_t;

/* The phase table of one rank (host-only; what cdprobe_run hands to that rank's kernel when every pair is mapped). */
typedef struct {
  uint32_t abi;
  uint32_t n_phases;
  uint32_t peer_mask;                              /* ranks in this rank's cross-GPU barrier */
  uint32_t reserved;
  uint8_t kind[2][CDPROBE_MAX_PHASES];             /* [job][phase]: 0 none, 1 read, 2 write, 3 verify, 4 warm-up */
  int8_t peer[2][CDPROBE_MAX_PHASES];              /* rank whose memory the job touches */
  uint8_t slot[2][CDPROBE_MAX_PHASES];             /* landing slot (write/verify) or source slice (read/warm) */
  uint8_t writer[2][CDPROBE_MAX_PHASES];           /* verify: the rank that wrote the slot */
  uint16_t cta0[2][CDPROBE_MAX_PHASES], nctas[2][CDPROBE_MAX_PHASES];
  uint8_t sync_all[CDPROBE_MAX_PHASES];            /* closing barrier spans all ranks */
  uint16_t sync_mask[CDPROBE_MAX_PHASES];          /* ranks this rank exchanges flags with when the phase closes */
  uint16_t post_mask[CDPROBE_MAX_PHASES];          /* ranks it only signals then (no wait) */
  uint8_t wait_barrier[2][CDPROBE_MAX_PHASES];     /* [job][phase] verify jobs: 1-based barrier index whose signal from
                                                      `writer` the job waits for before reading the slot (0 = none) */
} cdprobe_schedule_t;

/* Node topology as NVML reports it (no CUDA; internal/common topology enumeration, SURVEY §8f n2). */
typedef struct {
  uint32_t abi;
  uint32_t n;                                     /* GPUs NVML enumerates, in NVML index order */
  char uuid[CDPROBE_MAX_GPUS][96];                /* nvmlDeviceGetUUID */
  char pci_bus_id[CDPROBE_MAX_GPUS][32];
  uint8_t mig[CDPROBE_MAX_GPUS];                  /* MIG mode currently enabled */
  uint8_t links_active[CDPROBE_MAX_GPUS];         /* NvLinkState == ENABLED over the 18 links */
  uint32_t link_mask[CDPROBE_MAX_GPUS];           /* bit l set: link l is ENABLED (which physical link is down, not only how many) */
  uint8_t fabric_state[CDPROBE_MAX_GPUS];         /* nvmlGpuFabricInfo_t.state */
  char clique_id[96];                             /* "<clusterUUID>.<cliqueId>" or "" (nvlib.go:208-363) */
  char clique_error[160];                         /* non-empty: getCliqueID would return this error */
} cdprobe_topology_t;

CDPROBE_API uint32_t cdprobe_abi_version(void);
CDPROBE_API const char* cdprobe_strerror(int code);
/* Detail of the last failure on the calling thread ("cuMemMap: CUDA_ERROR_..."), "" if none. */
CDPROBE_API const char* cdprobe_last_error(void);

/* Entry points and the reference interface each one extends or stands in for (paths relative to
 * NVIDIA/k8s-dra-driver-gpu @ 2240711):
 *
 *   cdprobe_open      once per daemon process, from run():          cmd/compute-domain-daemon/main.go:212-347
 *                     (also in the cliqueID == "" branch, main.go:244-250, which today only blocks on ctx)
 *   cdprobe_run       the probe pass; at start and on every daemon-set change delivered by
 *                     GetDaemonInfoUpdateChan():                    cmd/compute-domain-daemon/controller.go:137-139,
 *                     update loops main.go:351-431.  Its verdict is what check() consults next to the IMEX gate:
 *                                                                   cmd/compute-domain-daemon/main.go:435-459
 *   cdprobe_close     on ctx cancel, before the child is stopped:   cmd/compute-domain-daemon/main.go:87-102
 *   cdprobe_topology  NVML device walk + clique id, replaces the ad-hoc walk of getCliqueIDStrict/Legacy:
 *                                                                   cmd/compute-domain-kubelet-plugin/nvlib.go:195-363,
 *                     vendor/github.com/NVIDIA/go-nvlib/pkg/nvlib/device/device.go:268-310,464-495
 *   cdprobe_strerror / cdprobe_last_error   text of the Go error:   fmt.Errorf convention of main.go
 *   cdprobe_remap_peer / cdprobe_unmap_peer  emulate NodeUnprepare/NodePrepare churn around a live domain:
 *                                                                   cmd/compute-domain-kubelet-plugin/driver.go:165-232
 *   cdprobe_gather, cdprobe_info, cdprobe_trace, cdprobe_set_option, cdprobe_corrupt, cdprobe_peek, cdprobe_plan,
 *   cdprobe_schedule, cdprobe_gate, cdprobe_ce_copy, cdprobe_rendezvous_selftest: diagnostics, benches, fault injection; the reference has
 *   no counterpart (it has no probe, SURVEY.md F1).
 */
CDPROBE_API int cdprobe_open(const cdprobe_config_t* cfg, cdprobe_t** out);
CDPROBE_API int cdprobe_run(cdprobe_t* h, cdprobe_result_t* out);
/* Collective over all processes of the domain: completes rows of other processes. No-op for world_size <= 1. */
CDPROBE_API int cdprobe_gather(cdprobe_t* h, cdprobe_result_t* inout);
CDPROBE_API int cdprobe_info(cdprobe_t* h, cdprobe_info_t* out);
CDPROBE_API int cdprobe_trace(cdprobe_t* h, uint32_t local, cdprobe_trace_t* out);
/* Runtime options (no reopen needed; the bench sweeps them). */
#define CDPROBE_OPT_EVENT_TIMING 1u  /* value 0/1: bracket each kernel with CUDA events, report event_ms */
#define CDPROBE_OPT_CTAS 2u          /* CTAs of the persistent kernel (0 = one per SM) */
#define CDPROBE_OPT_PATH 3u          /* 0 = TMA bulk copies, 1 = ld/st.global.v4 (128-bit), 2 = ld/st.global.v8 (256-bit) */
#define CDPROBE_OPT_TIMEOUT_MS 4u
#define CDPROBE_OPT_OVERLAP_VERIFY 5u /* value 0/1 */
#define CDPROBE_OPT_VERIFY_CTAS 6u   /* CTAs given to the overlapped verify (default 32) */
#define CDPROBE_OPT_UNIDIRECTIONAL 7u /* value 0/1: see CDPROBE_FLAG_UNIDIRECTIONAL */
#define CDPROBE_OPT_WARMUP 8u        /* link wake-up phase: 0 never, 1 auto = after > 5 ms idle (default), 2 always */
#define CDPROBE_OPT_DEBUG_SKIP_RANK 10u /* fault injection: 1-based local rank whose kernel is not launched (0 = off) */
#define CDPROBE_OPT_WARMUP_BYTES 9u  /* bytes each rank streams from its first partner when warming (default 8 MiB, capped at bytes_per_pair) */
#define CDPROBE_OPT_CTAS_RANK 11u    /* value = ((local rank + 1) << 16) | ctas: CTA count of ONE local rank (tests: a throttled issuer) */
#define CDPROBE_OPT_MIN_FRACTION_PPM 12u /* min_fraction x 1e6 (0 = default) */
#define CDPROBE_OPT_LINK_PEAK_MBPS 13u   /* link_peak_gbps x 1e3 (0 = calibrated reference) */
#define CDPROBE_OPT_SOLO_RANK 14u    /* profiling: 1-based local rank that runs ALONE — only its own read/write jobs, no
                                        cross-GPU barrier, nobody verifies its writes (reach_write stays 0).  A single
                                        self-contained kernel is what `ncu` can replay: NVLink byte counters per launch. */
#define CDPROBE_OPT_ALL_RANK_BARRIERS 15u /* value 0/1: see CDPROBE_FLAG_ALL_RANK_BARRIERS */
#define CDPROBE_OPT_PAIR_BARRIERS 16u     /* value 0/1: see CDPROBE_FLAG_PAIR_BARRIERS */
#define CDPROBE_OPT_DEBUG_DAMAGE_WRITE 17u /* fault injection: value = ((local rank + 1) << 16) | (target rank << 8) | code,
                                              0 = off.  In every run while set, once that local rank's write job into
                                              `target`'s landing slot is over and before anyone is told so, the kernel
                                              damages the slot (the writer's own checksum stays that of the clean
                                              pattern): 1 = flip bit 0 of the first word (S and X change); 2 = flip
                                              bit 63 of the last word; 3 = add 0x9E3779B97F4A7C15 to the first word
                                              and subtract it from the last (S unchanged, only X sees it); 4 = swap words
                                              0 and 1 (S and X unchanged: a blind spot of the checksum, the verify
                                              passes).  ERR_ARG for a bad local rank, a target past the domain or
                                              the rank itself when the diagonal is not probed, or a code outside
                                              1..4. */
CDPROBE_API int cdprobe_set_option(cdprobe_t* h, uint32_t option, uint64_t value);
/* Copy-engine reference on the probe's own buffers (the same-box ceiling the roofline is quoted against; not part
 * of a probe): copy k moves `bytes` (capped at the source / landing size) `reps` times back to back between local
 * rank local[k] and rank peer[k] — push != 0: local source -> peer landing area, else peer source -> local landing
 * area — on local[k]'s stream.  All n_copies are enqueued before any is waited for (bidirectional: two copies in
 * one call, or one call per process after a host barrier).  ms_out[k] = CUDA-event time of copy k's `reps` copies. */
CDPROBE_API int cdprobe_ce_copy(cdprobe_t* h, uint32_t n_copies, const uint32_t* local, const uint32_t* peer, uint32_t push,
                                uint64_t bytes, uint32_t reps, double* ms_out);
/* Storm/unprepare emulation (SURVEY H10): unmap + remap rank `peer` in local rank `local`'s address space. */
CDPROBE_API int cdprobe_remap_peer(cdprobe_t* h, uint32_t local, uint32_t peer);
/* Fault injection for parity tests: drop local rank's mapping of `peer` (cell becomes unreachable, run still returns). */
CDPROBE_API int cdprobe_unmap_peer(cdprobe_t* h, uint32_t local, uint32_t peer);
/* Fault injection: XOR one 64-bit word of local rank's source buffer (`byte_offset` from the start of the source). */
CDPROBE_API int cdprobe_corrupt(cdprobe_t* h, uint32_t local, uint64_t byte_offset, uint64_t xor_mask);
/* Diagnostics: copy `bytes` from local rank `local`'s own probe allocation, starting `byte_offset` bytes from its
 * base (Ctrl at 0, source at 2 MiB, landing slots after the source rounded up to 2 MiB; DESIGN §4), into `out`.
 * Ordered after everything enqueued on that rank's stream (a finished cdprobe_run). Never reads outside the allocation. */
CDPROBE_API int cdprobe_peek(cdprobe_t* h, uint32_t local, uint64_t byte_offset, uint64_t bytes, void* out);
CDPROBE_API void cdprobe_close(cdprobe_t* h);

/* Host-only helpers (no CUDA): schedule + slice arithmetic; the fd/blob rendezvous self-test. */
CDPROBE_API int cdprobe_plan(uint32_t n, uint64_t bytes, uint32_t mode, uint32_t flags, cdprobe_plan_t* out);
/* strict != 0: getCliqueIDStrict (feature gate CrashOnNVLinkFabricErrors, default on), else the legacy walk. */
CDPROBE_API int cdprobe_topology(uint32_t strict, cdprobe_topology_t* out);
CDPROBE_API int cdprobe_schedule(uint32_t n, uint32_t rank, uint64_t bytes, uint32_t mode, uint32_t ops, uint32_t flags,
                                 uint32_t ctas, uint32_t verify_ctas, cdprobe_schedule_t* out);
CDPROBE_API int cdprobe_rendezvous_selftest(const char* session, uint32_t rank, uint32_t world, uint32_t timeout_ms);
/* The GB/s gate cdprobe_run would apply to reads / writes for this configuration in an n-rank domain (0: bandwidth is
 * not judged — reach-only mode, n == 1).  Host-only arithmetic: lets a caller log or test the threshold without a GPU. */
CDPROBE_API int cdprobe_gate(const cdprobe_config_t* cfg, uint32_t n_total, float* gate_read_gbps, float* gate_write_gbps);

#ifdef __cplusplus
}
#endif
#endif /* CDPROBE_H_ */
