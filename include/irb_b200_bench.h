/*
 * irb_b200_bench.h -- MEASUREMENT AIDS of libirb_b200.so.  NOT part of the drop-in boundary (that is irb_b200.h): nothing
 * here stands for a reference interface, and nothing in the product path calls it.  bench.py, bench_configs.py and the
 * A/B tests use these entry points to time kernels in isolation, to select the other form of a kernel, and to measure
 * the platform's ceilings (HBM read stream, host<->device copies) that the engine's numbers are held against.
 * Implemented in irbaboon_b200/csrc/irb_benchaids.cu, a translation unit of its own.
 */
#ifndef IRB_B200_BENCH_H
#define IRB_B200_BENCH_H

#include <stddef.h>
#include "irb_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Launch-policy knobs (irbaboon_b200/csrc/irb_tuning.hpp) by name: "mac_persistent", "fuse_split", "mac_tma", "mac_wide", "mac_u",
 * "fdl_plain", "producer_sleep_ns", "no_graph", "deconv_sub", "deconv_streams", "release_fence", "release_dep", "persistent_ctas", "unit_narrowing", "ir_replicas", "stagger_ns", "ring_stages".
 * The library itself never reads the environment; the defaults are compiled in.  _get returns the value (or IRB_ERR_ARG). */
int irbx_set_tuning(const char* name, int value);
int irbx_get_tuning(const char* name);

/* The pure FDL multiply-accumulate of the engine's current state (no forward / inverse FFT) into a device buffer of
 * n_channels * M complex: times the roofline kernel's inner loop in isolation. */
int irbx_engine_mac_only_device(irb_engine* e, float* acc_dev);
/* Phase time stamps of the latency-path kernel (k_mac_slots): with a device array of 64 x 16 uint64 set, thread 0 of CTA b < 64
 * stores at [16 b + phase] the %globaltimer (ns) at kernel start, after the set-up, after the forward transform, after the partition loop, before and after
 * each cluster barrier and at the end.  NULL switches it off (the default). */
int irbx_engine_set_stamps(irb_engine* e, unsigned long long* stamps_dev);
/* identical copies of the IR spectra the engine keeps (the h_reps the block steps read and every IR load writes) */
int irbx_engine_ir_copies(const irb_engine* e);
/* With the same pointer set (at least 4096 x 4 uint64), the persistent block-step kernel k_mac_p logs per launch, at
 * [4 (launch % 4096) + {0,1,2,3}], CTA 0's {%globaltimer at start, SM cycle counter at start, %globaltimer at end, cycle counter at end}:
 * cycles / ns is the SM clock the step ran at. */

/* GB/s of a kernel that does nothing but read `bytes` of device memory once per iteration with 32-byte streaming loads
 * (L1 no-allocate, L2 evict-first), grid = resident CTAs; averaged over `iters` launches after one warm-up: the read-only
 * ceiling an FDL stream can be held against (the roofline's `peak` stays the driver-measured copy bandwidth).
 * write_every = n > 0: every n-th 16 KB piece is written instead of read; store_kind: 0 plain, 1 .cs, 2 L2 evict-first
 * hint, 3 .wt, 4 .cg, 5 L2 evict-last hint. */
int irbx_hbm_read_probe(size_t bytes, int iters, int write_every, int store_kind, double* gbs);

/* Copy-only host<->device ceiling: what the platform gives the engine's host-buffer path when no kernel runs.
 * _create allocates `bytes` of host memory per direction (host_mode 0: cudaMallocHost; 1: input write-combined; 2: anonymous
 * mmap with transparent-huge-page advice, cudaHostRegister'ed) and the matching device buffers on `device`.
 * _run times `iters` rounds of: direction 1 = H2D only, 2 = D2H only, 3 = both at once on two streams, every transfer cut
 * into pieces of chunk_bytes (0: one piece), and returns the wall seconds of the whole call (one process = one GPU; the caller
 * aggregates over ranks between barriers). */
typedef struct irbx_copy_probe irbx_copy_probe;
int irbx_copy_probe_create(irbx_copy_probe** out, int device, size_t bytes, int host_mode);
int irbx_copy_probe_run(irbx_copy_probe* p, int iters, int direction, size_t chunk_bytes, double* seconds);
int irbx_copy_probe_destroy(irbx_copy_probe* p);

#ifdef __cplusplus
}
#endif
#endif /* IRB_B200_BENCH_H */
