// irb_kernels.cuh -- sm_100a kernels of the partitioned-convolution (UPOLA) block step.
//
// One CTA owns a TILE of 2048 packed complex bins = ROWS = 2048/M whole spectra ("rows": one stream-channel
// in the streaming engine, one output block in the offline functions).  256 compute threads work in two
// layouts over the same 16 KB of shared memory:
//   * FFT layout : M/8 threads per row, 8 complex points each (irb_fft.cuh);
//   * MAC layout : each thread owns V float4 (= 2V bins) of K rows, K*V = 4; in the streaming kernels the float4 come in
//                  adjacent pairs read with one 32-byte load, so that one warp instruction reads 1 KB of a
//                  frequency-domain delay line (FDL) row (MacLayout).
// A 9th warp is the TMA producer that streams impulse-response partition spectra into a shared-memory
// ring (cp.async.bulk + mbarrier), so every row of the tile -- every stream sharing that IR -- reuses them.
//
// Reference loops replaced (paths relative to /root/reference):
//   k_fwd       fp/convolution.cpp:106-125 (IR partition load + FFT), :128-149 (audio block load + FFT),
//               Source/PluginProcessor.cpp:430-436,455-461 (incl. the round-robin IR refresh rows)
//   k_mac_tma   the streaming block step of shared-IR tiles in ONE launch (FFT half sizes >= 256): k_fwd's work for the tile's new
//               blocks, then fp/convolution.cpp:160-215 / Source/PluginProcessor.cpp:480-510 with the FDL slots AND the IR
//               partitions streamed by TMA into a 3-stage shared-memory ring, inverse FFT, overlap-add
//   k_mac       the same loop with the FDL staged through registers (coalesced 16- / 32-byte loads): offline form, two-launch
//               streaming form, small FFT sizes; with FUSE also k_fwd's work (the A/B partner of k_mac_tma)
//   k_mac_slots the same loop when there are so few rows that each row's partitions are split over tile slots and the CTAs of a
//               thread-block cluster (the latency path; with the fused step cluster rank 0 runs the forward transform itself)
//   k_mac_p     (irb_mac_p.cuh) the persistent block step: shared-IR tiles and per-stream IRs, one launch per step
//   k_ola_tail  fp/convolution.cpp:210-213 for the offline (all blocks at once) formulation
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "irb_fft.cuh"

namespace irb {

constexpr int kThreads = 256;          // compute threads per CTA
constexpr int kTile = 2048;            // packed complex bins per CTA tile (16 KB)
constexpr int kStages = 4;             // IR ring stages

template <int M> struct Tile {
    static constexpr int V = M > 512 ? M / 512 : 1;      // float4 per thread per row
    static constexpr int TPR = M / (2 * V);              // MAC-layout threads per row
    static constexpr int G = kThreads / TPR;             // row groups
    static constexpr int K = 4 / V;                      // rows per MAC thread
    static constexpr int ROWS = kTile / M;               // rows per CTA (= G*K)
    static constexpr int TPF = M / kPts;                 // FFT-layout threads per row
};

// ---- PTX wrappers: named barrier, mbarrier, 1-D bulk TMA, streaming 128-bit load -----------------
__device__ __forceinline__ void bar_compute() { asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory"); }
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
// Consumer release of a TMA-filled stage.  `dep` is zero at run time but DERIVED FROM THE VALUES the warp read out of the stage
// (bits & MacArgs::zero), so the arrive cannot issue before those ld.shared have returned their data.  Without the
// dependency ptxas places the arrive right behind the last LDS; under load (three CTAs per SM, other CTAs in their FFT
// phases) that LDS was observed to execute AFTER the producer had seen the stage free and its next bulk copy had landed:
// one warp then multiplied partition g by the spectrum of partition g + kStages (profiles/r01_ring_release_race.md).
__device__ __forceinline__ void mbar_arrive_after(uint64_t* b, uint32_t dep) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b) + dep) : "memory");
}
// Orders this thread's earlier generic-proxy accesses to shared memory (the ld.shared of a ring stage) ahead of later
// async-proxy accesses (the bulk copy that refills the stage once it is released): issued by every lane before the warp's
// release of a TMA-filled stage.  mbar_arrive_after's data dependency stays as the second line of defence.
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ bool mbar_try_wait(uint64_t* b, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(smem_u32(b)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
    while (!mbar_try_wait(b, parity)) {}
}
// The producer runs kStages ahead and spends most of its life waiting for a free stage: sleeping between polls keeps its
// spin loop (a fifth of the kernel's instructions otherwise) off the issue ports and out of the power budget.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* b, uint32_t parity, int ns) {
    while (!mbar_try_wait(b, parity)) { if (ns) __nanosleep(ns); }
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// 32-byte streaming load (sm_100: LDG.E.NA.EFL2.256): read-once FDL data, not allocated in L1, first in line for L2 eviction
__device__ __forceinline__ void ldg_stream256(const float4* p, float4& a, float4& b) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(p));
}
// ---- sample formats of the streaming block step's audio rows (irb_sample_format in include/irb_b200.h) ----------------
// The new block a step reads (load_in) and the output block it writes (store_out) are float32, int16 or packed little-endian
// 24-bit integers; element i of a row sits at byte i * fmt_bytes(fmt).  Every access is one element wide (three single bytes
// for 24-bit), so any element-aligned pointer works.  The format is a launch argument, uniform over the launch.
constexpr int kFmtF32 = 0, kFmtS16 = 1, kFmtS24 = 2;
__host__ __device__ __forceinline__ int fmt_bytes(int fmt) { return fmt == kFmtS16 ? 2 : fmt == kFmtS24 ? 3 : 4; }
// integer -> float: value / 2^(bits-1), exact in float (formats::readWav)
__device__ __forceinline__ float load_in(const void* p, int fmt, long long i) {
    if (fmt == kFmtS16) return __fmul_rn((float) reinterpret_cast<const int16_t*>(p)[i], 1.0f / 32768.0f);
    if (fmt == kFmtS24) {
        const unsigned char* b = reinterpret_cast<const unsigned char*>(p) + 3 * i;
        const int v = (int) ((unsigned) b[0] << 8 | (unsigned) b[1] << 16 | (unsigned) b[2] << 24) >> 8;      // sign-extended
        return __fmul_rn((float) v, 1.0f / 8388608.0f);
    }
    return reinterpret_cast<const float*>(p)[i];
}
// float -> integer: the integer-WAV writer's rule (formats::writeWav), in double: y <= -1 -> INT32_MIN, y >= 1 -> INT32_MAX,
// NaN -> 0, otherwise round-half-even(2147483647 * y); then an arithmetic shift right by 32 - bits (toward -infinity, no dither)
__device__ __forceinline__ int quantise_s32(float y) {
    const double d = (double) y;
    if (d <= -1.0) return (int) 0x80000000u;
    if (d >= 1.0) return 0x7fffffff;
    if (d != d) return 0;
    return __double2int_rn(__dmul_rn(2147483647.0, d));
}
__device__ __forceinline__ void store_out(void* p, int fmt, long long i, float y) {
    if (fmt == kFmtS16) { reinterpret_cast<int16_t*>(p)[i] = (int16_t) (quantise_s32(y) >> 16); return; }
    if (fmt == kFmtS24) {
        const int q = quantise_s32(y) >> 8;
        unsigned char* b = reinterpret_cast<unsigned char*>(p) + 3 * i;
        b[0] = (unsigned char) q; b[1] = (unsigned char) (q >> 8); b[2] = (unsigned char) (q >> 16);
        return;
    }
    reinterpret_cast<float*>(p)[i] = y;
}

// MAC layout of the shared-IR kernel: a thread owns V float4 of each of K rows (K*V = 4).  Narrow: the float4 are TPR apart
// (a warp instruction reads 512 contiguous bytes).  WIDE: they come in adjacent pairs, one 32-byte load each (1 KB per warp
// instruction, half the load instructions for the same bytes in flight).
template <int M, bool WIDE> struct MacLayout {
    static constexpr int CH = M > 1024 ? M / 1024 : 1;                    // 32-byte chunks per thread per row (WIDE)
    static constexpr int V = WIDE ? 2 * CH : Tile<M>::V;
    static constexpr int TPR = WIDE ? M / (4 * CH) : Tile<M>::TPR;        // threads per row
    static constexpr int G = kThreads / TPR;
    static constexpr int K = 4 / V;
    static_assert(G * K == kTile / M, "the layout covers the tile");
    __device__ static __forceinline__ int f4(int c0, int vv) { return WIDE ? 2 * (c0 + (vv >> 1) * TPR) + (vv & 1) : c0 + vv * TPR; }
};

// ---- full M-point transform of the 8 registers of an FFT-layout thread ----------------------------
template <int M, bool INV, int PASS = 0, int PS = 1>
__device__ __forceinline__ void fft_run(float2 (&v)[kPts], int t, float2* srow, const float2* __restrict__ W) {
    constexpr int R = pass_radix(M, PASS);
    fft_pass<M, R, PS, INV, PASS>(v, t, W);
    if constexpr (PS * R < M) {
        bar_compute();                       // every earlier read of the tile has completed
        fft_scatter<M, R, PS>(v, t, srow);
        bar_compute();
        fft_gather_sw<M>(v, t, srow);
        fft_run<M, INV, PASS + 1, PS * R>(v, t, srow, W);
    }
}

// ===================================================================================================
// k_fwd: rows of <= B real samples -> zero-padded 2M-point real FFT -> packed spectrum rows.
// row = chan * blocks_per_chan + blk; the samples are src[chan*src_chan_stride + blk*B + i], i < clamp(L - blk*B, 0, B).
// Destination slot: blk (offline / IR preparation) or, when head != nullptr, the next ring slot of chan
// (streaming: the kernel also advances head[chan]).
struct FwdArgs {
    const void* src;           // device samples, format src_fmt (load_in)
    int src_fmt;
    const float* src2;         // optional second channel folded in as (a + b) / 2  (tools::sumToMono, fp/tools.cpp:25-29)
    long long src_chan_stride; // elements
    int L;                     // samples per channel
    int B;                     // block size (<= M)
    int blocks_per_chan;
    int n_rows;
    float2* dst;               // packed spectra
    long long dst_chan_stride; // float2 units between channel groups
    int dst_group;             // channels per group (0/1: plain [chan][slot][M]); see MacArgs::fdl_group
    long long dst_slot_stride; // float2 units between slots (0: M)
    int* head;                 // per-chan ring head (nullable)
    int ring;                  // ring slots per chan
    const float2* W;           // N = 2M roots of unity
    // Round-robin IR refresh rows (Source/PluginProcessor.cpp:455-461): after the ceil(n_rows/ROWS) tiles of audio rows
    // come ceil(n_rr/ROWS) tiles whose row i re-transforms partition rr_pos[ir] of the staged taps of ir = rr_list[i]
    // into H[ir] and then advances rr_pos[ir] (mod nparts[ir]).  rr_taps[ir] holds nparts[ir]*B zero-extended samples.
    int n_rr;
    const int* rr_list;
    const float* const* rr_taps;
    int* rr_pos;
    const int* nparts;
    float2* H;
    long long ir_stride;       // float2 units
    int h_reps;                // refresh rows write every copy of the IR spectra (MacArgs::h_reps)
    long long h_rep_stride;
};

struct FwdRow {                // what one row of k_fwd reads (p in format fmt) and writes
    const void* p; const float* q; int len; float2* d; bool live; int reps; int fmt;
};
template <int ROWS, int M>
__device__ __forceinline__ FwdRow fwd_row(const FwdArgs& a, int main_tiles, int tile, int r) {
    FwdRow w{nullptr, nullptr, 0, nullptr, false, 1, kFmtF32};
    if (tile < main_tiles) {
        const int row = tile * ROWS + r;
        if (row >= a.n_rows) return w;
        const int chan = row / a.blocks_per_chan, blk = row % a.blocks_per_chan;
        int len = a.L - blk * a.B;
        w.len = len < 0 ? 0 : (len > a.B ? a.B : len);
        const long long off = chan * a.src_chan_stride + (long long) blk * a.B;
        w.p = reinterpret_cast<const unsigned char*>(a.src) + off * fmt_bytes(a.src_fmt);
        w.fmt = a.src_fmt;
        w.q = a.src2 ? a.src2 + off : nullptr;
        int slot = blk;
        if (a.head) { slot = a.head[chan] + 1; if (slot >= a.ring) slot = 0; }
        const int grp = a.dst_group > 1 ? a.dst_group : 1;
        w.d = a.dst + (chan / grp) * a.dst_chan_stride + (long long) (chan % grp) * M + (long long) slot * (a.dst_slot_stride ? a.dst_slot_stride : M);
    } else {
        const int i = (tile - main_tiles) * ROWS + r;
        if (i >= a.n_rr) return w;
        const int ir = a.rr_list[i], p = a.rr_pos[ir];
        w.len = a.B;
        w.p = a.rr_taps[ir] + (long long) p * a.B;
        w.d = a.H + ir * a.ir_stride + (long long) p * M;
        w.reps = a.h_reps > 1 ? a.h_reps : 1;
    }
    w.live = true;
    return w;
}

template <int M>
__global__ void __launch_bounds__(kThreads) k_fwd(const FwdArgs a) {
    using T = Tile<M>;
    __shared__ __align__(16) float2 s_spec[kTile];
    const int tid = threadIdx.x;
    const int main_tiles = (a.n_rows + T::ROWS - 1) / T::ROWS;
    {   // FFT layout
        const int rf = tid / T::TPF, t = tid % T::TPF;
        const FwdRow w = fwd_row<T::ROWS, M>(a, main_tiles, blockIdx.x, rf);
        float2 v[kPts];
#pragma unroll
        for (int j = 0; j < kPts; ++j) v[j] = make_float2(0.f, 0.f);
        if (w.live) {
#pragma unroll
            for (int j = 0; j < kPts; ++j) {
                const int m = 2 * (t + j * T::TPF);
                float x0 = 0.f, x1 = 0.f;
                if (m < w.len) x0 = load_in(w.p, w.fmt, m);
                if (m + 1 < w.len) x1 = load_in(w.p, w.fmt, m + 1);
                if (w.q) {
                    if (m < w.len) { x0 += w.q[m]; x0 /= 2.0f; }
                    if (m + 1 < w.len) { x1 += w.q[m + 1]; x1 /= 2.0f; }
                }
                v[j] = make_float2(x0, x1);
            }
        }
        float2* srow = s_spec + rf * M;
        fft_run<M, false>(v, t, srow, a.W);
        bar_compute();
#pragma unroll
        for (int j = 0; j < kPts; ++j) srow[t + j * T::TPF] = v[j];
    }
    bar_compute();
    {   // MAC layout: split into the packed real spectrum and store 16 B per lane
        const int g = tid / T::TPR, c0 = tid % T::TPR;
#pragma unroll
        for (int s = 0; s < T::K; ++s) {
            const int rl = s * T::G + g;
            const FwdRow w = fwd_row<T::ROWS, M>(a, main_tiles, blockIdx.x, rl);
            if (!w.live) continue;
            const float2* z = s_spec + rl * M;
#pragma unroll
            for (int vv = 0; vv < T::V; ++vv) {
                const int k = 2 * (c0 + vv * T::TPR);
                const float2 x0 = real_split(z[k], z[(M - k) & (M - 1)], root<false>(a.W, k), k);
                const float2 x1 = real_split(z[k + 1], z[M - k - 1], root<false>(a.W, k + 1), k + 1);
                for (int rep = 0; rep < w.reps; ++rep)
                    *reinterpret_cast<float4*>(w.d + rep * a.h_rep_stride + k) = make_float4(x0.x, x0.y, x1.x, x1.y);
            }
        }
    }
    // advance the ring heads / round-robin positions once every read of the old value is done
    if ((int) blockIdx.x < main_tiles) {
        if (a.head) {
            bar_compute();
            if (tid < T::ROWS) {
                const int row = blockIdx.x * T::ROWS + tid;
                if (row < a.n_rows) { int h = a.head[row] + 1; a.head[row] = h >= a.ring ? 0 : h; }
            }
        }
    } else {
        bar_compute();
        if (tid < T::ROWS) {
            const int i = (blockIdx.x - main_tiles) * T::ROWS + tid;
            if (i < a.n_rr) { const int ir = a.rr_list[i]; int p = a.rr_pos[ir] + 1; a.rr_pos[ir] = p >= a.nparts[ir] ? 0 : p; }
        }
    }
}

// ===================================================================================================
// k_mac: Y[row][bin] = sum_{p < nvalid} FDL[row][(head - p) mod ring][bin] * H[ir][p][bin], ascending p
// (the summation order of fp/convolution.cpp:171-202), then -- when INV -- inverse FFT and overlap-add.
struct MacArgs {
    // packed spectra rows.  Plain layout [chan][slot][M]: fdl + chan*fdl_chan_stride + slot*M.  Streaming engine: the
    // fdl_group = ROWS channels of a kernel tile are interleaved per slot, [chan/ROWS][slot][chan%ROWS][M], so one block
    // step reads ONE contiguous ROWS*M*8-byte piece per tile and partition (16 KB) instead of ROWS pieces 0.8 MB apart.
    const float2* fdl;
    long long fdl_chan_stride; // float2 units between channel groups
    int fdl_group;             // channels per group (0/1: plain layout)
    long long fdl_slot_stride; // float2 units between slots (0: M)
    const int* head;           // per-chan newest slot; nullptr => head = blk (offline: block index)
    int ring;                  // slots per chan (wrap); offline: unused because nvalid <= blk+1
    int blocks_per_chan;
    int n_rows;
    const float2* H;           // IR partition spectra: H + ir*ir_stride + p*M
    long long ir_stride;       // float2 units
    const int* ir_of_chan;     // nullptr => IR 0 for every row
    const int* nparts;         // partitions per IR
    const float2* W;
    // !INV: accumulator spectra out
    float2* Y;                 // [row][M]
    // INV: time-domain epilogue
    int B;
    void* out;                 // element chan*out_chan_stride + blk*B + m, m < clamp(Lout - blk*B, 0, B), format out_fmt (store_out)
    int out_fmt;
    long long out_chan_stride;
    int Lout;
    float* ov;                 // streaming: overlap state [chan][B] (read, then replaced); offline: nullptr
    float* tail;               // offline: second halves [row][B]
    int split_in;              // k_mac_slots: tile slots that share one row (power of two, >= 1)
    int head_back;             // streaming: the newest spectrum of this step sits head_back slots behind head (callback order)
    // k_mac<FUSE>: the step's forward transform runs in the MAC kernel's prologue (no k_fwd launch): in[chan*in_chan_stride + i],
    // i < B, is the new block of every row; its spectrum goes to slot head+1, is used from registers as partition 0, and
    // head[chan] is advanced by this kernel.  `head` must not be const for that.  The new blocks are in format in_fmt (load_in).
    const void* in;
    int in_fmt;
    long long in_chan_stride;  // elements
    int* head_rw;
    int producer_sleep_ns;     // the TMA producer sleeps this long between polls of a busy stage (0: spin)
    unsigned zero;             // always 0; unknown to the compiler (mbar_arrive_after)
    int release_fence;         // fence.proxy.async before a ring stage is released (irb_tuning.hpp)
    int release_dep;           // the release carries a data dependency on the values read from the stage (mbar_arrive_after)
    // k_mac_p (persistent block step): work[0] = next unit, work[1] = CTAs that have finished (the last one clears both);
    // the launch's units in fetch order: unit_n[l] units of max(1, ROWS >> l) rows each, l = 0 .. 3
    int* work;
    int unit_n[4];
    // Shared IRs are kept in h_reps identical copies h_rep_stride float2 apart; CTA b streams copy b % h_reps.  CTAs of one
    // launch move through the partitions in lockstep, so without the copies every CTA would ask the same few L2 lines for
    // the same 4 KB partition at the same moment.
    int h_reps;
    long long h_rep_stride;
    int stagger_ns;            // k_mac_p: CTA starts are spread over this many nanoseconds
    int ring_stages;           // k_mac_p: use only this many of the ring's stages (0: all; measurement)
    unsigned long long* stamps;  // measurement (irbx_engine_set_stamps): thread 0 of CTA b < 64 stores %globaltimer at stamps[16 b + phase] in k_mac_slots
};
// the copy of the shared IR spectra this CTA streams
__device__ __forceinline__ const float2* ir_replica(const MacArgs& a) {
    return a.h_reps > 1 ? a.H + (long long) (blockIdx.x % (unsigned) a.h_reps) * a.h_rep_stride : a.H;
}

// Time-domain epilogue of a tile whose accumulated packed spectra sit in shared memory, row r at tile + r*M
// (r < rows_in_tile): packed merge -> inverse M-point FFT -> x 1/N -> overlap-add -> output block
// (fp/convolution.cpp:206-230).  Called by all kThreads compute threads.
// phase time stamp of the latency path (measurement aid: a null pointer in every product launch)
__device__ __forceinline__ void stamp(const MacArgs& a, int i) {
    if (a.stamps && blockIdx.x < 64 && threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); a.stamps[blockIdx.x * 16 + i] = t; }
}

// LAT (the few-row latency kernel, which has registers to spare): the overlap values are requested before the merge and the
// transform instead of after them, and the phases are time-stamped when a stamp buffer is set.
template <int M, bool LAT = false>
__device__ __forceinline__ void inv_epilogue(const MacArgs& a, float2* tile, int tid, int row0, int rows_in_tile) {
    using T = Tile<M>;
    const int rf = tid / T::TPF, t = tid % T::TPF;
    float2* srow = tile + rf * M;
    const int row = row0 + rf;
    const bool live = rf < rows_in_tile && row < a.n_rows;
    const int chan = live ? row / a.blocks_per_chan : 0, blk = live ? row % a.blocks_per_chan : 0;
    int olen = a.Lout - blk * a.B;
    olen = olen < 0 ? 0 : (olen > a.B ? a.B : olen);
    const long long out0 = chan * a.out_chan_stride + (long long) blk * a.B;      // element index of the output row
    float* ovp = a.ov ? a.ov + (long long) chan * a.B : nullptr;
    float* tailp = a.tail ? a.tail + (long long) row * a.B : nullptr;
    // The overlap of the previous block, all 2 x kPts values of a thread requested back to back (predicated loads, no branches:
    // one load per basic block used to cost one L2 latency EACH, 1.8 us on the latency path).
    const bool has_ov = live && ovp != nullptr;
    float ovv[2 * kPts];
    auto load_overlap = [&]() {
#pragma unroll
        for (int j = 0; j < kPts; ++j) {
            const int m = 2 * (t + j * T::TPF);
            ovv[2 * j] = (has_ov && m < a.B) ? ovp[m] : 0.0f;
            ovv[2 * j + 1] = (has_ov && m + 1 < a.B) ? ovp[m + 1] : 0.0f;
        }
    };
    if constexpr (LAT) load_overlap();
    float2 v[kPts];
#pragma unroll
    for (int j = 0; j < kPts; ++j) {
        const int k = t + j * T::TPF;
        v[j] = real_merge(srow[k], srow[(M - k) & (M - 1)], root<false>(a.W, k), k);
    }
    if constexpr (LAT) stamp(a, 10);
    fft_run<M, true>(v, t, srow, a.W);
    if constexpr (LAT) stamp(a, 11);
    if constexpr (!LAT) load_overlap();
    const float scale = 1.0f / (float) (2 * M);      // the 1/N of performRealOnlyInverseTransform
    // fp/convolution.cpp:210-213: y[i] += overlap[i]; overlap[i] = y[B + i]   (a product rounded, then a sum rounded: no FMA)
#pragma unroll
    for (int j = 0; j < kPts; ++j) {
        const int m = 2 * (t + j * T::TPF);
        v[j].x = __fmul_rn(v[j].x, scale); v[j].y = __fmul_rn(v[j].y, scale);
        if (has_ov && m < a.B) v[j].x = __fadd_rn(v[j].x, ovv[2 * j]);
        if (has_ov && m + 1 < a.B) v[j].y = __fadd_rn(v[j].y, ovv[2 * j + 1]);
    }
    if constexpr (LAT) stamp(a, 12);
    if (a.ov) bar_compute();                           // all overlap reads precede the overlap writes
    if constexpr (LAT) stamp(a, 13);
    if (live) {
        // Integer output (streaming only, so the barrier above has ended every read of the row): the output half is parked in the
        // thread's own places of the row and converted by a rolled loop, so that the double-precision rule (store_out) does not
        // run in 2 x kPts unrolled copies next to the live transform values.
        const bool pcm = a.out_fmt != kFmtF32;
        float* park = reinterpret_cast<float*>(srow);
        float* outp = reinterpret_cast<float*>(a.out) + out0;
#pragma unroll
        for (int j = 0; j < kPts; ++j) {
            const int m = 2 * (t + j * T::TPF);
            const float val[2] = {v[j].x, v[j].y};
#pragma unroll
            for (int e = 0; e < 2; ++e) {                   // one predicated store per sample: output block, or the next overlap / the tail
                const int mm = m + e;
                const bool first = mm < a.B;
                float* dst = first ? (pcm ? park : outp) + mm : (ovp ? ovp : tailp) + (mm - a.B);
                if (first ? mm < olen : mm < 2 * a.B) *dst = val[e];
            }
        }
        if (pcm) {
#pragma unroll 1
            for (int i = 0; i < 2 * kPts; ++i) {
                const int m = 2 * (t + (i >> 1) * T::TPF) + (i & 1);
                if (m < olen) store_out(a.out, a.out_fmt, out0 + m, park[m]);
            }
        }
    }
}

__device__ __forceinline__ long long fdl_row_offset(const MacArgs& a, int chan, int M) {
    const int grp = a.fdl_group > 1 ? a.fdl_group : 1;
    return (chan / grp) * a.fdl_chan_stride + (long long) (chan % grp) * M;
}
template <int M> __device__ __forceinline__ long long fdl_slot_stride(const MacArgs& a) { return a.fdl_slot_stride ? a.fdl_slot_stride : M; }

// ---- steps shared by the streaming block-step kernels (k_mac<FUSE>, k_mac_tma, k_mac_slots, k_mac_p, k_mac_mx) ----------

// ac += xv * h for one float4 (two packed bins) of a partition product, bin0: the float4 holds bin 0, the packed {DC, Nyquist}
// pair, which takes two real products instead of a complex one.  This fmaf sequence, in ascending partition order, is what
// makes the block-step kernels bit-identical to one another; k_mac and k_mac_slots call it, k_mac_tma, k_mac_p and
// k_mac_mx spell it out (as a call it changes their instruction schedule).
__device__ __forceinline__ void cmac4(float4& ac, const float4& xv, const float4& h, bool bin0) {
    const float h0i = bin0 ? 0.f : h.y, h0q = bin0 ? h.y : h.x;
    ac.x = fmaf(xv.x, h.x, fmaf(-xv.y, h0i, ac.x));
    ac.y = fmaf(xv.y, h0q, fmaf(xv.x, h0i, ac.y));
    ac.z = fmaf(xv.z, h.z, fmaf(-xv.w, h.w, ac.z));
    ac.w = fmaf(xv.w, h.z, fmaf(xv.z, h.w, ac.w));
}

// Barriers of an n-stage ring, set up by one thread: full[i] completes on the producer's expect_tx and the bytes of its bulk
// copies, empty[i] on one arrive of each compute warp.  The fence makes the initialised barriers visible to the async proxy.
__device__ __forceinline__ void ring_init(uint64_t* full, uint64_t* empty, int n) {
    for (int i = 0; i < n; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], kThreads / 32); }
    mbar_fence_init();
}

// A compute warp's release of a TMA-filled ring stage it has read: every lane orders its ld.shared of the stage ahead of the
// bulk copy that refills it (fence.proxy.async, if release_fence), then the warp's first lane arrives, carrying a data
// dependency on the values read from the stage if release_dep (mbar_arrive_after).
__device__ __forceinline__ void release_stage(uint64_t* b, uint32_t dep, const MacArgs& a, int tid) {
    if (a.release_fence) fence_proxy_async_smem();
    __syncwarp();
    if ((tid & 31) == 0) {
        if (a.release_dep) mbar_arrive_after(b, dep & a.zero);
        else mbar_arrive(b);
    }
}

// Shared-IR kernel: the whole tile is bound to one IR and a ring stage holds U consecutive partitions of it.
template <int M, int U>
struct MacSmem {
    float2 spec[kTile];                                  // tile in both layouts (inverse path)
    float2 h[kStages][U][M];                             // IR ring
    uint64_t full[kStages], empty[kStages];
};

template <int M, int U, bool INV, bool FUSE = false, bool WIDE = false>
__global__ void __launch_bounds__(kThreads + 32, U == 1 ? 3 : 2) k_mac(const MacArgs a) {
    static_assert(!FUSE || INV, "the fused forward transform belongs to the streaming block step");
    using T = Tile<M>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    MacSmem<M, U>& sm = *reinterpret_cast<MacSmem<M, U>*>(smem_raw);
    const int tid = threadIdx.x;
    const int row0 = blockIdx.x * T::ROWS;

    // shared mode: by contract every row of a tile is bound to the same IR (the host checks / pads)
    const int chan_first = row0 / a.blocks_per_chan;
    const int ir = a.ir_of_chan ? a.ir_of_chan[chan_first] : 0;
    const int np = a.nparts[ir];
    // number of partitions any row of this tile needs
    int pmax = np;
    if (!a.head) {          // offline: row = chan*blocks_per_chan + blk, blocks_per_chan % ROWS == 0 (host pads)
        int last = row0 + T::ROWS - 1;
        if (last >= a.n_rows) last = a.n_rows - 1;
        const int kmax = last % a.blocks_per_chan;
        if (kmax + 1 < pmax) pmax = kmax + 1;
    }
    const int ngroups = (pmax + U - 1) / U;

    if (tid == 0) ring_init(sm.full, sm.empty, kStages);
    __syncthreads();

    if (tid >= kThreads) {
        // ===== TMA producer warp: stream the IR partition spectra through the ring =====
        if (tid == kThreads) {
            const float2* hsrc = ir_replica(a) + ir * a.ir_stride;
            for (int g = 0; g < ngroups; ++g) {
                const int st = g % kStages;
                if (g >= kStages) mbar_wait_relaxed(&sm.empty[st], ((g / kStages) - 1) & 1, a.producer_sleep_ns);
                int cnt = pmax - g * U;
                if (cnt > U) cnt = U;
                const uint32_t bytes = (uint32_t) cnt * M * sizeof(float2);
                mbar_expect_tx(&sm.full[st], bytes);
                tma_bulk_g2s(&sm.h[st][0][0], hsrc + (long long) g * U * M, bytes, &sm.full[st]);
            }
        }
        return;
    }

    if constexpr (FUSE) {
        // ===== the block step's forward transform (k_fwd's work) for the rows of this tile, FFT layout; the IR ring fills meanwhile =====
        const int rf = tid / T::TPF, t = tid % T::TPF;
        const int row = row0 + rf;
        float2 v[kPts];
#pragma unroll
        for (int j = 0; j < kPts; ++j) v[j] = make_float2(0.f, 0.f);
        if (row < a.n_rows) {
            const long long i0 = (long long) row * a.in_chan_stride;
#pragma unroll
            for (int j = 0; j < kPts; ++j) {
                const int m = 2 * (t + j * T::TPF);                  // scalar loads: a row starts at an odd float offset when B is odd
                if (m < a.B) v[j].x = load_in(a.in, a.in_fmt, i0 + m);
                if (m + 1 < a.B) v[j].y = load_in(a.in, a.in_fmt, i0 + m + 1);
            }
        }
        float2* srow = sm.spec + rf * M;
        fft_run<M, false>(v, t, srow, a.W);
        bar_compute();
#pragma unroll
        for (int j = 0; j < kPts; ++j) srow[t + j * T::TPF] = v[j];
        bar_compute();
    }

    // ===== compute threads, MAC layout =====
    using L = MacLayout<M, WIDE>;
    const int g_ = tid / L::TPR, c0 = tid % L::TPR;
    const float4* xptr[L::K];      // row of the next partition to load (partition 0 = the newest slot)
    int slot[L::K], nvalid[L::K];
    float4 xa[U][L::K][L::V], xb[U][L::K][L::V];
#pragma unroll
    for (int s = 0; s < L::K; ++s) {
        const int rl = s * L::G + g_, row = row0 + rl;
        nvalid[s] = 0; slot[s] = 0; xptr[s] = nullptr;
        if (row < a.n_rows) {
            const int chan = row / a.blocks_per_chan, blk = row % a.blocks_per_chan;
            int hd = blk;
            if (a.head) { hd = a.head[chan] - a.head_back; if (hd < 0) hd += a.ring; }
            nvalid[s] = a.head ? np : (blk + 1 < np ? blk + 1 : np);
            slot[s] = hd;
            xptr[s] = reinterpret_cast<const float4*>(a.fdl + fdl_row_offset(a, chan, M) + (long long) hd * fdl_slot_stride<M>(a));
            if constexpr (FUSE) {
                // packed spectrum of the new block: into the slot after the old head, and kept as partition 0's operand;
                // the loads below then start at partition 1 = the old head
                const int ns = hd + 1 >= a.ring ? 0 : hd + 1;
                const float2* z = sm.spec + rl * M;
                float4* d = reinterpret_cast<float4*>(const_cast<float2*>(a.fdl) + fdl_row_offset(a, chan, M) + (long long) ns * fdl_slot_stride<M>(a));
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv) {
                    const int k = 2 * L::f4(c0, vv);
                    const float2 x0 = real_split(z[k], z[(M - k) & (M - 1)], root<false>(a.W, k), k);
                    const float2 x1 = real_split(z[k + 1], z[M - k - 1], root<false>(a.W, k + 1), k + 1);
                    xa[0][s][vv] = make_float4(x0.x, x0.y, x1.x, x1.y);
                    d[L::f4(c0, vv)] = xa[0][s][vv];
                }
            }
        } else if constexpr (FUSE) {
#pragma unroll
            for (int vv = 0; vv < L::V; ++vv) xa[0][s][vv] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    if constexpr (FUSE) {
        bar_compute();                                    // every read of the tile and of the old heads is done
        if (tid < T::ROWS && row0 + tid < a.n_rows) { const int h = a.head_rw[row0 + tid] + 1; a.head_rw[row0 + tid] = h >= a.ring ? 0 : h; }
    }
    float4 acc[L::K][L::V];
#pragma unroll
    for (int s = 0; s < L::K; ++s)
#pragma unroll
        for (int vv = 0; vv < L::V; ++vv) acc[s][vv] = make_float4(0.f, 0.f, 0.f, 0.f);

    const long long sstep = fdl_slot_stride<M>(a) / 2;    // float4 between ring slots
    const long long swrap = (long long) (a.ring - 1) * sstep;   // from slot 0 back to the top of the ring
    // Streaming with the fused prologue: every live row needs all np partitions, so the per-partition "is this row still
    // valid" predicate is dropped -- rows past n_rows just re-read the tile's first row (their sums are never stored).
    if constexpr (FUSE && WIDE) {
        const int chan0 = row0 / a.blocks_per_chan;       // the first row of a launched tile is always live
        const int hd0 = a.head[chan0];
#pragma unroll
        for (int s = 0; s < L::K; ++s)
            if (!xptr[s]) {
                xptr[s] = reinterpret_cast<const float4*>(a.fdl + fdl_row_offset(a, chan0, M) + (long long) hd0 * fdl_slot_stride<M>(a));
                slot[s] = hd0;
            }
    }
    auto load_group = [&](float4 (&x)[U][L::K][L::V], int g) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = g * U + u;
            if (FUSE && p == 0) continue;                 // partition 0 already sits in xa[0] (registers)
#pragma unroll
            for (int s = 0; s < L::K; ++s) {
                if constexpr (FUSE && WIDE) {
#pragma unroll
                    for (int vv = 0; vv < L::V; vv += 2) ldg_stream256(xptr[s] + L::f4(c0, vv), x[u][s][vv], x[u][s][vv + 1]);
                    const bool wrap = slot[s] == 0;
                    slot[s] = wrap ? a.ring - 1 : slot[s] - 1;
                    xptr[s] += wrap ? swrap : -sstep;
                    continue;
                }
                const bool ok = p < nvalid[s];
                if constexpr (WIDE) {
#pragma unroll
                    for (int vv = 0; vv < L::V; vv += 2) {
                        x[u][s][vv] = x[u][s][vv + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ok) ldg_stream256(xptr[s] + L::f4(c0, vv), x[u][s][vv], x[u][s][vv + 1]);
                    }
                } else {
#pragma unroll
                    for (int vv = 0; vv < L::V; ++vv)
                        x[u][s][vv] = ok ? ldg_stream(xptr[s] + L::f4(c0, vv)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                // step one slot back in the ring (wrap to the top)
                if (ok) {
                    if (slot[s] == 0) { slot[s] = a.ring - 1; xptr[s] += swrap; }
                    else { --slot[s]; xptr[s] -= sstep; }
                }
            }
        }
    };
    auto consume_group = [&](float4 (&x)[U][L::K][L::V], int g) {
        const int st = g % kStages;
        mbar_wait(&sm.full[st], (g / kStages) & 1);
        uint32_t dep = 0;                                 // carries every value read from the stage into the release
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (g * U + u < pmax) {
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv) {
                    const int c = L::f4(c0, vv);
                    const float4 h = *reinterpret_cast<const float4*>(&sm.h[st][u][2 * c]);
                    dep |= __float_as_uint(h.x);
#pragma unroll
                    for (int s = 0; s < L::K; ++s) cmac4(acc[s][vv], x[u][s][vv], h, c == 0);
                }
            }
        }
        release_stage(&sm.empty[st], dep, a, tid);
    };

    if (ngroups > 0) load_group(xa, 0);
    for (int g = 0; g < ngroups; g += 2) {
        if (g + 1 < ngroups) load_group(xb, g + 1);
        consume_group(xa, g);
        if (g + 1 < ngroups) {
            if (g + 2 < ngroups) load_group(xa, g + 2);
            consume_group(xb, g + 1);
        }
    }

    if constexpr (!INV) {
#pragma unroll
        for (int s = 0; s < L::K; ++s) {
            const int row = row0 + s * L::G + g_;
            if (row >= a.n_rows) continue;
#pragma unroll
            for (int vv = 0; vv < L::V; ++vv)
                reinterpret_cast<float4*>(a.Y + (long long) row * M)[L::f4(c0, vv)] = acc[s][vv];
        }
    } else {
        // ---- accumulators -> shared tile (MAC layout), then inverse real FFT in FFT layout ----
#pragma unroll
        for (int s = 0; s < L::K; ++s)
#pragma unroll
            for (int vv = 0; vv < L::V; ++vv)
                reinterpret_cast<float4*>(sm.spec + (s * L::G + g_) * M)[L::f4(c0, vv)] = acc[s][vv];
        bar_compute();
        inv_epilogue<M>(a, sm.spec, tid, row0, T::ROWS);
    }
}

// ===================================================================================================
// k_mac_tma: the fused streaming block step (k_mac<FUSE>'s job) with the FDL ITSELF streamed through TMA.
//
// A ring stage holds one partition of the tile's IR (M spectra bins) AND the tile's FDL slots for that partition (all ROWS rows,
// 16 KB), both written by bulk async copies of the producer warp's elected lane; the eight compute warps read them with
// conflict-free 16-byte shared-memory loads.  Against the register-staged loads of k_mac this keeps 3 stages x 20 KB x 3 CTAs
// = 180 KB of reads in flight per SM instead of 96 KB, issues no global load, no pointer or ring-wrap arithmetic in the
// compute warps, and frees the registers of the double buffer.  With the tile-interleaved FDL and equal heads (the normal
// case) a stage's FDL part is ONE 16 KB copy; rows with different heads, or the plain layout, get one copy per row.
// Stage 0's FDL area doubles as the FFT / epilogue tile: the prologue is finished with it before any warp releases stage 0
// for the first time (group 0 needs no FDL data: partition 0 is the new block's spectrum, held in registers), and the
// epilogue takes it back behind a barrier that follows every warp's last group.
// Same fmaf sequence per bin as k_mac / k_fwd: results are bit-identical to the two-launch form.
constexpr int kTmaStages = 3;
template <int M>
struct TmaSmem {
    struct Stage { float2 x[kTile]; float2 h[M]; };
    Stage st[kTmaStages];
    uint64_t full[kTmaStages], empty[kTmaStages];
    int hd[kTile / M];                                   // old heads of the tile's rows (-1: dead row)
};
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tma_bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}

template <int M>
__global__ void __launch_bounds__(kThreads + 32, M <= 1024 ? 3 : 2) k_mac_tma(const MacArgs a) {
    using T = Tile<M>;
    using L = MacLayout<M, false>;                        // narrow: consecutive lanes read consecutive float4 of shared memory
    extern __shared__ __align__(128) unsigned char smem_raw[];
    TmaSmem<M>& sm = *reinterpret_cast<TmaSmem<M>*>(smem_raw);
    float2* spec = sm.st[0].x;
    const int tid = threadIdx.x;
    const int row0 = blockIdx.x * T::ROWS;                // blocks_per_chan == 1: a row is a channel
    const int ir = a.ir_of_chan ? a.ir_of_chan[row0] : 0;
    const int np = a.nparts[ir];

    if (tid == 0) ring_init(sm.full, sm.empty, kTmaStages);
    if (tid < T::ROWS) {
        int hd = -1;
        if (row0 + tid < a.n_rows) { hd = a.head[row0 + tid] - a.head_back; if (hd < 0) hd += a.ring; }
        sm.hd[tid] = hd;
    }
    __syncthreads();                                      // the heads are read; they are advanced after the prologue

    if (tid >= kThreads) {
        // ===== TMA producer =====
        if (tid == kThreads) {
            const float2* hsrc = ir_replica(a) + ir * a.ir_stride;
            const long long sstride = fdl_slot_stride<M>(a);
            int nlive = 0;
            bool uni = a.fdl_group == T::ROWS;
            for (int r = 0; r < T::ROWS; ++r) {
                if (sm.hd[r] >= 0) { ++nlive; uni = uni && sm.hd[r] == sm.hd[0]; }
            }
            const uint64_t pol = l2_policy_evict_first();
            int back = 0;                                 // partition g >= 1 meets slot (hd - (g - 1)) mod ring
            for (int g = 0; g < np; ++g) {
                const int st = g % kTmaStages;
                if (g >= kTmaStages) mbar_wait_relaxed(&sm.empty[st], ((g / kTmaStages) - 1) & 1, a.producer_sleep_ns);
                const uint32_t hb = M * sizeof(float2);
                mbar_expect_tx(&sm.full[st], hb + (g > 0 ? (uint32_t) nlive * hb : 0u));
                tma_bulk_g2s(sm.st[st].h, hsrc + (long long) g * M, hb, &sm.full[st]);
                if (g > 0) {
                    if (uni) {
                        int sl = sm.hd[0] - back; if (sl < 0) sl += a.ring;
                        tma_bulk_g2s_hint(sm.st[st].x, a.fdl + fdl_row_offset(a, row0, M) + (long long) sl * sstride, (uint32_t) nlive * hb, &sm.full[st], pol);
                    } else {
                        for (int r = 0; r < nlive; ++r) {
                            int sl = sm.hd[r] - back; if (sl < 0) sl += a.ring;
                            tma_bulk_g2s_hint(sm.st[st].x + r * M, a.fdl + fdl_row_offset(a, row0 + r, M) + (long long) sl * sstride, hb, &sm.full[st], pol);
                        }
                    }
                    if (++back >= a.ring) back = 0;
                }
            }
        }
        return;
    }

    // ===== forward transform of the tile's new blocks (FFT layout), spectrum -> FDL slot head+1 and registers =====
    {
        const int rf = tid / T::TPF, t = tid % T::TPF;
        const int row = row0 + rf;
        float2 v[kPts];
#pragma unroll
        for (int j = 0; j < kPts; ++j) v[j] = make_float2(0.f, 0.f);
        if (row < a.n_rows) {
            const long long i0 = (long long) row * a.in_chan_stride;
#pragma unroll
            for (int j = 0; j < kPts; ++j) {
                const int m = 2 * (t + j * T::TPF);
                if (m < a.B) v[j].x = load_in(a.in, a.in_fmt, i0 + m);
                if (m + 1 < a.B) v[j].y = load_in(a.in, a.in_fmt, i0 + m + 1);
            }
        }
        float2* srow = spec + rf * M;
        fft_run<M, false>(v, t, srow, a.W);
        bar_compute();
#pragma unroll
        for (int j = 0; j < kPts; ++j) srow[t + j * T::TPF] = v[j];
        bar_compute();
    }
    const int g_ = tid / L::TPR, c0 = tid % L::TPR;
    float4 x0[L::K][L::V], acc[L::K][L::V];
#pragma unroll
    for (int s = 0; s < L::K; ++s) {
        const int rl = s * L::G + g_, hd = sm.hd[rl];
#pragma unroll
        for (int vv = 0; vv < L::V; ++vv) { x0[s][vv] = make_float4(0.f, 0.f, 0.f, 0.f); acc[s][vv] = make_float4(0.f, 0.f, 0.f, 0.f); }
        if (hd >= 0) {
            const int ns = hd + 1 >= a.ring ? 0 : hd + 1;
            const float2* z = spec + rl * M;
            float4* d = reinterpret_cast<float4*>(const_cast<float2*>(a.fdl) + fdl_row_offset(a, row0 + rl, M) + (long long) ns * fdl_slot_stride<M>(a));
#pragma unroll
            for (int vv = 0; vv < L::V; ++vv) {
                const int k = 2 * L::f4(c0, vv);
                const float2 s0 = real_split(z[k], z[(M - k) & (M - 1)], root<false>(a.W, k), k);
                const float2 s1 = real_split(z[k + 1], z[M - k - 1], root<false>(a.W, k + 1), k + 1);
                x0[s][vv] = make_float4(s0.x, s0.y, s1.x, s1.y);
                d[L::f4(c0, vv)] = x0[s][vv];
            }
        }
    }
    // the tile (stage 0's FDL area) was written and read through the generic proxy; the bulk copy of partition kTmaStages writes it
    // through the async proxy once every warp has released stage 0: order the two proxies once per tile, ahead of that release
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    bar_compute();                                        // the tile is free; nobody has released stage 0 yet
    if (tid < T::ROWS && row0 + tid < a.n_rows) { const int h = a.head_rw[row0 + tid] + 1; a.head_rw[row0 + tid] = h >= a.ring ? 0 : h; }

    // ===== multiply-accumulate over the partitions, ascending (fp/convolution.cpp:171-202) =====
    for (int g = 0; g < np; ++g) {
        const int st = g % kTmaStages;
        mbar_wait(&sm.full[st], (g / kTmaStages) & 1);
        uint32_t dep = 0;                                 // see mbar_arrive_after
#pragma unroll
        for (int vv = 0; vv < L::V; ++vv) {
            const int c = L::f4(c0, vv);
            const float4 h = *reinterpret_cast<const float4*>(&sm.st[st].h[2 * c]);
            dep |= __float_as_uint(h.x);
            const float h0i = c == 0 ? 0.f : h.y, h0q = c == 0 ? h.y : h.x;        // bin 0 = packed {DC, Nyquist}
#pragma unroll
            for (int s = 0; s < L::K; ++s) {
                float4 xv = x0[s][vv];
                if (g > 0) {
                    xv = *reinterpret_cast<const float4*>(&sm.st[st].x[(s * L::G + g_) * M + 2 * c]);
                    dep |= __float_as_uint(xv.x);
                }
                float4& ac = acc[s][vv];
                ac.x = fmaf(xv.x, h.x, fmaf(-xv.y, h0i, ac.x));
                ac.y = fmaf(xv.y, h0q, fmaf(xv.x, h0i, ac.y));
                ac.z = fmaf(xv.z, h.z, fmaf(-xv.w, h.w, ac.z));
                ac.w = fmaf(xv.w, h.z, fmaf(xv.z, h.w, ac.w));
            }
        }
        release_stage(&sm.empty[st], dep, a, tid);
    }

    bar_compute();                                        // every warp is through its last group: stage 0 is the tile again
#pragma unroll
    for (int s = 0; s < L::K; ++s)
#pragma unroll
        for (int vv = 0; vv < L::V; ++vv)
            reinterpret_cast<float4*>(spec + (s * L::G + g_) * M)[L::f4(c0, vv)] = acc[s][vv];
    bar_compute();
    inv_epilogue<M>(a, spec, tid, row0, T::ROWS);
}

// ===================================================================================================
// k_mac_slots: the MAC for (a) rows that do NOT share an IR inside a tile (per-stream IRs, BASELINE config 4) and
// (b) FEW rows (the single-stream latency path, BASELINE config 2), where one CTA per tile would leave the GPU idle
// and the load chain of a single row is latency-bound.
//
// A tile has ROWS = 2048/M SLOTS.  Slot r works for row  row0 + r / split_in  on the partition range number
// q = cluster_rank * split_in + r % split_in  of nsplit = cluster_size * split_in equal ranges of that row's IR, and
// stages its OWN IR partition per ring step (one bulk TMA copy per slot).  With nsplit == 1 a slot is a row.
// Otherwise the partial sums of a row are added in ascending q (i.e. ascending partition order between ranges)
// through distributed shared memory: every CTA of the cluster reduces 1/cluster_size of the tile and writes it
// into rank 0, which runs the inverse-FFT epilogue.  Streaming only (head != nullptr).
constexpr int kSlotStages = 8;           // IR ring stages of the slot kernel: a short partition range is staged all at once
constexpr int kSlotDepth = 4;            // FDL load groups a thread keeps in flight (registers)
template <int M>
struct SlotSmem {
    float2 spec[kTile];                                  // fused step: the forward transform's tile; then the partial sums, slot-major
    float2 h[kSlotStages][kTile / M][M];                 // IR ring: one partition per slot and stage; reused as the reduced tile
    float2 xnew[kTile];                                  // fused step, cluster rank 0: packed spectra of the rows' new blocks (partition 0's operand)
    uint64_t full[kSlotStages], empty[kSlotStages];
    int pbeg[kTile / M], pcnt[kTile / M], ngroups;
    int hd[kTile / M];                                   // head of every slot's row as the kernel found it
};

__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_size() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
}
__device__ __forceinline__ uint32_t dsmem_addr(const void* local, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(local)), "r"(rank));
    return r;
}
__device__ __forceinline__ float4 dsmem_ld4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void dsmem_st4(uint32_t addr, float4 v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

template <int M, bool INV, bool WIDE = true>
__global__ void __launch_bounds__(kThreads + 32, 1) k_mac_slots(const MacArgs a) {
    using T = Tile<M>;
    using L = MacLayout<M, WIDE>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    SlotSmem<M>& sm = *reinterpret_cast<SlotSmem<M>*>(smem_raw);
    const int tid = threadIdx.x;
    const int CL = (int) cluster_size(), crank = (int) cluster_rank();
    const int split_in = a.split_in, nsplit = split_in * CL;
    const int rpt = T::ROWS / split_in;                   // rows per tile
    const int row0 = (blockIdx.x / CL) * rpt;
    stamp(a, 0);

    if (tid == 0) {
        ring_init(sm.full, sm.empty, kSlotStages);
        sm.ngroups = 0;
    }
    __syncthreads();
    // partition range of every slot: row r's nv partitions are cut into nsplit ranges of ceil(nv / nsplit)
    if (tid < T::ROWS) {
        const int row = row0 + tid / split_in;
        int pb = 0, pc = 0;
        int hd = 0;
        if (row < a.n_rows) {
            const int chan = row / a.blocks_per_chan;
            const int nv = a.nparts[a.ir_of_chan ? a.ir_of_chan[chan] : 0];
            hd = a.head[chan];
            if (a.in != nullptr && CL > 1) {
                // Fused step on a cluster: rank 0 also runs the forward transform, so it takes partition 0 alone (its operand is the
                // transform's result); the other ranks share partitions 1 .. nv-1.  Ranges stay in ascending order of (rank, slot).
                if (crank == 0) { pb = 0; pc = (tid % split_in == 0 && nv > 0) ? 1 : 0; }
                else {
                    const int nsl = (CL - 1) * split_in, per = (nv - 1 + nsl - 1) / nsl;
                    pb = 1 + ((crank - 1) * split_in + tid % split_in) * per;
                    pc = nv - pb;
                    pc = pc < 0 ? 0 : (pc > per ? per : pc);
                }
            } else {
                const int per = (nv + nsplit - 1) / nsplit;
                pb = (crank * split_in + tid % split_in) * per;
                pc = nv - pb;
                pc = pc < 0 ? 0 : (pc > per ? per : pc);
            }
        }
        sm.pbeg[tid] = pb; sm.pcnt[tid] = pc; sm.hd[tid] = hd;
        if (pc > 0) atomicMax(&sm.ngroups, pc);
    }
    __syncthreads();
    const int ngroups = sm.ngroups;
    stamp(a, 1);

    if (tid >= kThreads) {
        // ===== TMA producer warp: one bulk copy per (slot, step); lanes split the slots of the tile =====
        // Everything a copy's address depends on is fetched BEFORE the loop: with the IR index loaded inside it every ring step
        // started one L2 latency after the previous one (phase stamps: 0.4 - 0.55 us per partition, whatever the loads did).
        const int lane = tid - kThreads;
        constexpr int SPL = (T::ROWS + 31) / 32;           // slots per lane
        const float2* hsrc[SPL];
        int pcn[SPL];
#pragma unroll
        for (int j = 0; j < SPL; ++j) {
            const int r = lane + 32 * j;
            pcn[j] = r < T::ROWS ? sm.pcnt[r] : 0;
            hsrc[j] = a.H;
            if (pcn[j] > 0) {
                const int chan = (row0 + r / split_in) / a.blocks_per_chan;
                const int irr = a.ir_of_chan ? a.ir_of_chan[chan] : 0;
                hsrc[j] = a.H + irr * a.ir_stride + (long long) sm.pbeg[r] * M;
            }
        }
        for (int g = 0; g < ngroups; ++g) {
            const int st = g % kSlotStages;
            if (g >= kSlotStages) mbar_wait_relaxed(&sm.empty[st], ((g / kSlotStages) - 1) & 1, a.producer_sleep_ns);
            uint32_t total = 0;
#pragma unroll
            for (int j = 0; j < SPL; ++j) if (g < pcn[j]) total += M * sizeof(float2);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
            if (lane == 0) mbar_expect_tx(&sm.full[st], total);
            __syncwarp();
#pragma unroll
            for (int j = 0; j < SPL; ++j)
                if (g < pcn[j]) tma_bulk_g2s(&sm.h[st][lane + 32 * j][0], hsrc[j] + (long long) g * M, M * sizeof(float2), &sm.full[st]);
        }
    } else {
        // ===== compute threads =====
        // Fused step (a.in != nullptr): the heads still name the PREVIOUS block; the new block's spectrum goes to slot head + 1 and is
        // partition 0's operand.  Cluster rank 0 owns partition 0 of every row of the tile, so it alone runs the forward transform
        // (k_fwd's work for these rows), writes the spectrum to the FDL and keeps a packed copy in shared memory; the other ranks
        // start on their partition ranges (which only meet older slots) right away.  Rank 0 advances the heads after the
        // cluster's first barrier, when every rank has read them.
        const bool fused = a.in != nullptr;
        if (fused && crank == 0) {
            const int rf = tid / T::TPF, t = tid % T::TPF;
            const int row = row0 + rf;
            float2 v[kPts];
#pragma unroll
            for (int j = 0; j < kPts; ++j) v[j] = make_float2(0.f, 0.f);
            if (rf < rpt && row < a.n_rows) {
                const long long i0 = (long long) row * a.in_chan_stride;
#pragma unroll
                for (int j = 0; j < kPts; ++j) {
                    const int m = 2 * (t + j * T::TPF);
                    if (m < a.B) v[j].x = load_in(a.in, a.in_fmt, i0 + m);
                    if (m + 1 < a.B) v[j].y = load_in(a.in, a.in_fmt, i0 + m + 1);
                }
            }
            float2* srow = sm.spec + rf * M;
            fft_run<M, false>(v, t, srow, a.W);
            bar_compute();
#pragma unroll
            for (int j = 0; j < kPts; ++j) srow[t + j * T::TPF] = v[j];
            bar_compute();
            for (int o = tid; o < rpt * (M / 2); o += kThreads) {
                const int r = o / (M / 2), k = 2 * (o % (M / 2)), rw = row0 + r;
                if (rw >= a.n_rows) continue;
                const float2* z = sm.spec + r * M;
                const float2 x0 = real_split(z[k], z[(M - k) & (M - 1)], root<false>(a.W, k), k);
                const float2 x1 = real_split(z[k + 1], z[M - k - 1], root<false>(a.W, k + 1), k + 1);
                const float4 xv = make_float4(x0.x, x0.y, x1.x, x1.y);
                int ns = sm.hd[r * split_in] + 1; if (ns >= a.ring) ns = 0;
                *reinterpret_cast<float4*>(const_cast<float2*>(a.fdl) + fdl_row_offset(a, rw, M) + (long long) ns * fdl_slot_stride<M>(a) + k) = xv;
                *reinterpret_cast<float4*>(sm.xnew + r * M + k) = xv;
            }
            bar_compute();                                // xnew is complete; sm.spec is free for the partial sums
        }
        stamp(a, 2);
        // MAC layout: thread owns V float4 of the K slots s*G + g_
        const int g_ = tid / L::TPR, c0 = tid % L::TPR;
        const float4* xptr[L::K];
        int slot[L::K], nvalid[L::K];
        bool first[L::K];                                 // this slot's range starts at partition 0 of a fused step: operand in sm.xnew
#pragma unroll
        for (int s = 0; s < L::K; ++s) {
            const int sl = s * L::G + g_;
            const int row = row0 + sl / split_in;
            nvalid[s] = sm.pcnt[sl]; slot[s] = 0; xptr[s] = nullptr; first[s] = false;
            if (nvalid[s] > 0) {
                const int chan = row / a.blocks_per_chan;
                int hd = (sm.hd[sl] + (fused ? 1 : 0) - a.head_back - sm.pbeg[sl]) % a.ring;      // partition p meets slot (newest - p) mod ring
                if (hd < 0) hd += a.ring;
                slot[s] = hd;
                xptr[s] = reinterpret_cast<const float4*>(a.fdl + fdl_row_offset(a, chan, M) + (long long) hd * fdl_slot_stride<M>(a));
                first[s] = fused && sm.pbeg[sl] == 0;
            }
        }
        float4 acc[L::K][L::V];
#pragma unroll
        for (int s = 0; s < L::K; ++s)
#pragma unroll
            for (int vv = 0; vv < L::V; ++vv) acc[s][vv] = make_float4(0.f, 0.f, 0.f, 0.f);

        float4 xq[kSlotDepth][L::K][L::V];
        const long long sstep = fdl_slot_stride<M>(a) / 2;    // float4 between ring slots
        auto load_group = [&](float4 (&x)[L::K][L::V], int g) {
#pragma unroll
            for (int s = 0; s < L::K; ++s) {
                const bool ok = g < nvalid[s];
                if (g == 0 && first[s]) {                 // the new block's spectrum is not in global memory for this kernel to read: it sits in sm.xnew
                    const float4* xn = reinterpret_cast<const float4*>(sm.xnew + ((s * L::G + g_) / split_in) * M);
#pragma unroll
                    for (int vv = 0; vv < L::V; ++vv) x[s][vv] = ok ? xn[L::f4(c0, vv)] : make_float4(0.f, 0.f, 0.f, 0.f);
                } else if constexpr (WIDE) {
#pragma unroll
                    for (int vv = 0; vv < L::V; vv += 2) {
                        x[s][vv] = x[s][vv + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ok) ldg_stream256(xptr[s] + L::f4(c0, vv), x[s][vv], x[s][vv + 1]);
                    }
                } else {
#pragma unroll
                    for (int vv = 0; vv < L::V; ++vv) x[s][vv] = ok ? ldg_stream(xptr[s] + L::f4(c0, vv)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                if (ok) {
                    if (slot[s] == 0) { slot[s] = a.ring - 1; xptr[s] += (long long) (a.ring - 1) * sstep; }
                    else { --slot[s]; xptr[s] -= sstep; }
                }
            }
        };
        auto consume_group = [&](float4 (&x)[L::K][L::V], int g) {
            const int st = g % kSlotStages;
            mbar_wait(&sm.full[st], (g / kSlotStages) & 1);
            uint32_t dep = 0;                              // see mbar_arrive_after
#pragma unroll
            for (int vv = 0; vv < L::V; ++vv) {
                const int c = L::f4(c0, vv);
#pragma unroll
                for (int s = 0; s < L::K; ++s) {
                    if (g >= nvalid[s]) continue;          // this slot's range is shorter: its stage entry was not filled
                    const float4 h = *reinterpret_cast<const float4*>(&sm.h[st][s * L::G + g_][2 * c]);
                    dep |= __float_as_uint(h.x);
                    cmac4(acc[s][vv], x[s][vv], h, c == 0);
                }
            }
            release_stage(&sm.empty[st], dep, a, tid);
        };
        // kSlotDepth groups of FDL loads stay in flight (round 1 kept one), the IR ring holds kSlotStages partitions: the 6 or 7
        // partitions a slot has on the latency path are requested at once.
#pragma unroll
        for (int i = 0; i < kSlotDepth; ++i) if (i < ngroups) load_group(xq[i], i);
        for (int g = 0; g < ngroups; g += kSlotDepth) {
#pragma unroll
            for (int i = 0; i < kSlotDepth; ++i) {
                if (g + i < ngroups) {
                    consume_group(xq[i], g + i);
                    if (g + i + kSlotDepth < ngroups) load_group(xq[i], g + i + kSlotDepth);
                }
            }
        }
        stamp(a, 3);
        if (!INV && nsplit == 1) {
#pragma unroll
            for (int s = 0; s < L::K; ++s) {
                const int row = row0 + s * L::G + g_;
                if (row >= a.n_rows) continue;
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv) reinterpret_cast<float4*>(a.Y + (long long) row * M)[L::f4(c0, vv)] = acc[s][vv];
            }
        } else {
#pragma unroll
            for (int s = 0; s < L::K; ++s)
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv)
                    reinterpret_cast<float4*>(sm.spec + (s * L::G + g_) * M)[L::f4(c0, vv)] = acc[s][vv];
        }
    }
    if (!INV && nsplit == 1) return;

    float2* fin = sm.spec;                                // tile the epilogue reads: rows at fin + r*M
    if (nsplit > 1) {
        // ---- sum the nsplit partial spectra of every row in ascending range order: first the split_in slots of a row inside
        // this CTA (shared memory), then the per-CTA sums across the cluster (distributed shared memory) into rank 0 ----
        float4* part = reinterpret_cast<float4*>(&sm.h[0][0][0]);          // this CTA's row sums; the IR ring is idle by now
        float4* red = part + kTile / 2;                                     // rank 0: the reduced tile
        const int n4 = rpt * (M / 2);                     // float4 of the reduced tile; n4 % CL == 0 (host guarantees)
        if (tid < kThreads) {
            bar_compute();                                // all partial sums of this CTA are in sm.spec
            const float4* sp = reinterpret_cast<const float4*>(sm.spec);
            for (int o = tid; o < n4; o += kThreads) {
                const int fr = o / (M / 2), c = o % (M / 2);
                float4 sum = sp[(fr * split_in) * (M / 2) + c];
                for (int sub = 1; sub < split_in; ++sub) {
                    const float4 v = sp[(fr * split_in + sub) * (M / 2) + c];
                    sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
                }
                part[o] = sum;
            }
        }
        stamp(a, 4);
        cluster_sync_all();                               // every CTA's row sums are visible cluster-wide
        stamp(a, 5);
        if (a.in != nullptr && crank == 0 && tid < rpt && row0 + tid < a.n_rows) {      // fused step: every rank has read the old heads
            const int hnew = sm.hd[tid * split_in] + 1;
            a.head_rw[row0 + tid] = hnew >= a.ring ? 0 : hnew;
        }
        if (tid < kThreads && CL > 1) {
            const int per = n4 / CL;
            const uint32_t red0 = dsmem_addr(red, 0);
            for (int o = crank * per + tid; o < (crank + 1) * per; o += kThreads) {
                float4 sum = dsmem_ld4(dsmem_addr(part, 0) + (uint32_t) (o * sizeof(float4)));
                for (int rk = 1; rk < CL; ++rk) {
                    const float4 v = dsmem_ld4(dsmem_addr(part, (uint32_t) rk) + (uint32_t) (o * sizeof(float4)));
                    sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
                }
                dsmem_st4(red0 + (uint32_t) (o * sizeof(float4)), sum);
            }
        }
        stamp(a, 6);
        cluster_sync_all();                               // rank 0 holds the reduced tile; nobody reads remote memory any more
        stamp(a, 7);
        if (crank != 0) return;
        fin = reinterpret_cast<float2*>(CL > 1 ? red : part);
    }
    if (tid >= kThreads) return;
    if (nsplit == 1) {
        bar_compute();                                    // the tile is complete in shared memory
        if (a.in != nullptr && tid < rpt && row0 + tid < a.n_rows) {       // fused step without a split: the heads move here
            const int hnew = sm.hd[tid] + 1;
            a.head_rw[row0 + tid] = hnew >= a.ring ? 0 : hnew;
        }
    }
    if constexpr (INV) {
        inv_epilogue<M, true>(a, fin, tid, row0, rpt);
    } else {
        for (int o = tid; o < rpt * (M / 2); o += kThreads) {
            const int row = row0 + o / (M / 2);
            if (row < a.n_rows) reinterpret_cast<float4*>(a.Y + (long long) row * M)[o % (M / 2)] = reinterpret_cast<const float4*>(fin)[o];
        }
    }
    stamp(a, 8);
}

// (a + b) / 2 : tools::sumToMono (fp/tools.cpp:25-29)
static __global__ void k_fold_mono(const float* l, const float* r, float* out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float v = l[i];
    v += r[i];
    v /= 2.0f;
    out[i] = v;
}

// offline: out[chan][blk*B + m] += tail[chan][blk-1][m]   (the overlap of the previous block)
static __global__ void k_ola_tail(float* out, long long out_chan_stride, int Lout, const float* tail, int B, int blocks_per_chan, int n_chans) {
    const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
    const long long per_chan = (long long) blocks_per_chan * B;
    if (i >= per_chan * n_chans) return;
    const int chan = (int) (i / per_chan);
    const long long r = i % per_chan;
    const int blk = (int) (r / B), m = (int) (r % B);
    if (blk == 0) return;
    const long long o = (long long) blk * B + m;
    if (o >= Lout) return;
    out[chan * out_chan_stride + o] += tail[((long long) chan * blocks_per_chan + (blk - 1)) * B + m];
}

}  // namespace irb
