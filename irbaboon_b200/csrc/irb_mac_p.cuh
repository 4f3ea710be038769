// irb_mac_p.cuh -- k_mac_p: the PERSISTENT streaming block step (sm_100a).
//
// One launch per block step, grid = resident CTAs (two per SM).  A CTA keeps taking UNITS of work -- up to ROWS = 2048/M
// stream-channels ("rows") of one kernel tile -- from a device-side counter until none is left, and for every unit does the
// whole UPOLA step of its rows (fp/convolution.cpp:128-149,160-215 / Source/PluginProcessor.cpp:430-436,480-510):
//   forward real FFT of the new blocks -> packed spectrum into FDL slot head+1 (and kept in registers as partition 0's operand),
//   Y[bin] = sum_p FDL[(head-p) mod ring][bin] * H[p][bin] in ascending p with FP32 FMA accumulators in registers,
//   packed merge -> inverse FFT -> x 1/N -> overlap-add -> output block.
// What the persistent form buys over one CTA per tile (k_mac_tma):
//   * the ninth warp (the TMA producer) runs AHEAD ACROSS UNITS: while the eight compute warps are in a unit's inverse FFT and
//     the next unit's forward FFT, the next unit's FDL slots and IR partitions are already landing in the shared-memory ring
//     (NS stages of 16 KB FDL + the IR partition(s)).  The FFT tile is the FDL area of the stage the compute warps consumed last:
//     they keep that one stage back through the epilogue and the next unit's prologue and release it afterwards, the
//     producer meanwhile fills the other NS-1 stages;
//   * less wave quantisation: CTAs take units as they finish, so a launch ends when the last unit does instead of after
//     ceil(tiles / CTAs) lock-step waves.  The host can also size the LAST partial wave as units of fewer rows (ROWS/2, ROWS/4 ...;
//     unit_n[1..3], tuning knob unit_narrowing); that form is bit-exact but measured slower (a narrow unit has proportionally less
//     in flight), so it is off by default and every unit is a full tile;
//   * PERROW = true replaces the register-staged per-stream-IR kernel (BASELINE configs[3]): every row of a unit stages its
//     own IR partition per ring stage, FDL and IR both through TMA, the forward transform fused -- one launch per block step.
// The fmaf sequence per bin is the one of k_mac / k_mac_tma / k_fwd: results are bit-identical to the two-launch form.
#pragma once
#include "irb_kernels.cuh"

namespace irb {

template <int M, bool PERROW> struct PCfg {
    static constexpr int ROWS = kTile / M;
    static constexpr int HF2 = PERROW ? kTile : M;                           // float2 of IR spectra per ring stage
    static constexpr int STAGE_BYTES = (kTile + HF2) * (int) sizeof(float2);
    // two CTAs per SM: (228 KB - 2 x 1 KB reserved) / 2 = 113 KB each; minus 1 KB of barriers / descriptors.  There is no separate
    // FFT tile: between two units the compute warps HOLD the ring stage they consumed last and use its FDL area as the tile.
    static constexpr int BUDGET = 113 * 1024 - 1024;
    static constexpr int NS = BUDGET / STAGE_BYTES > 8 ? 8 : BUDGET / STAGE_BYTES;
    static_assert(NS >= 2, "at least two ring stages");
};

struct PDesc {                     // what the producer tells the compute warps about a unit
    int row0, nrows, np;           // first row, live rows (0: no more work), partitions to stream (max over the rows)
    int hd[8];                     // old head of every row (-1: dead row)
    int npr[8];                    // partitions of every row's IR (PERROW)
};

template <int M, bool PERROW>
struct PSmem {
    using C = PCfg<M, PERROW>;
    struct Stage { float2 x[kTile]; float2 h[C::HF2]; };
    Stage st[C::NS];               // st[hold].x doubles as the FFT-layout <-> MAC-layout exchange tile of the epilogue and the next prologue
    uint64_t full[C::NS], empty[C::NS], u_full[2], u_empty[2];
    PDesc desc[2];
};

template <int M, bool PERROW>
__global__ void __launch_bounds__(kThreads + 32, 2) k_mac_p(const MacArgs a) {
    using T = Tile<M>;
    using L = MacLayout<M, false>;                        // consecutive lanes read consecutive float4 of shared memory
    using C = PCfg<M, PERROW>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PSmem<M, PERROW>& sm = *reinterpret_cast<PSmem<M, PERROW>*>(smem_raw);
    const int tid = threadIdx.x;
    const int NSE = a.ring_stages > 0 && a.ring_stages < C::NS ? a.ring_stages : C::NS;       // ring stages in use
    // measurement aid (null in every product launch): CTA 0 logs {globaltimer, SM cycle counter} at its start and end into a ring
    // of 4096 launches indexed by work[2], the launch sequence number -- the SM clock a block step actually ran at
    unsigned long long* stamp_row = nullptr;
    if (a.stamps && blockIdx.x == 0 && tid == 0) {
        stamp_row = a.stamps + (size_t) ((unsigned) a.work[2] % 4096u) * 4;
        unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        stamp_row[0] = t; stamp_row[1] = (unsigned long long) clock64();
    }

    if (tid == 0) {
        for (int i = 0; i < 2; ++i) { mbar_init(&sm.u_full[i], 1); mbar_init(&sm.u_empty[i], kThreads / 32); }
        ring_init(sm.full, sm.empty, C::NS);
    }
    __syncthreads();

    if (tid >= kThreads) {
        // ===== TMA producer: fetch units, publish their descriptors, stream their partitions through the ring =====
        if (tid == kThreads) {
            const int n_units = a.unit_n[0] + a.unit_n[1] + a.unit_n[2] + a.unit_n[3];
            const long long sstride = fdl_slot_stride<M>(a);
            const uint32_t hb = M * sizeof(float2);
            const uint64_t pol = l2_policy_evict_first();
            const float2* Hsh = ir_replica(a);            // this CTA's copy of the shared IR spectra
            if (a.stagger_ns > 0) {
                // CTAs of a launch run in lockstep (equal work, fair shares of the memory system): spreading their starts
                // spreads where in the partition sequence they are, for the whole launch
                unsigned long long t0, t;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                const unsigned long long wait = (unsigned long long) a.stagger_ns * (blockIdx.x % 64u) / 64u;
                do { asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); } while (t - t0 < wait);
            }
            int st = 0;
            unsigned round = 0;                           // laps of the ring completed by the producer
            for (unsigned ui = 0;; ++ui) {
                const int u = atomicAdd(a.work, 1);
                const int us = ui & 1;
                if (ui >= 2) mbar_wait_relaxed(&sm.u_empty[us], ((ui >> 1) - 1) & 1, a.producer_sleep_ns);     // the compute warps are done with unit ui-2
                PDesc& d = sm.desc[us];
                if (u >= n_units) { d.nrows = 0; mbar_arrive(&sm.u_full[us]); break; }
                int idx = u, base = 0, rows = T::ROWS, lvl = 0;
                while (lvl < 3 && idx >= a.unit_n[lvl]) { idx -= a.unit_n[lvl]; base += a.unit_n[lvl] * rows; rows = rows > 1 ? rows >> 1 : 1; ++lvl; }
                const int row0 = base + idx * rows;
                const int nrows = a.n_rows - row0 < rows ? a.n_rows - row0 : rows;
                int np = 0, ir0 = 0;
                bool uni = a.fdl_group == T::ROWS;        // one copy per slot piece when the rows sit interleaved and move in lockstep
                int hd[T::ROWS], irr[T::ROWS], npr[T::ROWS];
#pragma unroll
                for (int r = 0; r < T::ROWS; ++r) {
                    hd[r] = -1; irr[r] = 0; npr[r] = 0;
                    if (r < nrows) {
                        hd[r] = a.head[row0 + r];
                        irr[r] = (PERROW || r == 0) ? (a.ir_of_chan ? a.ir_of_chan[row0 + r] : 0) : 0;
                    }
                }
#pragma unroll
                for (int r = 0; r < T::ROWS; ++r) {
                    if (r < nrows) {
                        npr[r] = (PERROW || r == 0) ? a.nparts[irr[r]] : npr[0];
                        if (!PERROW) irr[r] = irr[0];
                        np = npr[r] > np ? npr[r] : np;
                        uni = uni && hd[r] == hd[0] && npr[r] == npr[0];
                    }
                    d.hd[r] = hd[r]; d.npr[r] = npr[r];
                }
                ir0 = irr[0];
                d.row0 = row0; d.nrows = nrows; d.np = np;
                mbar_arrive(&sm.u_full[us]);              // release: the descriptor is visible to whoever sees this phase complete
                const float2* fdl0 = a.fdl + fdl_row_offset(a, row0, M);      // row `row0` of its group, slot 0
                int back = 0;                             // partition g >= 1 meets slot (hd - (g - 1)) mod ring
                for (int g = 0; g < np; ++g) {
                    mbar_wait_relaxed(&sm.empty[st], round & 1, a.producer_sleep_ns);      // release number `round` of this stage (number 0: the start-up one)
                    typename PSmem<M, PERROW>::Stage& S = sm.st[st];
                    // bytes this stage will receive
                    uint32_t bytes = 0;
                    if (!PERROW) bytes = hb + (g > 0 ? (uint32_t) nrows * hb : 0u);
                    else {
#pragma unroll
                        for (int r = 0; r < T::ROWS; ++r) if (g < npr[r]) bytes += hb + (g > 0 ? hb : 0u);
                    }
                    mbar_expect_tx(&sm.full[st], bytes);
                    if (!PERROW) tma_bulk_g2s(S.h, Hsh + ir0 * a.ir_stride + (long long) g * M, hb, &sm.full[st]);
                    else {
#pragma unroll
                        for (int r = 0; r < T::ROWS; ++r)
                            if (g < npr[r]) tma_bulk_g2s_hint(S.h + r * M, a.H + irr[r] * a.ir_stride + (long long) g * M, hb, &sm.full[st], pol);
                    }
                    if (g > 0) {
                        if (uni) {
                            int sl = hd[0] - back; if (sl < 0) sl += a.ring;
                            tma_bulk_g2s_hint(S.x, fdl0 + (long long) sl * sstride, (uint32_t) nrows * hb, &sm.full[st], pol);
                        } else {
#pragma unroll
                            for (int r = 0; r < T::ROWS; ++r) {
                                if (g < npr[r]) {
                                    int sl = hd[r] - back; if (sl < 0) sl += a.ring;
                                    tma_bulk_g2s_hint(S.x + r * M, a.fdl + fdl_row_offset(a, row0 + r, M) + (long long) sl * sstride, hb, &sm.full[st], pol);
                                }
                            }
                        }
                        if (++back >= a.ring) back = 0;
                    }
                    if (++st == NSE) { st = 0; ++round; }
                }
            }
        }
        __syncwarp();                                     // the idle lanes rejoin the elected one before the block-wide barrier below
    } else {
        // ===== compute warps =====
        const int g_ = tid / L::TPR, c0 = tid % L::TPR;
        int st = 0;
        unsigned round = 0;
        // Every stage starts out released except the last one of the ring, which the compute warps hold as their first tile.
        int hold = NSE - 1;
        if ((tid & 31) == 0) for (int i = 0; i < NSE - 1; ++i) mbar_arrive(&sm.empty[i]);
        for (unsigned ui = 0;; ++ui) {
            const int us = ui & 1;
            mbar_wait(&sm.u_full[us], (ui >> 1) & 1);
            const PDesc& d = sm.desc[us];
            const int nrows = d.nrows;
            if (nrows == 0) break;
            const int row0 = d.row0, np = d.np;
            float2* tile = sm.st[hold].x;

            // ---- forward transform of the unit's new blocks (FFT layout) ----
            {
                const int rf = tid / T::TPF, t = tid % T::TPF;
                float2 v[kPts];
#pragma unroll
                for (int j = 0; j < kPts; ++j) v[j] = make_float2(0.f, 0.f);
                if (rf < nrows) {
                    const long long i0 = (long long) (row0 + rf) * a.in_chan_stride;
#pragma unroll
                    for (int j = 0; j < kPts; ++j) {
                        const int m = 2 * (t + j * T::TPF);              // scalar loads: a row starts at an odd float offset when B is odd
                        if (m < a.B) v[j].x = load_in(a.in, a.in_fmt, i0 + m);
                        if (m + 1 < a.B) v[j].y = load_in(a.in, a.in_fmt, i0 + m + 1);
                    }
                }
                float2* srow = tile + rf * M;
                fft_run<M, false>(v, t, srow, a.W);
                bar_compute();
#pragma unroll
                for (int j = 0; j < kPts; ++j) srow[t + j * T::TPF] = v[j];
                bar_compute();
            }
            // ---- split into the packed real spectrum (MAC layout): to FDL slot head+1 and into registers as partition 0's operand ----
            float4 x0[L::K][L::V], acc[L::K][L::V];
            int npr[L::K];
#pragma unroll
            for (int s = 0; s < L::K; ++s) {
                const int rl = s * L::G + g_, hd = d.hd[rl];
                npr[s] = PERROW ? d.npr[rl] : np;
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv) { x0[s][vv] = make_float4(0.f, 0.f, 0.f, 0.f); acc[s][vv] = make_float4(0.f, 0.f, 0.f, 0.f); }
                if (hd >= 0) {
                    const int ns = hd + 1 >= a.ring ? 0 : hd + 1;
                    const float2* z = tile + rl * M;
                    float4* dst = reinterpret_cast<float4*>(const_cast<float2*>(a.fdl) + fdl_row_offset(a, row0 + rl, M) + (long long) ns * fdl_slot_stride<M>(a));
#pragma unroll
                    for (int vv = 0; vv < L::V; ++vv) {
                        const int k = 2 * L::f4(c0, vv);
                        const float2 s0 = real_split(z[k], z[(M - k) & (M - 1)], root<false>(a.W, k), k);
                        const float2 s1 = real_split(z[k + 1], z[M - k - 1], root<false>(a.W, k + 1), k + 1);
                        x0[s][vv] = make_float4(s0.x, s0.y, s1.x, s1.y);
                        dst[L::f4(c0, vv)] = x0[s][vv];
                    }
                }
            }
            if (tid < nrows) { const int h = d.hd[tid] + 1; a.head_rw[row0 + tid] = h >= a.ring ? 0 : h; }
            if (np > 0) {
                // this warp is done with the tile: hand the held stage to the producer (generic-proxy writes and reads of the
                // tile precede the async-proxy refill, hence the proxy fence; the stage is free once all eight warps arrived)
                fence_proxy_async_smem();
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&sm.empty[hold]);
            }

            // ---- multiply-accumulate over the partitions, ascending (fp/convolution.cpp:171-202) ----
            for (int g = 0; g < np; ++g) {
                mbar_wait(&sm.full[st], round & 1);
                const typename PSmem<M, PERROW>::Stage& S = sm.st[st];
                uint32_t dep = 0;                         // see mbar_arrive_after
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv) {
                    const int c = L::f4(c0, vv);
                    float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (!PERROW) { h = *reinterpret_cast<const float4*>(&S.h[2 * c]); dep |= __float_as_uint(h.x); }
#pragma unroll
                    for (int s = 0; s < L::K; ++s) {
                        const int rl = s * L::G + g_;
                        if (PERROW) {
                            if (g >= npr[s]) continue;     // this row's IR is shorter (or the row is dead): nothing was staged for it
                            h = *reinterpret_cast<const float4*>(&S.h[rl * M + 2 * c]);
                            dep |= __float_as_uint(h.x);
                        }
                        const float h0i = c == 0 ? 0.f : h.y, h0q = c == 0 ? h.y : h.x;        // bin 0 = packed {DC, Nyquist}
                        float4 xv = x0[s][vv];
                        if (g > 0) {
                            xv = *reinterpret_cast<const float4*>(&S.x[rl * M + 2 * c]);
                            dep |= __float_as_uint(xv.x);
                        }
                        float4& ac = acc[s][vv];
                        ac.x = fmaf(xv.x, h.x, fmaf(-xv.y, h0i, ac.x));
                        ac.y = fmaf(xv.y, h0q, fmaf(xv.x, h0i, ac.y));
                        ac.z = fmaf(xv.z, h.z, fmaf(-xv.w, h.w, ac.z));
                        ac.w = fmaf(xv.w, h.z, fmaf(xv.z, h.w, ac.w));
                    }
                }
                if (g + 1 < np) {
                    release_stage(&sm.empty[st], dep, a, tid);
                } else {
                    hold = st;                            // the last stage of the unit is kept: its FDL area becomes the tile
                }
                if (++st == NSE) { st = 0; ++round; }
            }
            tile = sm.st[hold].x;

            // ---- accumulators -> tile (MAC layout), inverse real FFT in FFT layout, overlap-add, output ----
            bar_compute();                                // every warp is through its last stage: nobody reads the held stage any more
#pragma unroll
            for (int s = 0; s < L::K; ++s)
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv)
                    reinterpret_cast<float4*>(tile + (s * L::G + g_) * M)[L::f4(c0, vv)] = acc[s][vv];
            bar_compute();
            inv_epilogue<M>(a, tile, tid, row0, nrows);
            __syncwarp();
            if ((tid & 31) == 0) mbar_arrive(&sm.u_empty[us]);       // this warp has read everything it needs from the descriptor
        }
    }
    // the last CTA to finish clears the work counter for the next launch (every CTA has stopped fetching by then)
    __syncthreads();
    if (tid == 0) {
        if (stamp_row) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); stamp_row[2] = t; stamp_row[3] = (unsigned long long) clock64(); }
        __threadfence();
        const int done = atomicAdd(a.work + 1, 1);
        if (done == (int) gridDim.x - 1) { a.work[0] = 0; a.work[1] = 0; a.work[2] += 1; __threadfence(); }
    }
}

}  // namespace irb
