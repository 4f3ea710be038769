// irb_mac_mx.cuh -- k_mac_mx: the persistent block step of the IR-MATRIX engine (sm_100a).
//
// The streams come in GROUPS of INS input channels that produce OUTS output channels each:
//   out[g*OUTS + o] = sum_i conv(in[g*INS + i], IR ir[g][i*OUTS + o])
// (mono -> stereo: INS = 1, OUTS = 2; true stereo: INS = OUTS = 2, IRs LL, LR, RL, RR).  Every INPUT keeps one FDL ring with
// exactly the spectra a plain engine row would hold; what differs from k_mac_p is that the ring is read ONCE per block step for
// all the IRs it feeds: a group streams INS delay lines instead of the INS*OUTS a plain engine needs on duplicated inputs.
//
// Built like k_mac_p (irb_mac_p.cuh), same ring protocol: 8 compute warps and one TMA producer warp, units taken from the work
// counter, the producer running ahead across units, every stage released behind fence.proxy.async and a data-dependent arrive,
// the stage consumed last held back as the FFT tile, two CTAs per SM.  A unit is ROWS = kTile/M OUTPUT rows = ROWS/OUTS whole
// groups, so the accumulators per thread and the inverse-FFT tile are exactly k_mac_p's and inv_epilogue<M> is reused with
// output-row indexing.  Per unit:
//   * the prologue forward-transforms the unit's INPUT rows only, writes their packed spectra to FDL slot head+1, keeps them in
//     registers as partition 0's operand and advances the input heads;
//   * a ring stage holds the unit's input rows' FDL piece (one bulk copy when their heads agree) followed by the IR partitions:
//     the INS*OUTS of the unit's matrix (PERGROUP = false: every group of the unit is bound to the same matrix), or every
//     group's own INS*OUTS (PERGROUP = true, the analogue of k_mac_p's PERROW);
//   * matrix IRs may differ in length: the unit streams the longest, a shorter IR contributes nothing past its end.
// Accumulation order (fixed): ascending partition p; within p ascending input i; per term the fmaf sequence of k_mac_p.  For
// INS = 1 an output row is therefore bit-identical to a plain engine row bound to the same IR.
#pragma once
#include "irb_kernels.cuh"

namespace irb {

template <int M, int INS, int OUTS, bool PERGROUP> struct MxCfg {
    static constexpr int ROWS = kTile / M;                 // output rows per unit (k_mac_p's tile)
    static constexpr int GROUPS = ROWS / OUTS;             // groups per unit
    static constexpr int IN_ROWS = GROUPS * INS;           // input rows (FDL rows) per unit
    static constexpr int TERMS = INS * OUTS;               // IRs of one matrix
    static constexpr int HS = PERGROUP ? GROUPS * TERMS : TERMS;      // IR partitions per ring stage
    static constexpr int XF2 = IN_ROWS * M;                // float2 of FDL per ring stage
    static constexpr int HF2 = HS * M;                     // float2 of IR spectra per ring stage
    // The stage held back between units is the FFT tile of the epilogue (ROWS output rows = kTile float2) and spans the stage's
    // FDL AND IR areas; mono -> stereo at M = 256 has less than that per stage and is padded up to it.
    static constexpr int SF2 = XF2 + HF2 > kTile ? XF2 + HF2 : kTile;
    static constexpr int STAGE_BYTES = SF2 * (int) sizeof(float2);
    static constexpr int BUDGET = 113 * 1024 - 1024;       // two CTAs per SM, as k_mac_p
    static constexpr int NS = BUDGET / STAGE_BYTES > 8 ? 8 : BUDGET / STAGE_BYTES;
    static_assert(GROUPS >= 1 && GROUPS * OUTS == ROWS, "groups never straddle a unit");
    static_assert(IN_ROWS <= 8 && HS <= 16, "descriptor capacity");
    static_assert(NS >= 2, "at least two ring stages");
};

struct MxDesc {                    // what the producer tells the compute warps about a unit
    int g0, ng, np;                // first group, live groups (0: no more work), partitions to stream (max over the IRs)
    int hd[8];                     // old head of every input row (-1: dead row)
    int npt[16];                   // partitions of the IR of every stage slot (0: dead group)
};

template <int M, int INS, int OUTS, bool PERGROUP>
struct MxSmem {
    using C = MxCfg<M, INS, OUTS, PERGROUP>;
    float2 st[C::NS][C::SF2];      // [0, XF2): FDL of the input rows; [XF2, XF2 + HF2): IR partitions; st[hold] is the FFT tile
    uint64_t full[C::NS], empty[C::NS], u_full[2], u_empty[2];
    MxDesc desc[2];
};

// a.n_rows = output rows (n_groups * OUTS); a.head / a.head_rw / a.fdl / a.in are over input rows; a.ov / a.out over output
// rows; a.ir_of_chan is the matrix table [n_groups][INS * OUTS]; a.unit_n[0] = units of GROUPS groups (the last one may be
// partial).
template <int M, int INS, int OUTS, bool PERGROUP>
__global__ void __launch_bounds__(kThreads + 32, 2) k_mac_mx(const MacArgs a) {
    using T = Tile<M>;
    using L = MacLayout<M, false>;
    using C = MxCfg<M, INS, OUTS, PERGROUP>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    MxSmem<M, INS, OUTS, PERGROUP>& sm = *reinterpret_cast<MxSmem<M, INS, OUTS, PERGROUP>*>(smem_raw);
    const int tid = threadIdx.x;
    const int NSE = a.ring_stages > 0 && a.ring_stages < C::NS ? a.ring_stages : C::NS;

    if (tid == 0) {
        for (int i = 0; i < 2; ++i) { mbar_init(&sm.u_full[i], 1); mbar_init(&sm.u_empty[i], kThreads / 32); }
        ring_init(sm.full, sm.empty, C::NS);
    }
    __syncthreads();

    if (tid >= kThreads) {
        // ===== TMA producer =====
        if (tid == kThreads) {
            const int n_units = a.unit_n[0];
            const int n_groups = a.n_rows / OUTS;
            const long long sstride = fdl_slot_stride<M>(a);
            const uint32_t hb = M * sizeof(float2);
            const uint64_t pol = l2_policy_evict_first();
            const float2* Hsh = ir_replica(a);
            int st = 0;
            unsigned round = 0;
            for (unsigned ui = 0;; ++ui) {
                const int u = atomicAdd(a.work, 1);
                const int us = ui & 1;
                if (ui >= 2) mbar_wait_relaxed(&sm.u_empty[us], ((ui >> 1) - 1) & 1, a.producer_sleep_ns);
                MxDesc& d = sm.desc[us];
                if (u >= n_units) { d.ng = 0; mbar_arrive(&sm.u_full[us]); break; }
                const int g0 = u * C::GROUPS;
                const int ng = n_groups - g0 < C::GROUPS ? n_groups - g0 : C::GROUPS;
                const int nin = ng * INS, r0 = g0 * INS;
                int hd[C::IN_ROWS], irs[C::HS], npt[C::HS];
                bool uni = a.fdl_group == C::IN_ROWS;     // the unit's input rows are one contiguous piece per slot
#pragma unroll
                for (int r = 0; r < C::IN_ROWS; ++r) {
                    hd[r] = r < nin ? a.head[r0 + r] : -1;
                    if (r < nin) uni = uni && hd[r] == hd[0];
                    d.hd[r] = hd[r];
                }
                int np = 0;
#pragma unroll
                for (int j = 0; j < C::HS; ++j) {
                    const int q = PERGROUP ? j / C::TERMS : 0;
                    irs[j] = q < ng ? a.ir_of_chan[(g0 + q) * C::TERMS + j % C::TERMS] : 0;
                    npt[j] = q < ng ? a.nparts[irs[j]] : 0;
                    np = npt[j] > np ? npt[j] : np;
                    d.npt[j] = npt[j];
                }
                d.g0 = g0; d.ng = ng; d.np = np;
                mbar_arrive(&sm.u_full[us]);              // release: the descriptor is visible to whoever sees this phase complete
                const float2* fdl0 = a.fdl + fdl_row_offset(a, r0, M);
                int back = 0;                             // partition g >= 1 meets slot (hd - (g - 1)) mod ring
                for (int g = 0; g < np; ++g) {
                    mbar_wait_relaxed(&sm.empty[st], round & 1, a.producer_sleep_ns);
                    float2* X = sm.st[st];
                    float2* Hs = X + C::XF2;
                    uint32_t bytes = g > 0 ? (uint32_t) nin * hb : 0u;
#pragma unroll
                    for (int j = 0; j < C::HS; ++j) if (g < npt[j]) bytes += hb;
                    mbar_expect_tx(&sm.full[st], bytes);
#pragma unroll
                    for (int j = 0; j < C::HS; ++j) {
                        if (g < npt[j]) {
                            if (!PERGROUP) tma_bulk_g2s(Hs + j * M, Hsh + irs[j] * a.ir_stride + (long long) g * M, hb, &sm.full[st]);
                            else tma_bulk_g2s_hint(Hs + j * M, a.H + irs[j] * a.ir_stride + (long long) g * M, hb, &sm.full[st], pol);
                        }
                    }
                    if (g > 0) {
                        if (uni) {
                            int sl = hd[0] - back; if (sl < 0) sl += a.ring;
                            tma_bulk_g2s_hint(X, fdl0 + (long long) sl * sstride, (uint32_t) nin * hb, &sm.full[st], pol);
                        } else {
#pragma unroll
                            for (int r = 0; r < C::IN_ROWS; ++r) {
                                if (r < nin) {
                                    int sl = hd[r] - back; if (sl < 0) sl += a.ring;
                                    tma_bulk_g2s_hint(X + r * M, a.fdl + fdl_row_offset(a, r0 + r, M) + (long long) sl * sstride, hb, &sm.full[st], pol);
                                }
                            }
                        }
                        if (++back >= a.ring) back = 0;
                    }
                    if (++st == NSE) { st = 0; ++round; }
                }
            }
        }
        __syncwarp();
    } else {
        // ===== compute warps =====
        const int g_ = L::G == 1 ? 0 : tid / L::TPR, c0 = tid % L::TPR;
        // group (within the unit) and output index of the thread's output row s = s * G + g_, written so that the compiler sees
        // which rows share a group (G == 1: consecutive rows) or an output index (G a multiple of OUTS: all of them)
        auto row_q = [&](int s) { return L::G % OUTS == 0 ? s * (L::G / OUTS) + g_ / OUTS : (s * L::G + g_) / OUTS; };
        auto row_o = [&](int s) { return L::G % OUTS == 0 ? g_ % OUTS : (s * L::G + g_) % OUTS; };
        int st = 0;
        unsigned round = 0;
        int hold = NSE - 1;                               // every stage starts out released except the one held as the first tile
        if ((tid & 31) == 0) for (int i = 0; i < NSE - 1; ++i) mbar_arrive(&sm.empty[i]);
        for (unsigned ui = 0;; ++ui) {
            const int us = ui & 1;
            mbar_wait(&sm.u_full[us], (ui >> 1) & 1);
            const MxDesc& d = sm.desc[us];
            const int ng = d.ng;
            if (ng == 0) break;
            const int g0 = d.g0, np = d.np, nin = ng * INS, r0 = g0 * INS;
            float2* tile = sm.st[hold];

            // ---- forward transform of the unit's new input blocks (FFT layout) ----
            {
                const int rf = tid / T::TPF, t = tid % T::TPF;
                float2 v[kPts];
#pragma unroll
                for (int j = 0; j < kPts; ++j) v[j] = make_float2(0.f, 0.f);
                if (rf < nin) {
                    const long long i0 = (long long) (r0 + rf) * a.in_chan_stride;
#pragma unroll
                    for (int j = 0; j < kPts; ++j) {
                        const int m = 2 * (t + j * T::TPF);
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
            // ---- packed spectra of the inputs every output row of this thread reads: partition 0's operands in registers; the
            //      thread of output 0 of a group also writes them to FDL slot head+1 ----
            float4 x0[L::K][INS][L::V], acc[L::K][L::V];
            int nps[L::K][INS];                           // partitions of every (output row, input) term, 0 for a dead group
#pragma unroll
            for (int s = 0; s < L::K; ++s) {
                const int q = row_q(s), o = row_o(s);
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv) acc[s][vv] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int i = 0; i < INS; ++i) {
                    const int ri = q * INS + i, hd = d.hd[ri];
                    nps[s][i] = hd >= 0 ? d.npt[(PERGROUP ? q * C::TERMS : 0) + i * OUTS + o] : 0;
                    if (L::G == 1 && s % OUTS != 0) {     // the thread's previous output row belongs to the same group: same inputs
#pragma unroll
                        for (int vv = 0; vv < L::V; ++vv) x0[s][i][vv] = x0[s - 1][i][vv];
                        continue;
                    }
#pragma unroll
                    for (int vv = 0; vv < L::V; ++vv) x0[s][i][vv] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (hd >= 0) {
                        const int ns = hd + 1 >= a.ring ? 0 : hd + 1;
                        const float2* z = tile + ri * M;
                        float4* dst = reinterpret_cast<float4*>(const_cast<float2*>(a.fdl) + fdl_row_offset(a, r0 + ri, M) + (long long) ns * fdl_slot_stride<M>(a));
#pragma unroll
                        for (int vv = 0; vv < L::V; ++vv) {
                            const int k = 2 * L::f4(c0, vv);
                            const float2 s0 = real_split(z[k], z[(M - k) & (M - 1)], root<false>(a.W, k), k);
                            const float2 s1 = real_split(z[k + 1], z[M - k - 1], root<false>(a.W, k + 1), k + 1);
                            x0[s][i][vv] = make_float4(s0.x, s0.y, s1.x, s1.y);
                            if (o == 0) dst[L::f4(c0, vv)] = x0[s][i][vv];
                        }
                    }
                }
            }
            if (tid < nin) { const int h = d.hd[tid] + 1; a.head_rw[r0 + tid] = h >= a.ring ? 0 : h; }
            if (np > 0) {
                // done with the tile: hand the held stage to the producer (generic-proxy accesses precede its async-proxy refill)
                fence_proxy_async_smem();
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&sm.empty[hold]);
            }

            // ---- multiply-accumulate: ascending partition, within a partition ascending input ----
            for (int g = 0; g < np; ++g) {
                mbar_wait(&sm.full[st], round & 1);
                const float2* X = sm.st[st];
                const float2* Hs = X + C::XF2;
                uint32_t dep = 0;                         // see mbar_arrive_after
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv) {
                    const int c = L::f4(c0, vv);
#pragma unroll
                    for (int s = 0; s < L::K; ++s) {
                        const int q = row_q(s), o = row_o(s);
                        float4& ac = acc[s][vv];
#pragma unroll
                        for (int i = 0; i < INS; ++i) {
                            if (g >= nps[s][i]) continue;            // this IR is shorter (or the group is dead): nothing staged
                            const float4 h = *reinterpret_cast<const float4*>(&Hs[((PERGROUP ? q * C::TERMS : 0) + i * OUTS + o) * M + 2 * c]);
                            dep |= __float_as_uint(h.x);
                            const float h0i = c == 0 ? 0.f : h.y, h0q = c == 0 ? h.y : h.x;        // bin 0 = packed {DC, Nyquist}
                            float4 xv = x0[s][i][vv];
                            if (g > 0) {
                                xv = *reinterpret_cast<const float4*>(&X[(q * INS + i) * M + 2 * c]);
                                dep |= __float_as_uint(xv.x);
                            }
                            ac.x = fmaf(xv.x, h.x, fmaf(-xv.y, h0i, ac.x));
                            ac.y = fmaf(xv.y, h0q, fmaf(xv.x, h0i, ac.y));
                            ac.z = fmaf(xv.z, h.z, fmaf(-xv.w, h.w, ac.z));
                            ac.w = fmaf(xv.w, h.z, fmaf(xv.z, h.w, ac.w));
                        }
                    }
                }
                if (g + 1 < np) {
                    release_stage(&sm.empty[st], dep, a, tid);
                } else {
                    hold = st;                            // the last stage of the unit is kept: it becomes the tile
                }
                if (++st == NSE) { st = 0; ++round; }
            }
            tile = sm.st[hold];

            // ---- accumulators -> tile (MAC layout), inverse real FFT, overlap-add, output rows ----
            bar_compute();
#pragma unroll
            for (int s = 0; s < L::K; ++s)
#pragma unroll
                for (int vv = 0; vv < L::V; ++vv)
                    reinterpret_cast<float4*>(tile + (s * L::G + g_) * M)[L::f4(c0, vv)] = acc[s][vv];
            bar_compute();
            inv_epilogue<M>(a, tile, tid, g0 * OUTS, ng * OUTS);
            __syncwarp();
            if ((tid & 31) == 0) mbar_arrive(&sm.u_empty[us]);
        }
    }
    // the last CTA to finish clears the work counter for the next launch
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        const int done = atomicAdd(a.work + 1, 1);
        if (done == (int) gridDim.x - 1) { a.work[0] = 0; a.work[1] = 0; a.work[2] += 1; __threadfence(); }
    }
}

}  // namespace irb
