// irb_ir_load.cuh -- k_ir_load: every IR of a batch turned into the engine's partition spectra in one launch
// (irb_engine_set_irs / _stage_irs; the per-IR irb_engine_set_ir / _stage_ir are its one-row case).
//
// The launch covers three kinds of tiles, in this order:
//   * spectra rows: row r is partition p = r % ring of item j = r / ring of the spectra list.  p < P_j: k_fwd's IR-partition
//     row (the same load with the stereo fold, fft_run<M, false>, real_split), stored to every copy of the spectra; p >= P_j:
//     the partition is cleared in every copy.  The fixed stride `ring` lets a row find its item with one division.
//   * staging pieces: kPiece samples of the round-robin buffer of an item of the staging list (the taps, zero-extended to
//     ring * B, folded as above), in the rr_taps table k_fwd's refresh rows read; piece 0 also restarts rr_pos when asked.
// Spectra are bit-identical to k_fwd's, so a batch load gives what a loop of per-IR loads gave.
#pragma once
#include "irb_kernels.cuh"

namespace irb {

// one item of a load (a row of the caller's batch), 24 bytes
struct IrLoadItem {
    long long off;             // first sample, relative to IrLoadArgs::src (and src2)
    int len;                   // samples to read (spectra: n_taps; staging: the taps kept)
    int ir;                    // destination IR
    int P;                     // spectra list: partitions transformed (the rest of the ring is cleared); staging list: restart rr_pos when 1
    int pad;
};

struct IrLoadArgs {
    const IrLoadItem* items;   // [n_x] spectra list, then [n_s] staging list
    int n_x, n_s;
    const float* src;          // taps, any 4-byte alignment
    const float* src2;         // nullable: folded in as (a + b) / 2
    int B, ring;
    float2* H;
    long long ir_stride;       // float2 units
    int h_reps;
    long long h_rep_stride;
    const float2* W;
    float* const* rr_taps;     // round-robin buffers [ir], ring * B samples each
    int* rr_pos;
};

constexpr int kPiece = 2048;   // samples of a round-robin buffer per staging tile

__device__ __forceinline__ float ir_load_sample(const IrLoadArgs& a, long long i) {
    float x = a.src[i];
    if (a.src2) { x += a.src2[i]; x /= 2.0f; }
    return x;
}

template <int M>
__global__ void __launch_bounds__(kThreads) k_ir_load(const IrLoadArgs a) {
    using T = Tile<M>;
    __shared__ __align__(16) float2 s_spec[kTile];
    const int tid = threadIdx.x;
    const long long x_rows = (long long) a.n_x * a.ring;
    const long long x_tiles = (x_rows + T::ROWS - 1) / T::ROWS;
    if ((long long) blockIdx.x >= x_tiles) {          // a staging piece (the whole CTA returns here)
        const long long t = blockIdx.x - x_tiles, cap = (long long) a.ring * a.B;
        const long long pieces = (cap + kPiece - 1) / kPiece;
        const IrLoadItem it = a.items[a.n_x + t / pieces];
        const long long i0 = (t % pieces) * kPiece;
        float* dst = a.rr_taps[it.ir];
        for (long long i = i0 + tid; i < i0 + kPiece && i < cap; i += kThreads) dst[i] = i < it.len ? ir_load_sample(a, it.off + i) : 0.f;
        if (i0 == 0 && tid == 0 && it.P) a.rr_pos[it.ir] = 0;
        return;
    }
    // row of this thread in the FFT layout, then in the MAC layout: (item, partition); xf: a transform row, else cleared (or dead)
    struct Row { float2* d; const float* p; const float* q; int len; bool live, xf; };
    auto row = [&](int r) {
        Row w{nullptr, nullptr, nullptr, 0, false, false};
        const long long g = (long long) blockIdx.x * T::ROWS + r;
        if (g >= x_rows) return w;
        const int j = (int) (g / a.ring), p = (int) (g % a.ring);
        const IrLoadItem it = a.items[j];
        w.live = true;
        w.d = a.H + it.ir * a.ir_stride + (long long) p * M;
        if (p >= it.P) return w;
        w.xf = true;
        const int len = it.len - p * a.B;
        w.len = len > a.B ? a.B : len;
        w.p = a.src + it.off + (long long) p * a.B;
        w.q = a.src2 ? a.src2 + it.off + (long long) p * a.B : nullptr;
        return w;
    };
    const int rf = tid / T::TPF, t = tid % T::TPF;
    const Row wf = row(rf);
    if (__syncthreads_or(wf.xf)) {                    // some row of the tile is transformed: the whole CTA runs the FFT
        float2 v[kPts];
#pragma unroll
        for (int j = 0; j < kPts; ++j) v[j] = make_float2(0.f, 0.f);
        if (wf.xf) {
#pragma unroll
            for (int j = 0; j < kPts; ++j) {
                const int m = 2 * (t + j * T::TPF);
                float x0 = 0.f, x1 = 0.f;
                if (m < wf.len) x0 = wf.p[m];
                if (m + 1 < wf.len) x1 = wf.p[m + 1];
                if (wf.q) {
                    if (m < wf.len) { x0 += wf.q[m]; x0 /= 2.0f; }
                    if (m + 1 < wf.len) { x1 += wf.q[m + 1]; x1 /= 2.0f; }
                }
                v[j] = make_float2(x0, x1);
            }
        }
        float2* srow = s_spec + rf * M;
        fft_run<M, false>(v, t, srow, a.W);
        bar_compute();
#pragma unroll
        for (int j = 0; j < kPts; ++j) srow[t + j * T::TPF] = v[j];
        bar_compute();
    }
    // MAC layout: the packed real spectrum (or zeros) to every copy, 16 B per lane
    const int g = tid / T::TPR, c0 = tid % T::TPR;
    const int reps = a.h_reps > 1 ? a.h_reps : 1;
#pragma unroll
    for (int s = 0; s < T::K; ++s) {
        const int rl = s * T::G + g;
        const Row w = row(rl);
        if (!w.live) continue;
        const float2* z = s_spec + rl * M;
#pragma unroll
        for (int vv = 0; vv < T::V; ++vv) {
            const int k = 2 * (c0 + vv * T::TPR);
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            if (w.xf) {
                const float2 x0 = real_split(z[k], z[(M - k) & (M - 1)], root<false>(a.W, k), k);
                const float2 x1 = real_split(z[k + 1], z[M - k - 1], root<false>(a.W, k + 1), k + 1);
                o = make_float4(x0.x, x0.y, x1.x, x1.y);
            }
            for (int rep = 0; rep < reps; ++rep) *reinterpret_cast<float4*>(w.d + rep * a.h_rep_stride + k) = o;
        }
    }
}

}  // namespace irb
