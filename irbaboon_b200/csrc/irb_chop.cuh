// irb_chop.cuh -- sm_100a kernels of fp::ir::IRchop followed by fp::tools::normalize (fp/fp_b200.cpp) on many rows at once:
// the last step of a batched IR capture, which turns each deconvolved row of N samples into an IR of ir_length samples.
//
// Per row x[0, n) (include/irb_b200.h, irb_ir_chop_batch_device, states the rule in full):
//   peak = max |x_i| from 0 with NaN ignored, q = its first index (0 when every sample is NaN);
//   walked = the smallest k >= consecutive such that the walk positions k-consecutive .. k-1 (position j is sample q - j mod n)
//            are all quiet, capped at ir_length (0 when consecutive <= 0); quiet(i) := linTodB(|x_i|) - linTodB(peak) < threshold_db;
//   start = q - walked (mod n), then ir_length samples from start (wrapping), the reference's fades and the normalisation.
// Two kernels: k_chop_peak reduces chunks of every row (several CTAs per row keep the whole GPU reading when the batch is
// small), k_chop_cut takes one row per CTA for the walk (flags and a run-length scan, a tile of positions at a time), the
// cut, the fades and the gain.  The fade and level arithmetic uses explicitly rounded operations (no FMA contraction), so that
// every value is the host's bit for bit.
#pragma once
#include <cuda_runtime.h>

namespace irb {

constexpr int kChopPeakThreads = 256;
constexpr int kChopCutThreads = 512;
constexpr long long kChopNone = 0x7fffffffffffffffLL;          // no index carries the peak (yet)
constexpr float kLn10f = 2.302585092994045684f;                // ln 10, correctly rounded to float (== glibc logf(10.0f))

// tools::linTodB(float) with the correctly rounded float log: v == 0 ? -333 : 20 * ln(v) / ln(10), evaluated left to right in float.
// The log is log((double) v) rounded to float (device double precision); glibc's logf is not correctly rounded, so a level can
// differ from the host's by one ulp on the inputs where the two logs differ.
__device__ __forceinline__ float chop_level_db(float v) {
    if (v == 0.0f) return -333.0f;
    return __fdiv_rn(__fmul_rn(20.0f, __double2float_rn(log((double) v))), kLn10f);
}

// (m, i) := the larger magnitude; on a tie the smaller index
__device__ __forceinline__ void chop_take(float& m, long long& i, float m2, long long i2) {
    if (m2 > m || (m2 == m && i2 < i)) { m = m2; i = i2; }
}

// (m, i) of the whole CTA, valid in every thread; red: 2 * (blockDim / 32) slots
__device__ __forceinline__ void chop_block_peak(float& m, long long& i, float* red_m, long long* red_i) {
    for (int o = 16; o; o >>= 1) chop_take(m, i, __shfl_xor_sync(0xffffffffu, m, o), __shfl_xor_sync(0xffffffffu, i, o));
    const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { red_m[w] = m; red_i[w] = i; }
    __syncthreads();
    m = red_m[0]; i = red_i[0];
    for (int k = 1; k < nw; ++k) chop_take(m, i, red_m[k], red_i[k]);
}

// One CTA per (row, chunk): the chunk's largest |x| (as std::max(m, fabs(x)) from m = 0: NaN never wins) and the first index
// that carries it.  VEC: rows and chunks start at multiples of 4 floats of a 16-byte aligned x.
template <bool VEC>
__global__ void __launch_bounds__(kChopPeakThreads) k_chop_peak(const float* __restrict__ x, long long len, int chunks, long long chunk_len,
                                                                float* __restrict__ part_m, long long* __restrict__ part_i) {
    __shared__ float red_m[kChopPeakThreads / 32];
    __shared__ long long red_i[kChopPeakThreads / 32];
    const long long row = blockIdx.x / chunks, b = (long long) (blockIdx.x % chunks) * chunk_len;
    const long long e = min(len, b + chunk_len);
    const float* p = x + row * len;
    float m = 0.0f;
    long long mi = kChopNone;
    auto see = [&](float v, long long i) {                 // indices of one thread increase: a tie keeps the first
        v = fabsf(v);
        if (v > m || (v == m && mi == kChopNone)) { m = v; mi = i; }
    };
    if (VEC) {
        const float4* p4 = reinterpret_cast<const float4*>(p);
        constexpr int U = 4;
        long long i4 = b / 4 + threadIdx.x;
        const long long e4 = e / 4;
        for (; i4 + (U - 1) * (long long) blockDim.x < e4; i4 += U * (long long) blockDim.x) {
            float4 v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) v[u] = __ldg(p4 + i4 + u * (long long) blockDim.x);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const long long i = 4 * (i4 + u * (long long) blockDim.x);
                see(v[u].x, i); see(v[u].y, i + 1); see(v[u].z, i + 2); see(v[u].w, i + 3);
            }
        }
        for (; i4 < e4; i4 += blockDim.x) {
            const float4 v = __ldg(p4 + i4);
            see(v.x, 4 * i4); see(v.y, 4 * i4 + 1); see(v.z, 4 * i4 + 2); see(v.w, 4 * i4 + 3);
        }
    } else {
        for (long long i = b + threadIdx.x; i < e; i += blockDim.x) see(__ldg(p + i), i);
    }
    chop_block_peak(m, mi, red_m, red_i);
    if (threadIdx.x == 0) { part_m[blockIdx.x] = m; part_i[blockIdx.x] = mi; }
}

struct ChopArgs {
    const float* x;               // [rows][len]
    long long len;
    int chunks;                   // k_chop_peak's chunks per row
    const float* part_m;          // [rows][chunks]
    const long long* part_i;
    int ir_length, consecutive, normalize;
    float threshold_db, goal_lin;
    float* out;                   // [rows][ir_length]
    int* pos;                     // [rows][2] = {q, start}, or null
};

// One CTA per row: the peak from the chunks, the backward walk, the cut with wrap, fade-out, fade-in, the gain.
__global__ void __launch_bounds__(kChopCutThreads) k_chop_cut(ChopArgs a) {
    constexpr int NW = kChopCutThreads / 32;
    __shared__ float red_m[NW];
    __shared__ long long red_i[NW];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const long long row = blockIdx.x, len = a.len;
    const float* p = a.x + row * len;
    float peak = 0.0f;
    long long q = kChopNone;
    for (int c = tid; c < a.chunks; c += blockDim.x) chop_take(peak, q, a.part_m[row * a.chunks + c], a.part_i[row * a.chunks + c]);
    chop_block_peak(peak, q, red_m, red_i);
    if (q == kChopNone) q = 0;
    const float peak_db = chop_level_db(peak);
    const int Lw = a.ir_length, cons = a.consecutive;
    // walked = (first tile position e with a run of >= cons quiet positions ending at e) + 1: run(e) = e - (last loud position <= e)
    long long walked = cons <= 0 ? 0 : Lw;
    if (cons > 0 && cons <= Lw) {
        long long carry = -1;                                // last loud position before the tile
        for (long long base = 0; base < Lw; base += blockDim.x) {
            const long long j = base + tid;
            long long loud = -1;
            if (j < Lw) {
                long long s = q - j;
                if (s < 0) s += len;
                if (!(__fsub_rn(chop_level_db(fabsf(p[s])), peak_db) < a.threshold_db)) loud = j;
            }
            for (int o = 1; o < 32; o <<= 1) {               // inclusive max-scan: in the warp, then over the warps
                const long long v = __shfl_up_sync(0xffffffffu, loud, o);
                if (lane >= o) loud = max(loud, v);
            }
            __syncthreads();
            if (lane == 31) red_i[w] = loud;
            __syncthreads();
            for (int k = 0; k < w; ++k) loud = max(loud, red_i[k]);
            loud = max(loud, carry);
            long long cand = (j < Lw && j - loud >= cons) ? j : kChopNone;
            for (int o = 16; o; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
            long long tile_loud = carry;
            for (int k = 0; k < NW; ++k) tile_loud = max(tile_loud, red_i[k]);
            __syncthreads();
            if (lane == 0) red_i[w] = cand;
            __syncthreads();
            long long e = kChopNone;
            for (int k = 0; k < NW; ++k) e = min(e, red_i[k]);
            if (e != kChopNone) { walked = e + 1; break; }
            carry = tile_loud;
        }
    }
    long long start = q - walked;
    if (start < 0) start += len;
    // the reference's fades: linearFade(IR, false, Lw-1-Lw/4, Lw/4) then linearFade(IR, true, 0, walked/4);
    // gain of sample i' of a fade: i' * step (in) or (float) (1.0 - (double) (i' * step)) (out), step = (float) (1.0 / count)
    const int n_out = Lw / 4, out0 = Lw - 1 - n_out, n_in = (int) (walked / 4);
    const float step_out = n_out ? __double2float_rn(__ddiv_rn(1.0, (double) n_out)) : 0.0f;
    const float step_in = n_in ? __double2float_rn(__ddiv_rn(1.0, (double) n_in)) : 0.0f;
    float* o = a.out + row * (long long) Lw;
    float mag = 0.0f;
    for (int j = tid; j < Lw; j += blockDim.x) {
        long long s = start + j;
        if (s >= len) s -= len;
        float v = p[s];
        if (j >= out0 && j < out0 + n_out) v = __fmul_rn(v, __double2float_rn(__dsub_rn(1.0, (double) __fmul_rn((float) (j - out0), step_out))));
        if (j < n_in) v = __fmul_rn(v, __fmul_rn((float) j, step_in));
        o[j] = v;
        const float av = fabsf(v);
        if (mag < av) mag = av;                             // std::max(mag, fabs(v)): NaN never wins
    }
    if (a.normalize) {                                      // tools::normalize: gain = dBToLin(goal) / getMagnitude, applyGain
        long long unused = 0;
        chop_block_peak(mag, unused, red_m, red_i);
        const float gain = __fdiv_rn(a.goal_lin, mag);
        for (int j = tid; j < Lw; j += blockDim.x) o[j] = __fmul_rn(o[j], gain);      // each thread rescales what it stored
    }
    if (a.pos && tid == 0) { a.pos[2 * row] = (int) q; a.pos[2 * row + 1] = (int) start; }
}

}  // namespace irb
