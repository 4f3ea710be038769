// irb_spectral.cuh -- sm_100a kernels of the single large real FFT path: fp::convolution::convolveNonPeriodic
// (fp/convolution.cpp:246-347), deconvolve (:351-403), averagingFilter (:406-546), tools::fftTransform /
// fftInvTransform (fp/tools.cpp:321-369).  These replace the third-party juce::dsp::FFT calls at
// fp/convolution.cpp:286-288,308,315,336 and fp/tools.cpp:331-335,359-363 for N = 2^4 ... 2^22.
//
// An N-point real transform is one M = N/2 point complex FFT of z[n] = x[2n] + i x[2n+1] plus a split pass.
// M <= 2048 is one shared-memory Stockham FFT per line.  Larger M = M1*M2 is the four-step scheme in two
// kernels launches of the same kernel: M2 column FFTs of length M1 (strided lines, tiled so every global access
// is a >= 64-byte segment) with the inter-pass twiddle exp(-2 pi i n2 k1 / M) computed in double, then M1 row
// FFTs of length M2 written back in NATURAL bin order, so every per-bin stage is a plain elementwise kernel.
#pragma once
#include "irb_kernels.cuh"

namespace irb {

template <int L> struct LineTile {
    static constexpr int TPF = L / kPts;                                   // threads per line
    static constexpr int G = kThreads / TPF;                               // lines transformed concurrently
    static constexpr int C = L >= 2048 ? 4 : (G > 8 ? G : 8);              // lines per CTA tile
    static constexpr int PITCH = L + 2;                                    // float2 per line in shared memory (bank spread)
    static constexpr size_t SMEM = sizeof(float2) * (size_t) C * PITCH;
};

struct LineArgs {
    const void* in;               // complex float2, or real float when in_real_len >= 0
    float2* out;
    long long in_elem_stride, in_line_stride, in_batch_stride;      // float2 units (complex view)
    long long out_elem_stride, out_line_stride, out_batch_stride;
    int n_lines;                  // lines per batch item (grid.y = batch)
    int in_real_len;              // >= 0: input is real, this many valid floats per batch item, zero beyond
    int tw_M;                     // > 0: multiply output element k of line l by exp(-+2 pi i l k / tw_M)
    const float2 *tw_hi, *tw_lo;  // that root as tw_hi[idx >> 10] * tw_lo[idx & 1023], idx = l k mod tw_M (tables built in double)
    float scale;                  // applied on store
    const float2* W;              // the 2L roots of unity of the line length
};
// Real-output window of an inverse transform's last pass (k_line_fft_win): the output element n = line * out_line_stride +
// j * out_elem_stride of batch item b is the pair of floats 2n, 2n+1 of that item's real result; only floats f in [off, off + len)
// are written, one scalar store each, to ((float*) out)[b * stride + f - off], so `out` needs 4-byte alignment only
// (out_batch_stride is unused)
struct LineWindow {
    long long off, stride;
    int len;
};

constexpr int kTwLoBits = 10;
// exp(-2 pi i idx / M) from the two-level table: one complex product of two correctly rounded factors
__device__ __forceinline__ float2 root_big(const float2* __restrict__ hi, const float2* __restrict__ lo, long long idx) {
    return cmul(__ldg(hi + (idx >> kTwLoBits)), __ldg(lo + (idx & ((1 << kTwLoBits) - 1))));
}

template <int L, bool INV>
#ifndef IRB_LINE_CTAS
#define IRB_LINE_CTAS 4                  // resident CTAs per SM the line kernels (L < 1024) are compiled for
#endif
static __global__ void __launch_bounds__(kThreads, L >= 1024 ? 2 : IRB_LINE_CTAS) k_line_fft(const LineArgs a) {
    using T = LineTile<L>;
    extern __shared__ __align__(16) float2 s_lines[];
    __shared__ float2 s_step[T::C][kPts];                 // inter-pass twiddle: root(line * TPF * j), the same for every thread of a line
    const int tid = threadIdx.x;
    const int line0 = blockIdx.x * T::C;
    const long long ib = (long long) blockIdx.y * a.in_batch_stride, ob = (long long) blockIdx.y * a.out_batch_stride;
    const bool in_contig = a.in_elem_stride == 1, out_contig = a.out_elem_stride == 1;
    if (a.tw_M > 0) {
        for (int i = tid; i < T::C * kPts; i += kThreads) {
            const int c = i / kPts, j = i % kPts;
            s_step[c][j] = root_big(a.tw_hi, a.tw_lo, ((long long) (line0 + c) * T::TPF * j) & (a.tw_M - 1));
        }
    }

    // all of a thread's loads are issued before the first shared-memory store: PER x 8 bytes in flight per thread
    constexpr int PER = T::C * L / kThreads;
    {
        float2 r[PER];
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int idx = tid + i * kThreads;
            const int c = in_contig ? idx / L : idx % T::C;
            const int j = in_contig ? idx % L : idx / T::C;
            const int line = line0 + c;
            float2 v = make_float2(0.f, 0.f);
            if (line < a.n_lines) {
                const long long off = (long long) line * a.in_line_stride + (long long) j * a.in_elem_stride;
                if (a.in_real_len < 0) v = reinterpret_cast<const float2*>(a.in)[ib + off];
                else {
                    const float* rp = reinterpret_cast<const float*>(a.in) + 2 * ib;
                    const long long e = 2 * off;
                    if (e + 1 < a.in_real_len) v = *reinterpret_cast<const float2*>(rp + e);
                    else if (e < a.in_real_len) v.x = rp[e];
                }
            }
            r[i] = v;
        }
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int idx = tid + i * kThreads;
            const int c = in_contig ? idx / L : idx % T::C;
            const int j = in_contig ? idx % L : idx / T::C;
            s_lines[c * T::PITCH + j] = r[i];
        }
    }
    bar_compute();
    {
        const int t = tid % T::TPF;
        for (int c = tid / T::TPF; c < T::C; c += T::G) {
            float2* srow = s_lines + c * T::PITCH;
            float2 v[kPts];
            fft_gather<L>(v, t, srow);
            fft_run<L, INV>(v, t, srow, a.W);
            const int line = line0 + c;
            float2 tw_base = make_float2(1.f, 0.f);
            if (a.tw_M > 0) tw_base = root_big(a.tw_hi, a.tw_lo, ((long long) line * t) & (a.tw_M - 1));
#pragma unroll
            for (int j = 0; j < kPts; ++j) {
                const int k = t + j * T::TPF;
                if (a.tw_M > 0) {
                    // root(line*k), k = t + j*TPF, as root(line*t) * root(line*TPF*j): the second factor is the same for
                    // the whole line and was looked up once per CTA (a broadcast read of shared memory here)
                    const float2 w = cmul(tw_base, s_step[c][j]);
                    v[j] = cmul(v[j], INV ? cconj(w) : w);
                }
                srow[k] = v[j];              // each thread rewrites exactly the elements it gathered last
            }
        }
    }
    bar_compute();
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int idx = tid + i * kThreads;
        const int c = out_contig ? idx / L : idx % T::C;
        const int j = out_contig ? idx % L : idx / T::C;
        const int line = line0 + c;
        if (line < a.n_lines) {
            float2 v = s_lines[c * T::PITCH + j];
            v.x *= a.scale; v.y *= a.scale;
            a.out[ob + (long long) line * a.out_line_stride + (long long) j * a.out_elem_stride] = v;
        }
    }
}

// k_line_fft<L, true> whose last pass stores only the window w of each batch item's real result (LineWindow).  A copy rather than
// a branch or a template argument of k_line_fft: any change to that kernel's source or arguments changes the code ptxas makes of
// it (a run-time branch cost the division's device path 2 %), and the plain transforms are the hot path of the batched division.
template <int L>
static __global__ void __launch_bounds__(kThreads, L >= 1024 ? 2 : IRB_LINE_CTAS) k_line_fft_win(const LineArgs a, const LineWindow w) {
    constexpr bool INV = true;
    using T = LineTile<L>;
    extern __shared__ __align__(16) float2 s_lines[];
    __shared__ float2 s_step[T::C][kPts];                 // inter-pass twiddle: root(line * TPF * j), the same for every thread of a line
    const int tid = threadIdx.x;
    const int line0 = blockIdx.x * T::C;
    const long long ib = (long long) blockIdx.y * a.in_batch_stride;
    const bool in_contig = a.in_elem_stride == 1, out_contig = a.out_elem_stride == 1;
    if (a.tw_M > 0) {
        for (int i = tid; i < T::C * kPts; i += kThreads) {
            const int c = i / kPts, j = i % kPts;
            s_step[c][j] = root_big(a.tw_hi, a.tw_lo, ((long long) (line0 + c) * T::TPF * j) & (a.tw_M - 1));
        }
    }

    // all of a thread's loads are issued before the first shared-memory store: PER x 8 bytes in flight per thread
    constexpr int PER = T::C * L / kThreads;
    {
        float2 r[PER];
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int idx = tid + i * kThreads;
            const int c = in_contig ? idx / L : idx % T::C;
            const int j = in_contig ? idx % L : idx / T::C;
            const int line = line0 + c;
            float2 v = make_float2(0.f, 0.f);
            if (line < a.n_lines) {
                const long long off = (long long) line * a.in_line_stride + (long long) j * a.in_elem_stride;
                if (a.in_real_len < 0) v = reinterpret_cast<const float2*>(a.in)[ib + off];
                else {
                    const float* rp = reinterpret_cast<const float*>(a.in) + 2 * ib;
                    const long long e = 2 * off;
                    if (e + 1 < a.in_real_len) v = *reinterpret_cast<const float2*>(rp + e);
                    else if (e < a.in_real_len) v.x = rp[e];
                }
            }
            r[i] = v;
        }
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int idx = tid + i * kThreads;
            const int c = in_contig ? idx / L : idx % T::C;
            const int j = in_contig ? idx % L : idx / T::C;
            s_lines[c * T::PITCH + j] = r[i];
        }
    }
    bar_compute();
    {
        const int t = tid % T::TPF;
        for (int c = tid / T::TPF; c < T::C; c += T::G) {
            float2* srow = s_lines + c * T::PITCH;
            float2 v[kPts];
            fft_gather<L>(v, t, srow);
            fft_run<L, INV>(v, t, srow, a.W);
            const int line = line0 + c;
            float2 tw_base = make_float2(1.f, 0.f);
            if (a.tw_M > 0) tw_base = root_big(a.tw_hi, a.tw_lo, ((long long) line * t) & (a.tw_M - 1));
#pragma unroll
            for (int j = 0; j < kPts; ++j) {
                const int k = t + j * T::TPF;
                if (a.tw_M > 0) {
                    // root(line*k), k = t + j*TPF, as root(line*t) * root(line*TPF*j): the second factor is the same for
                    // the whole line and was looked up once per CTA (a broadcast read of shared memory here)
                    const float2 w = cmul(tw_base, s_step[c][j]);
                    v[j] = cmul(v[j], INV ? cconj(w) : w);
                }
                srow[k] = v[j];              // each thread rewrites exactly the elements it gathered last
            }
        }
    }
    bar_compute();
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int idx = tid + i * kThreads;
        const int c = out_contig ? idx / L : idx % T::C;
        const int j = out_contig ? idx % L : idx / T::C;
        const int line = line0 + c;
        if (line < a.n_lines) {
            float2 v = s_lines[c * T::PITCH + j];
            v.x *= a.scale; v.y *= a.scale;
            const long long f = 2 * ((long long) line * a.out_line_stride + (long long) j * a.out_elem_stride) - w.off;
            float* o = reinterpret_cast<float*>(a.out) + blockIdx.y * w.stride + f;
            if (f >= 0 && f < w.len) o[0] = v.x;
            if (f + 1 >= 0 && f + 1 < w.len) o[1] = v.y;
        }
    }
}

// ---- elementwise stages on natural-order arrays; grid.y = batch item ------------------------------------
// W2M: the N = 2M roots exp(-2 pi i k / N) (table for M <= 2048, else computed in double)
__device__ __forceinline__ float2 root_N(const float2* __restrict__ W, int M, int k) {
    if (W) return __ldg(W + k);
    double sn, cs;
    sincospi((double) k / (double) M, &sn, &cs);
    return make_float2((float) cs, (float) -sn);
}

// Z (M complex) -> interleaved spectrum S: bins 0..M, and with `mirror` the conjugate bins M+1..2M-1 as the
// full complex transform of a real signal has them (2N floats per channel, N = 2M)
static __global__ void k_spec_split(const float2* Z, long long z_stride, float2* S, long long s_stride, int M, int mirror, const float2* W) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    const float2* z = Z + blockIdx.y * z_stride;
    float2* s = S + blockIdx.y * s_stride;
    float2 x;
    if (k == 0) x = make_float2(z[0].x + z[0].y, 0.f);
    else if (k == M) x = make_float2(z[0].x - z[0].y, 0.f);
    else x = real_split(z[k], z[M - k], root_N(W, M, k), k);
    s[k] = x;
    if (mirror && k > 0 && k < M) s[2 * M - k] = make_float2(x.x, -x.y);
}
// interleaved spectrum S (bins 0..M read) -> Z' (M complex) ready for the inverse complex FFT
static __global__ void k_spec_merge(const float2* S, long long s_stride, float2* Z, long long z_stride, int M, const float2* W) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= M) return;
    const float2* s = S + blockIdx.y * s_stride;
    float2* z = Z + blockIdx.y * z_stride;
    if (k == 0) {
        // the reference's inverse reads bins 0 and M as complex values; their imaginary parts enter the rebuilt
        // spectrum but cancel in a real output except through x[0] and the alternating term: keep the real parts
        z[0] = make_float2(s[0].x + s[M].x, s[0].x - s[M].x);
    } else z[k] = real_merge(s[k], s[M - k], root_N(W, M, k), k);
}
// tools::complexMul (fp/tools.cpp:44-52) / complexDivCartesian (:72-86) per bin
__device__ __forceinline__ float2 bin_mul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.y * b.x + a.x * b.y); }
__device__ __forceinline__ float2 bin_div(float2 a, float2 b) {
    if (b.x == 0.0f && b.y == 0.0f) return a;
    const float den = b.x * b.x + b.y * b.y;
    return make_float2((a.x * b.x + a.y * b.y) / den, (a.y * b.x - a.x * b.y) / den);
}
// S[k] = op(A[k], B[k]) on bins 0..M of interleaved spectra (B broadcast over the batch when b_stride == 0)
template <bool DIV>
static __global__ void k_spec_binop(float2* A, long long a_stride, const float2* Bs, long long b_stride, int M) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    float2* pa = A + blockIdx.y * a_stride;
    const float2 b = Bs[blockIdx.y * b_stride + k];
    pa[k] = DIV ? bin_div(pa[k], b) : bin_mul(pa[k], b);
}
// fused split -> per-bin op -> merge on the pair (k, M-k): Za op Zb -> Z' without materialising the spectra
template <bool DIV>
static __global__ void k_spec_fused(const float2* Za, long long a_stride, const float2* Zb, long long b_stride, float2* Zo, long long o_stride, int M,
                             const float2* W) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M / 2) return;
    const float2* za = Za + blockIdx.y * a_stride;
    const float2* zb = Zb + blockIdx.y * b_stride;
    float2* zo = Zo + blockIdx.y * o_stride;
    if (k == 0) {
        const float2 a0 = make_float2(za[0].x + za[0].y, 0.f), aM = make_float2(za[0].x - za[0].y, 0.f);
        const float2 b0 = make_float2(zb[0].x + zb[0].y, 0.f), bM = make_float2(zb[0].x - zb[0].y, 0.f);
        const float2 q0 = DIV ? bin_div(a0, b0) : bin_mul(a0, b0), qM = DIV ? bin_div(aM, bM) : bin_mul(aM, bM);
        zo[0] = make_float2(q0.x + qM.x, q0.x - qM.x);
        return;
    }
    const float2 w = root_N(W, M, k), wm = root_N(W, M, M - k);
    const float2 ak = za[k], am = za[M - k], bk = zb[k], bm = zb[M - k];
    const float2 A = real_split(ak, am, w, k), Am = real_split(am, ak, wm, M - k);
    const float2 B = real_split(bk, bm, w, k), Bm = real_split(bm, bk, wm, M - k);
    const float2 Q = DIV ? bin_div(A, B) : bin_mul(A, B), Qm = DIV ? bin_div(Am, Bm) : bin_mul(Am, Bm);
    zo[k] = real_merge(Q, Qm, w, k);
    if (2 * k != M) zo[M - k] = real_merge(Qm, Q, wm, M - k);
}

// ---- fused middle of the large transform pair (M = M1*M2 > 2048) ----------------------------------------------
// After the column pass the M-point spectrum of one signal lies as M1 rows of M2 values; row k1 becomes the bins
// k = k1 + M1*k2 once its M2-point row FFT is done.  The per-bin stage needs the bin pair (k, M-k), which lives in rows
// k1 and M1-k1, so ONE CTA takes that pair of rows through: forward row FFT -> split into the real signal's spectrum
// -> multiply / divide by the other operand's spectrum B -> merge back -> inverse row FFT -> inter-pass twiddle of
// the inverse transform, all in shared memory.  The inverse column pass then finishes.  Per signal this replaces
// forward row pass + bin kernel + inverse column pass with twiddle (3 x 8M bytes) by 1 x 8M bytes.
// B is given in the same row layout, already split: Brows[k1*M2 + k2] = B[k1 + M1*k2], Brows[0] = {B[0], B[M]} (both real).
template <int L> struct PairTile {
    static constexpr int TPF = L / kPts;                                   // threads per row
    static constexpr int G = kThreads / TPF;                               // rows transformed concurrently
    static constexpr int NP = G >= 2 ? G / 2 : 1;                          // row pairs per CTA
    static constexpr int PITCH = L + 2;
    static constexpr size_t SMEM = sizeof(float2) * (size_t) (2 * NP) * PITCH;
};
struct PairArgs {
    float2* Z;                   // [batch][M1][M2] rows, in place
    long long z_batch_stride;
    const float2* Brows;         // [nb][M1*M2]
    long long b_batch_stride;    // 0: one B for the whole batch
    int M1;                      // rows (M2 = L is the template parameter)
    const float2 *W;             // the 2L roots (row transforms)
    const float2 *Nhi, *Nlo;     // two-level table of the 2M-th roots (split / merge)
    const float2 *Mhi, *Mlo;     // two-level table of the M-th roots (inverse inter-pass twiddle)
};
// exp(-2 pi i j / 16), j = 0 .. 7 (correctly rounded)
__device__ __forceinline__ float2 root16(int j) {
    constexpr float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f, h = 0.70710678118654752440f;
    switch (j) {
        case 0: return make_float2(1.f, 0.f);
        case 1: return make_float2(c1, -s1);
        case 2: return make_float2(h, -h);
        case 3: return make_float2(s1, -c1);
        case 4: return make_float2(0.f, -1.f);
        case 5: return make_float2(-s1, -c1);
        case 6: return make_float2(-h, -h);
        default: return make_float2(-c1, -s1);
    }
}
// Z'[k] of the bin pair (k, M-k): split both bins of the real signal's spectrum, multiply by B, merge back.
// Division is multiplication by the reciprocal spectrum that k_split_rows prepares once for the whole batch.
__device__ __forceinline__ float2 pair_op(float2 zk, float2 zm, float2 bk, float2 bm, float2 w) {
    const float2 wm = make_float2(-w.x, w.y);                              // root of M-k = -conj(root of k)
    const float2 A = real_split(zk, zm, w, 1), Am = real_split(zm, zk, wm, 1);
    return real_merge(bin_mul(A, bk), bin_mul(Am, bm), w, 1);
}
// Every thread owns 8 values of ONE row from the global load to the global store (FFT layout: k2 = t + j*L/8).  The only
// traffic through shared memory besides the exchanges of the two transforms is one natural-order copy of the
// forward result, from which a thread reads the partners Z[M-k] of its own 8 bins; both owners of a pair evaluate
// the pair, each keeping its own half, which costs arithmetic but no second exchange.
template <int L>
#ifndef IRB_ROWPAIR_CTAS
#define IRB_ROWPAIR_CTAS 4               // resident CTAs per SM the row-pair kernel is compiled for (register budget)
#endif
static __global__ void __launch_bounds__(kThreads, IRB_ROWPAIR_CTAS) k_rowpair(const PairArgs a) {
    using T = PairTile<L>;
    extern __shared__ __align__(16) float2 s_lines[];
    __shared__ float2 s_step[2 * T::NP][kPts];            // inverse inter-pass twiddle steps root_M(row * TPF * j), one set per line
    const int tid = threadIdx.x, M1 = a.M1;
    const long long M = (long long) M1 * L;
    float2* Z = a.Z + blockIdx.y * a.z_batch_stride;
    const float2* Bq = a.Brows + blockIdx.y * a.b_batch_stride;
    // line 2i = row p, line 2i+1 = row M1-p, p = blockIdx.x*NP + i in 0 .. M1/2; rows 0 and M1/2 pair with themselves
    const int line = tid / T::TPF, t = tid % T::TPF;
    const int p = blockIdx.x * T::NP + line / 2;
    const bool selfrow = p == 0 || 2 * p == M1;
    const bool live = line < 2 * T::NP && p <= M1 / 2 && !((line & 1) && selfrow);
    const int row = live ? ((line & 1) ? M1 - p : p) : 0;
    const int prow = selfrow ? row : M1 - row;                            // the row holding the partners
    float2* srow = s_lines + line * T::PITCH;
    const float2* spart = selfrow ? srow : s_lines + (line ^ 1) * T::PITCH;
    float2* zrow = Z + (long long) row * L;
    float2 v[kPts];
#pragma unroll
    for (int j = 0; j < kPts; ++j) v[j] = live ? zrow[t + j * T::TPF] : make_float2(0.f, 0.f);
    if (t < kPts && line < 2 * T::NP) s_step[line][t] = root_big(a.Mhi, a.Mlo, ((long long) row * T::TPF * t) & (M - 1));
    // split / merge root of this thread's bins k = row + M1*(t + j*TPF): exp(-2 pi i k / 2M) = root_2M(row + M1*t) * exp(-2 pi i j / 16)
    // (M1 * TPF / 2M = 1/16), one table read and the sixteenth roots of unity as constants
    const float2 n_base = root_big(a.Nhi, a.Nlo, row + (long long) M1 * t);
    fft_run<L, false>(v, t, srow, a.W);                                   // forward row transform: v[j] = Z[row + M1*(t + j*TPF)]
    bar_compute();
#pragma unroll
    for (int j = 0; j < kPts; ++j) srow[t + j * T::TPF] = v[j];
    bar_compute();
    if (live) {
#pragma unroll
        for (int j = 0; j < kPts; ++j) {
            const int k2 = t + j * T::TPF;
            const int pk2 = row == 0 ? (L - k2) & (L - 1) : L - 1 - k2;      // element of M-k in its row
            const long long k = row + (long long) M1 * k2;
            if (k == 0) {
                const float2 z0 = v[j], b0 = __ldg(Bq);
                const float2 a0 = make_float2(z0.x + z0.y, 0.f), aM = make_float2(z0.x - z0.y, 0.f);
                const float2 bb0 = make_float2(b0.x, 0.f), bbM = make_float2(b0.y, 0.f);
                const float2 q0 = bin_mul(a0, bb0), qM = bin_mul(aM, bbM);
                v[j] = make_float2(q0.x + qM.x, q0.x - qM.x);
            } else {
                v[j] = pair_op(v[j], spart[pk2], __ldg(Bq + (long long) row * L + k2), __ldg(Bq + (long long) prow * L + pk2), cmul(n_base, root16(j)));
            }
        }
    }
    fft_run<L, true>(v, t, srow, a.W);                                    // its first barrier orders the partner reads before the scatter
    if (live) {
        // inter-pass twiddle conj(root_M(row*n2)), n2 = t + j*TPF, as root(row*t) * root(row*TPF*j) (one table line per warp)
        const float2 tw_base = root_big(a.Mhi, a.Mlo, ((long long) row * t) & (M - 1));
#pragma unroll
        for (int j = 0; j < kPts; ++j) {
            const float2 w = cmul(tw_base, s_step[line][j]);             // written before the first barrier of the forward transform
            zrow[t + j * T::TPF] = cmul(v[j], cconj(w));
        }
    }
}
// the other operand: Zrows (row layout after its own row FFTs, same place) -> Brows, the split spectrum in row layout
// reciprocal: Brows holds 1/B instead, with the reference's rule for an all-zero bin (tools::complexDivCartesian,
// fp/tools.cpp:72-76: the numerator stays as it is) expressed as the factor 1
__device__ __forceinline__ float2 bin_recip(float2 b) {
    if (b.x == 0.0f && b.y == 0.0f) return make_float2(1.0f, 0.0f);
    const float den = b.x * b.x + b.y * b.y;
    return make_float2(b.x / den, -b.y / den);
}
static __global__ void k_split_rows(const float2* Zrows, float2* Brows, int M1, int L, const float2* Nhi, const float2* Nlo, int reciprocal) {
    const long long M = (long long) M1 * L;
    const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const float2* z = Zrows + blockIdx.y * M;
    float2* b = Brows + blockIdx.y * M;
    const int k1 = (int) (i / L), k2 = (int) (i % L);
    const long long k = k1 + (long long) M1 * k2;
    if (k == 0) {
        float b0 = z[0].x + z[0].y, bM = z[0].x - z[0].y;
        if (reciprocal) { b0 = b0 == 0.0f ? 1.0f : 1.0f / b0; bM = bM == 0.0f ? 1.0f : 1.0f / bM; }
        b[0] = make_float2(b0, bM);
        return;
    }
    const int r = k1 == 0 ? 0 : M1 - k1, e = k1 == 0 ? (L - k2) & (L - 1) : L - 1 - k2;
    const float2 v = real_split(z[i], z[(long long) r * L + e], root_big(Nhi, Nlo, k), 1);
    b[i] = reciprocal ? bin_recip(v) : v;
}

// tools::fftTransform(formatAmplPhase = true): bins 0..M -> {amplitude, phase} (fp/tools.cpp:337-342,222-231)
static __global__ void k_spec_ampl_phase(float2* S, long long s_stride, int M) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    float2* s = S + blockIdx.y * s_stride;
    const float2 v = s[k];
    s[k] = make_float2((float) sqrt((double) v.x * (double) v.x + (double) v.y * (double) v.y), atan2f(v.y, v.x));
}

// ---- averagingFilter (fp/convolution.cpp:406-546), one pass = three kernels ------------------------------
__device__ __forceinline__ float round_1e16(float x) {                  // tools::roundTo1TenQuadrillionth, fp/tools.cpp:212-218
    if (!signbit(x) && (double) x < 1e-16) return 1e-16f;
    if (signbit(x) && (double) x > -1e-16) return -1e-16f;
    return x;
}
__device__ __forceinline__ float round_to_zero(float x, float thr) {   // tools::roundToZero, fp/tools.cpp:199-209
    if (!signbit(x) && x < thr) x = 0.0f;
    if (signbit(x) && x > -thr) x = 0.0f;
    return x;
}
// (0) once per call: the window [lo, hi] of every bin k <= M with the reference's double-precision operation order
// (fp/convolution.cpp:451-458): binFreq = k*freqPerBin; lo = round((binFreq / c) / freqPerBin); hi = round((binFreq * c) / freqPerBin)
static __global__ void k_avg_windows(int* lo, int* hi, int M, double freq_per_bin, double c_side) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    const double f = (double) k * freq_per_bin;
    lo[k] = (int) round((f / c_side) / freq_per_bin);
    hi[k] = (int) round((f * c_side) / freq_per_bin);
}
// (1) per bin k <= M: la[k] = log(clamp(|S[k]|)) (or the plain amplitude for the linear average)
__device__ __forceinline__ float avg_log_ampl(float2 v, int log_avg) {
    const float ampl = (float) sqrt((double) v.x * (double) v.x + (double) v.y * (double) v.y);     // tools::binAmpl
    return log_avg ? logf(round_1e16(ampl)) : ampl;
}
static __global__ void k_avg_prepare(const float2* S, long long s_stride, float* la, long long la_stride, int M, int log_avg) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    la[blockIdx.y * la_stride + k] = avg_log_ampl(S[blockIdx.y * s_stride + k], log_avg);
}
// (2) The running window sum of the log average is a FIXED sequence of float additions (fp/convolution.cpp:482-505): for
// bin k = 0, 1, ...: subtract la[b] for b in [lo[k-1], lo[k]), then add la[b] for b in (hi[k-1], hi[k]] (bins past
// Nyquist, M < b < 2M, hold amplitude 0 -> clamp -> log(1e-16); b >= 2M is skipped, "addBin < fftSize"), then record.
// The sequence depends on the windows only, so it is laid out ONCE per call as a list of signed bin codes:
//   ops[j] = b (add la[b]) or ~b (subtract la[b]);  endq[k] = index of the last operation before bin k is recorded.
static __global__ void k_avg_oplist(const int* lo, const int* hi, int* ops, int* endq, int M) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    const int l0 = k ? lo[k - 1] : 0, l1 = lo[k], h0 = k ? hi[k - 1] : -1, h1 = hi[k];
    int j = l0 + h0 + 1;
    for (int b = l0; b < l1; ++b) ops[j++] = ~b;
    for (int b = h0 + 1; b <= h1; ++b) ops[j++] = b;
    endq[k] = l1 + h1;
}
// first bin recorded in each chunk of kAvgChunk operations (kstart[nchunks] = M + 1)
constexpr int kAvgChunk = 2048;
static __global__ void k_avg_chunk_starts(const int* endq, int* kstart, int M, int nchunks) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    const int c1 = endq[k] / kAvgChunk, c0 = k ? endq[k - 1] / kAvgChunk : -1;
    for (int c = c0 + 1; c <= c1; ++c) kstart[c] = k;
    if (k == M) for (int c = c1 + 1; c <= nchunks; ++c) kstart[c] = M + 1;
}
// One CTA per spectrum: lane 0 of warp 0 carries the dependent add chain, nothing else (4 cycles per operation);
// warps 1..4 gather the operands of the next chunk into shared memory and write the previous chunk's sums back.
// The gather is branch-free and issues all of a thread's loads of one kind back to back (codes, then operands), so a
// chunk costs the producers two memory latencies, well under the chain's 2048 x 4 cycles.
constexpr int kAvgProducers = 128;
static __global__ void __launch_bounds__(32 + kAvgProducers) k_avg_scan(const float* la, long long la_stride, const int* __restrict__ ops,
                                                                 const int* __restrict__ endq, const int* __restrict__ kstart, int nchunks, int n_ops,
                                                                 float* rs, long long rs_stride, int M) {
    __shared__ __align__(16) float s_val[2][kAvgChunk], s_sum[2][kAvgChunk];
    const float* a = la + blockIdx.x * la_stride;
    float* out = rs + blockIdx.x * rs_stride;
    const int tid = threadIdx.x, ptid = tid - 32;
    const float log_floor = logf(1e-16f);
    constexpr int PER = kAvgChunk / kAvgProducers;
    auto fill = [&](int c) {
        float* dst = s_val[c & 1];
        const int j0 = c * kAvgChunk;
        int code[PER];
        float val[PER];
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int g = j0 + ptid + i * kAvgProducers;
            code[i] = __ldg(ops + (g < n_ops ? g : n_ops - 1));
        }
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int b = code[i] < 0 ? ~code[i] : code[i];
            val[i] = a[b <= M ? b : 0];
        }
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int g = j0 + ptid + i * kAvgProducers;
            const int b = code[i] < 0 ? ~code[i] : code[i];
            float v = b <= M ? val[i] : (b < 2 * M ? log_floor : 0.0f);
            v = code[i] < 0 ? -v : v;
            dst[ptid + i * kAvgProducers] = g < n_ops ? v : 0.0f;
        }
    };
    auto write_back = [&](int c) {
        const float* src = s_sum[c & 1];
        const int j0 = c * kAvgChunk, k0 = kstart[c], k1 = kstart[c + 1];
        for (int kb = k0; kb < k1; kb += 4 * kAvgProducers) {
            int e[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { const int k = kb + ptid + i * kAvgProducers; e[i] = __ldg(endq + (k < k1 ? k : k0)); }
#pragma unroll
            for (int i = 0; i < 4; ++i) { const int k = kb + ptid + i * kAvgProducers; if (k < k1) out[k] = src[e[i] - j0]; }
        }
    };
    if (tid >= 32) fill(0);
    __syncthreads();
    float running = 0.0f;
    for (int c = 0; c < nchunks; ++c) {
        if (tid == 0) {
            // operands are fetched 32 operations ahead so that the chain never waits for shared memory
            const float4* v4 = reinterpret_cast<const float4*>(s_val[c & 1]);
            float4* p4 = reinterpret_cast<float4*>(s_sum[c & 1]);
            constexpr int D = 8;
            float4 cur[D], nxt[D];
#pragma unroll
            for (int i = 0; i < D; ++i) cur[i] = v4[i];
#pragma unroll 1
            for (int j = 0; j < kAvgChunk / 4; j += D) {
                if (j + D < kAvgChunk / 4) {
#pragma unroll
                    for (int i = 0; i < D; ++i) nxt[i] = v4[j + D + i];
                }
#pragma unroll
                for (int i = 0; i < D; ++i) {
                    float4 p;
                    running += cur[i].x; p.x = running;
                    running += cur[i].y; p.y = running;
                    running += cur[i].z; p.z = running;
                    running += cur[i].w; p.w = running;
                    p4[j + i] = p;
                }
#pragma unroll
                for (int i = 0; i < D; ++i) cur[i] = nxt[i];
            }
        } else if (tid >= 32) {
            if (c + 1 < nchunks) fill(c + 1);
            if (c >= 1) write_back(c - 1);
        }
        __syncthreads();
    }
    if (tid >= 32) write_back(nchunks - 1);
}
// linear average: a fresh ascending sum per bin (fp/convolution.cpp:508-514) -- no sequential dependence
static __global__ void k_avg_linear_sum(const float* la, long long la_stride, const int* lo, const int* hi, float* rs, long long rs_stride, int M) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    const float* a = la + blockIdx.y * la_stride;
    float sum = 0.0f;
    for (int b = lo[k]; b <= hi[k]; ++b) sum += (b <= M ? a[b] : 0.0f);
    rs[blockIdx.y * rs_stride + k] = sum;
}
// (3) new amplitude = exp(sum / window length), bins rebuilt from it and the original phase (fp/convolution.cpp:518-543)
// returns the rebuilt bin; shared by the per-pass kernel and the fused three-pass kernel so both execute the same arithmetic
__device__ __forceinline__ float2 avg_rebuild_bin(float2 v, float sum, int lo_k, int hi_k, int log_avg, int include_phase, int include_ampl) {
    // the reference divides in double and rounds to float: (float) ((double) sum / len).  With both operands exactly representable in
    // float (the window length is an integer below 2^24) that is the correctly rounded float quotient -- double carries more than
    // 2 x 24 + 2 bits, so the second rounding cannot change the result -- i.e. IEEE float division, which is what `/` compiles to here.
    float ampl = sum / (float) (hi_k - lo_k + 1);
    if (log_avg) ampl = expf(ampl);
    ampl = round_1e16(ampl);
    const float re = round_to_zero(v.x, 1e-11f), im = round_to_zero(v.y, 1e-11f);
    float phase = atan2f(im, re);
    if (!include_ampl) ampl = 1.0f;
    if (!include_phase) phase = 0.0f;
    float sn, cs;
    sincosf(phase, &sn, &cs);                                            // one argument reduction for both; same values as sinf / cosf
    return make_float2(ampl * cs, ampl * sn);
}
// next_la != nullptr: also the log amplitudes of the rebuilt bins, i.e. the next pass's step (1)
static __global__ void k_avg_apply(float2* S, long long s_stride, const float* rs, long long rs_stride, const int* lo, const int* hi, int M, int log_avg,
                            int include_phase, int include_ampl, float* next_la, long long la_stride) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M) return;
    float2* s = S + blockIdx.y * s_stride;
    const float2 nv = avg_rebuild_bin(s[k], rs[blockIdx.y * rs_stride + k], lo[k], hi[k], log_avg, include_phase, include_ampl);
    s[k] = nv;
    if (next_la) next_la[blockIdx.y * la_stride + k] = avg_log_ampl(nv, log_avg);
}

// All passes of the log average in ONE launch.  Pass p + 1 needs the rebuilt bins of pass p only up to the upper window edge
// hi[k] ~ 1.027 k of the bin it is working on, so the passes run as a wavefront inside one CTA per spectrum: each pass has its own
// chain warp (lane 0 carries the dependent FADD sequence, as in k_avg_scan) and its own 128 producer threads, which gather the
// operands of the pass's next chunk, rebuild the bins the previous chunk recorded (step 3) and publish, in shared memory, how far
// the pass has got; the next pass's producers wait on that mark before they gather.  Three passes cost one pass plus 3 % instead
// of three chain traversals and six elementwise kernels.  Same additions in the same order, same per-bin arithmetic.
constexpr int kAvgMaxPasses = 3;
constexpr int kAvgPassThreads = 32 + kAvgProducers;
constexpr int kAvgPassSmemBytes = 4 * kAvgChunk * (int) sizeof(float);
__device__ __forceinline__ void avg_bar(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
static __global__ void __launch_bounds__(kAvgMaxPasses * kAvgPassThreads, 2)
k_avg_passes(float2* S, long long s_stride, float* la, long long la_stride, long long la_pass_stride, const int* __restrict__ ops, const int* __restrict__ endq,
             const int* __restrict__ kstart, const int* __restrict__ lo, const int* __restrict__ hi, int nchunks, int n_ops, int M, int passes, int include_phase,
             int include_ampl) {
    extern __shared__ __align__(16) unsigned char avg_raw[];
    __shared__ volatile int applied[kAvgMaxPasses];                        // bins [0, applied[p]) of pass p are rebuilt and visible
    if (threadIdx.x < kAvgMaxPasses) applied[threadIdx.x] = 0;
    __syncthreads();
    const int pass = threadIdx.x / kAvgPassThreads, tid = threadIdx.x % kAvgPassThreads, ptid = tid - 32;
    if (pass >= passes) return;
    float* mine = reinterpret_cast<float*>(avg_raw) + (size_t) pass * 4 * kAvgChunk;
    auto s_val = [&](int c) { return mine + (c & 1) * kAvgChunk; };
    auto s_sum = [&](int c) { return mine + (2 + (c & 1)) * kAvgChunk; };
    const float* a = la + pass * la_pass_stride + blockIdx.x * la_stride;
    float* a_next = pass + 1 < passes ? la + (pass + 1) * la_pass_stride + blockIdx.x * la_stride : nullptr;
    float2* s = S + blockIdx.x * s_stride;
    const float log_floor = logf(1e-16f);
    constexpr int PER = kAvgChunk / kAvgProducers;
    auto wait_for_previous_pass = [&](int c) {                             // every bin the operations of chunk c add is rebuilt
        if (pass == 0) return;
        int kn = __ldg(kstart + c + 1);
        kn = kn < M ? kn : M;
        int need = __ldg(hi + kn);
        need = need < M ? need : M;
        while (applied[pass - 1] <= need) __nanosleep(64);
        __threadfence_block();
    };
    auto fill = [&](int c) {
        float* dst = s_val(c);
        const int j0 = c * kAvgChunk;
        int code[PER];
        float val[PER];
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int g = j0 + ptid + i * kAvgProducers;
            code[i] = __ldg(ops + (g < n_ops ? g : n_ops - 1));
        }
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int b = code[i] < 0 ? ~code[i] : code[i];
            val[i] = a[b <= M ? b : 0];
        }
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int g = j0 + ptid + i * kAvgProducers;
            const int b = code[i] < 0 ? ~code[i] : code[i];
            float v = b <= M ? val[i] : (b < 2 * M ? log_floor : 0.0f);
            v = code[i] < 0 ? -v : v;
            dst[ptid + i * kAvgProducers] = g < n_ops ? v : 0.0f;
        }
    };
    auto rebuild = [&](int c) {                                            // step (3) for the bins chunk c recorded
        const float* src = s_sum(c);
        const int j0 = c * kAvgChunk, k0 = __ldg(kstart + c), k1 = __ldg(kstart + c + 1);
        for (int kb = k0; kb < k1; kb += 4 * kAvgProducers) {
            int e[4], l[4], h[4];
            float2 v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int k = kb + ptid + i * kAvgProducers, kk = k < k1 ? k : k0;
                e[i] = __ldg(endq + kk); l[i] = __ldg(lo + kk); h[i] = __ldg(hi + kk);
                v[i] = s[kk];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int k = kb + ptid + i * kAvgProducers;
                if (k < k1) {
                    const float2 nv = avg_rebuild_bin(v[i], src[e[i] - j0], l[i], h[i], 1, include_phase, include_ampl);
                    s[k] = nv;
                    if (a_next) a_next[k] = avg_log_ampl(nv, 1);
                }
            }
        }
        __threadfence_block();
        avg_bar(1 + kAvgMaxPasses + pass, kAvgProducers);                  // the pass's producers only
        if (ptid == 0) applied[pass] = k1;
    };
    if (tid >= 32) { wait_for_previous_pass(0); fill(0); }
    avg_bar(1 + pass, kAvgPassThreads);
    float running = 0.0f;
    for (int c = 0; c < nchunks; ++c) {
        if (tid == 0) {
            // operands are fetched 16 operations ahead so that the chain never waits for shared memory
            const float4* v4 = reinterpret_cast<const float4*>(s_val(c));
            float4* p4 = reinterpret_cast<float4*>(s_sum(c));
            constexpr int D = 4;
            float4 cur[D], nxt[D];
#pragma unroll
            for (int i = 0; i < D; ++i) cur[i] = v4[i];
#pragma unroll 1
            for (int j = 0; j < kAvgChunk / 4; j += D) {
                if (j + D < kAvgChunk / 4) {
#pragma unroll
                    for (int i = 0; i < D; ++i) nxt[i] = v4[j + D + i];
                }
#pragma unroll
                for (int i = 0; i < D; ++i) {
                    float4 p;
                    running += cur[i].x; p.x = running;
                    running += cur[i].y; p.y = running;
                    running += cur[i].z; p.z = running;
                    running += cur[i].w; p.w = running;
                    p4[j + i] = p;
                }
#pragma unroll
                for (int i = 0; i < D; ++i) cur[i] = nxt[i];
            }
        } else if (tid >= 32) {
            if (c >= 1) rebuild(c - 1);
            if (c + 1 < nchunks) { wait_for_previous_pass(c + 1); fill(c + 1); }
        }
        avg_bar(1 + pass, kAvgPassThreads);
    }
    if (tid >= 32) rebuild(nchunks - 1);
}

// out[i] = in[(i + h1) mod n] : ir::shifteroo (fp/ir.cpp:85-103), h1 = ceil(n/2)
static __global__ void k_shifteroo(const float* in, float* out, int n, long long stride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int h2 = n / 2, h1 = n - h2;
    out[blockIdx.y * stride + i] = in[blockIdx.y * stride + (i < h2 ? i + h1 : i - h2)];
}

// fp::ExpSineSweep::generate / generateInv (fp/ExpSineSweep.cpp:26-41,59-79), FP64:
// sweep[i] = g sin(K (exp(i / L) - 1)); inverse = reversed sweep times k^(i+1)
static __global__ void k_ess(double* out, int n, double g, double K, double L, int inverse, double kdecay) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = inverse ? n - 1 - i : i;
    double v = g * sin(K * (exp((double) j / L) - 1.0));
    if (inverse) v *= pow(kdecay, (double) (i + 1));
    out[i] = v;
}

}  // namespace irb
