// irb_spectral.cu -- host side of the single-large-FFT entry points of include/irb_b200.h:
// irb_convolve_nonperiodic, irb_convolve_batch(_device), irb_deconvolve(_batch), irb_averaging_filter, irb_fft_transform,
// irb_fft_inv_transform, irb_invert_filter, irb_ess_generate, irb_ir_chop_batch_device, irb_deconvolve_chop_batch.  Every
// arithmetic step is a kernel of irb_spectral.cuh or irb_chop.cuh; the host only sizes buffers, copies and launches.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "irb_chop.cuh"
#include "irb_common.hpp"
#include "irb_spectral.cuh"
#include "irb_tuning.hpp"

namespace {

using DevBuf = irbh::ScratchBuf;      // every buffer in this file is call-scoped scratch: recycled through the pool
using irbh::fail;
using irbh::g_launches;

constexpr int kMinM = 8;                 // smallest half size the Stockham passes take (N = 16)
constexpr int kMaxBigM = 1 << 21;        // N up to 2^22 (87 s at 48 kHz)
constexpr int kMaxGridY = 65535;         // largest grid.y of a launch: batch items per launch

// Real-output window of an inverse transform's last pass (irb::LineWindow): floats [off, off + len) of each batch item's real
// result go to out + b * stride - off; len < 0: the whole complex result is stored as float2 (irb::k_line_fft)
struct OutWindow {
    long long off = 0, stride = 0;
    int len = -1;
};

template <int L, bool INV, bool WIN = false>
int launch_line_t(const irb::LineArgs& a, const OutWindow& w, int batch, cudaStream_t st) {
    using T = irb::LineTile<L>;
    static thread_local int configured_dev = -1;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    if (configured_dev != dev) {
        if constexpr (WIN) CK(cudaFuncSetAttribute(irb::k_line_fft_win<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) T::SMEM));
        else CK(cudaFuncSetAttribute(irb::k_line_fft<L, INV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) T::SMEM));
        configured_dev = dev;
    }
    dim3 grid((a.n_lines + T::C - 1) / T::C, batch);
    if constexpr (WIN) irb::k_line_fft_win<L><<<grid, irb::kThreads, T::SMEM, st>>>(a, irb::LineWindow{w.off, w.stride, w.len});
    else irb::k_line_fft<L, INV><<<grid, irb::kThreads, T::SMEM, st>>>(a);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
int launch_line(int L, bool inv, const irb::LineArgs& a, int batch, cudaStream_t st, const OutWindow& w = {}) {
    if (w.len >= 0 && !inv) return fail(IRB_ERR_ARG, "an output window needs an inverse transform");
#define IRB_LINE_CASE(LL) case LL: return w.len >= 0 ? launch_line_t<LL, true, true>(a, w, batch, st) : inv ? launch_line_t<LL, true>(a, w, batch, st) : launch_line_t<LL, false>(a, w, batch, st);
    switch (L) {
        IRB_LINE_CASE(8) IRB_LINE_CASE(16) IRB_LINE_CASE(32) IRB_LINE_CASE(64) IRB_LINE_CASE(128) IRB_LINE_CASE(256)
        IRB_LINE_CASE(512) IRB_LINE_CASE(1024) IRB_LINE_CASE(2048)
        default: return fail(IRB_ERR_ARG, "unsupported FFT line length %d", L);
    }
#undef IRB_LINE_CASE
}

template <int L>
int launch_pair_t(const irb::PairArgs& a, int batch, cudaStream_t st) {
    using T = irb::PairTile<L>;
    static thread_local int configured_dev = -1;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    if (configured_dev != dev) {
        CK(cudaFuncSetAttribute(irb::k_rowpair<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) T::SMEM));
        configured_dev = dev;
    }
    dim3 grid((a.M1 / 2 + 1 + T::NP - 1) / T::NP, batch);
    irb::k_rowpair<L><<<grid, irb::kThreads, T::SMEM, st>>>(a);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
int launch_pair(int L, const irb::PairArgs& a, int batch, cudaStream_t st) {
#define IRB_PAIR_CASE(LL) case LL: return launch_pair_t<LL>(a, batch, st);
    switch (L) {
        IRB_PAIR_CASE(64) IRB_PAIR_CASE(128) IRB_PAIR_CASE(256) IRB_PAIR_CASE(512) IRB_PAIR_CASE(1024)
        default: return fail(IRB_ERR_ARG, "unsupported row length %d", L);
    }
#undef IRB_PAIR_CASE
}

// M-point complex FFT plan: one pass for M <= 2048, else M = M1 * M2 (both in [64, 1024])
struct Plan {
    int M = 0, M1 = 1, M2 = 0;
    const float2 *W1 = nullptr, *W2 = nullptr, *WN = nullptr;   // WN: table of the N = 2M roots when M <= 2048, else null (computed in double)
    const float2 *Thi = nullptr, *Tlo = nullptr;                // two-level table of the M-th roots (inter-pass twiddles)
    const float2 *Nhi = nullptr, *Nlo = nullptr;                // two-level table of the 2M-th roots (split / merge of the big transforms)
    bool big() const { return M1 > 1; }
    int init(int dev, int M_) {
        M = M_;
        if (M < kMinM || M > kMaxBigM || (M & (M - 1))) return fail(IRB_ERR_ARG, "FFT half size %d outside [%d, %d] or not a power of two", M, kMinM, kMaxBigM);
        int rc;
        if (M <= 2048) {
            M1 = 1; M2 = M;
            if ((rc = irbh::twiddles(dev, M, &W2))) return rc;
            WN = W2;                                             // the same table: 2M roots
        } else {
            int lg = 0;
            while ((1 << lg) < M) ++lg;
            M1 = 1 << (lg / 2);
            M2 = M / M1;
            if (M2 > 1024) { M2 = 1024; M1 = M / M2; }           // rows stay within the row-pair kernel's range; columns take up to 2048
            if ((rc = irbh::twiddles(dev, M1, &W1)) || (rc = irbh::twiddles(dev, M2, &W2)) || (rc = irbh::twiddles2(dev, M, &Thi, &Tlo)) ||
                (rc = irbh::twiddles2(dev, 2 * M, &Nhi, &Nlo)))
                return rc;
        }
        return 0;
    }
    // batch items at in + b*in_stride -> out + b*out_stride (float2 units); real_len >= 0: `in` is real data.
    // tmp: M complex per batch item (two-pass only; may alias neither in nor out).  win: real-output window of the result.
    int run(const void* in, long long in_stride, int real_len, float2* out, long long out_stride, float2* tmp, int batch, bool inv, float scale,
            cudaStream_t st, const OutWindow& win = {}) const {
        irb::LineArgs a{};
        if (M1 == 1) {                                           // batch items are the lines
            a.in = in; a.out = out; a.in_elem_stride = 1; a.in_line_stride = in_stride; a.in_batch_stride = 0;
            a.out_elem_stride = 1; a.out_line_stride = out_stride; a.out_batch_stride = 0;
            a.n_lines = batch; a.in_real_len = real_len; a.tw_M = 0; a.scale = scale; a.W = W2;
            if ((real_len >= 0 || win.len >= 0) && batch > 1) {
                // the real-input bounds check and the output window are per batch item: run items one grid.y slice each
                a.in_line_stride = 0; a.in_batch_stride = in_stride; a.out_line_stride = 0; a.out_batch_stride = out_stride; a.n_lines = 1;
                return launch_line(M2, inv, a, batch, st, win);
            }
            return launch_line(M2, inv, a, 1, st, win);
        }
        // pass 1: M2 column transforms of length M1 (element n1 of line n2 at n1*M2 + n2), twiddle exp(-+2 pi i n2 k1 / M)
        a.in = in; a.out = tmp; a.in_elem_stride = M2; a.in_line_stride = 1; a.in_batch_stride = in_stride;
        a.out_elem_stride = M2; a.out_line_stride = 1; a.out_batch_stride = M;
        a.n_lines = M2; a.in_real_len = real_len; a.tw_M = M; a.tw_hi = Thi; a.tw_lo = Tlo; a.scale = 1.0f; a.W = W1;
        int rc = launch_line(M1, inv, a, batch, st);
        if (rc) return rc;
        // pass 2: M1 row transforms of length M2 (line k1 at k1*M2), bin k1 + M1*k2 written in natural order
        a.in = tmp; a.out = out; a.in_elem_stride = 1; a.in_line_stride = M2; a.in_batch_stride = M;
        a.out_elem_stride = M1; a.out_line_stride = 1; a.out_batch_stride = out_stride;
        a.n_lines = M1; a.in_real_len = -1; a.tw_M = 0; a.scale = scale; a.W = W2;
        return launch_line(M2, inv, a, batch, st, win);
    }
    // ---- the fused pipeline of the big transforms (M1 > 1); rows = [batch][M1][M2] ------------------------------
    // column pass of the forward transform: signal (real when real_len >= 0) -> rows, inter-pass twiddle applied
    int cols_fwd(const void* in, long long in_stride, int real_len, float2* rows, int batch, cudaStream_t st) const {
        irb::LineArgs a{};
        a.in = in; a.out = rows; a.in_elem_stride = M2; a.in_line_stride = 1; a.in_batch_stride = in_stride;
        a.out_elem_stride = M2; a.out_line_stride = 1; a.out_batch_stride = M;
        a.n_lines = M2; a.in_real_len = real_len; a.tw_M = M; a.tw_hi = Thi; a.tw_lo = Tlo; a.scale = 1.0f; a.W = W1;
        return launch_line(M1, false, a, batch, st);
    }
    // row transforms in place (row k1 then holds the bins k1 + M1*k2), then the split spectrum of a real signal in row layout
    // (reciprocal: 1/B, for a division carried out as a multiplication)
    int rows_to_split_spectrum(float2* rows, float2* brows, int batch, bool reciprocal, cudaStream_t st) const {
        irb::LineArgs a{};
        a.in = rows; a.out = rows; a.in_elem_stride = 1; a.in_line_stride = M2; a.in_batch_stride = M;
        a.out_elem_stride = 1; a.out_line_stride = M2; a.out_batch_stride = M;
        a.n_lines = M1; a.in_real_len = -1; a.tw_M = 0; a.scale = 1.0f; a.W = W2;
        int rc = launch_line(M2, false, a, batch, st);
        if (rc) return rc;
        irb::k_split_rows<<<dim3((unsigned) ((M + 255) / 256), (unsigned) batch), 256, 0, st>>>(rows, brows, M1, M2, Nhi, Nlo, reciprocal ? 1 : 0);
        g_launches++;
        CK(cudaGetLastError());
        return 0;
    }
    // rows of `batch` signals: forward row FFT, per-bin multiply by brows, inverse row FFT + twiddle, in place
    int rows_binop(float2* rows, const float2* brows, long long b_stride, int batch, cudaStream_t st) const {
        irb::PairArgs a{};
        a.Z = rows; a.z_batch_stride = M; a.Brows = brows; a.b_batch_stride = b_stride; a.M1 = M1; a.W = W2;
        a.Nhi = Nhi; a.Nlo = Nlo; a.Mhi = Thi; a.Mlo = Tlo;
        return launch_pair(M2, a, batch, st);
    }
    // column pass of the inverse transform: rows -> out (natural order), scaled; win: real-output window
    int cols_inv(const float2* rows, float2* out, long long out_stride, int batch, float scale, cudaStream_t st, const OutWindow& win = {}) const {
        irb::LineArgs a{};
        a.in = rows; a.out = out; a.in_elem_stride = M2; a.in_line_stride = 1; a.in_batch_stride = M;
        a.out_elem_stride = M2; a.out_line_stride = 1; a.out_batch_stride = out_stride;
        a.n_lines = M2; a.in_real_len = -1; a.tw_M = 0; a.scale = scale; a.W = W1;
        return launch_line(M1, true, a, batch, st, win);
    }
};

inline dim3 grid1(long long n, int batch) { return dim3((unsigned) ((n + 255) / 256), (unsigned) batch); }
#define LAUNCHED() do { g_launches++; CK(cudaGetLastError()); } while (0)

// fp::convolution::averagingFilter state shared by every spectrum and pass of a call: windows, the operation list of
// the running sum and its chunking (irb_spectral.cuh), plus per-spectrum scratch
struct Smoother {
    DevBuf la, rs, lo, hi, ops, endq, kstart;
    int M = 0, n_ops = 0, nchunks = 0, la_n = 0;
    bool fused = false;
    int init(int M_, int batch, double octave_fraction, double sample_rate, int log_avg, cudaStream_t st) {
        M = M_;
        const double fract_per_side = octave_fraction / 2.0;
        const double nyquist = sample_rate / 2;
        const double freq_per_bin = nyquist / (double) M;                  // fp/convolution.cpp:425 (N/2 complex bins up to Nyquist)
        const double c_side = pow(2.0, fract_per_side);
        if (!(octave_fraction >= 0.0) || !(freq_per_bin > 0.0) || c_side * (double) M > 1.0e9) return fail(IRB_ERR_ARG, "averagingFilter: octave fraction %g / sample rate %g out of range", octave_fraction, sample_rate);
        int rc;
        // la: the log amplitudes every pass starts from (the fused kernel keeps one array per pass); rs: the recorded sums of the per-pass kernels
        fused = log_avg && irbh::g_tuning.avg_fused;
        la_n = batch;
        if ((rc = la.alloc(sizeof(float) * (size_t) (M + 1) * batch * (fused ? irb::kAvgMaxPasses : 1), false)) ||
            (!fused && (rc = rs.alloc(sizeof(float) * (size_t) (M + 1) * batch, false))) ||
            (rc = lo.alloc(sizeof(int) * (size_t) (M + 1), false)) || (rc = hi.alloc(sizeof(int) * (size_t) (M + 1), false)))
            return rc;
        irb::k_avg_windows<<<grid1(M + 1, 1), 256, 0, st>>>(lo.as<int>(), hi.as<int>(), M, freq_per_bin, c_side);
        LAUNCHED();
        if (log_avg) {
            // the same double operations as k_avg_windows for k = M give the length of the operation list
            const double f = (double) M * freq_per_bin;
            const long long T = (long long) round((f / c_side) / freq_per_bin) + (long long) round((f * c_side) / freq_per_bin) + 1;
            n_ops = (int) T;
            nchunks = (n_ops + irb::kAvgChunk - 1) / irb::kAvgChunk;
            if ((rc = ops.alloc(sizeof(int) * (size_t) n_ops, false)) || (rc = endq.alloc(sizeof(int) * (size_t) (M + 1), false)) ||
                (rc = kstart.alloc(sizeof(int) * (size_t) (nchunks + 1), false)))
                return rc;
            irb::k_avg_oplist<<<grid1(M + 1, 1), 256, 0, st>>>(lo.as<int>(), hi.as<int>(), ops.as<int>(), endq.as<int>(), M);
            LAUNCHED();
            irb::k_avg_chunk_starts<<<grid1(M + 1, 1), 256, 0, st>>>(endq.as<int>(), kstart.as<int>(), M, nchunks);
            LAUNCHED();
        }
        return 0;
    }
    // `passes` smoothing passes on interleaved spectra S[batch][>= M+1] (fp/convolution.cpp:389-394 runs three)
    int run(float2* S, long long s_stride, int batch, int passes, int log_avg, int include_phase, int include_ampl, cudaStream_t st) {
        const long long stride = M + 1;
        irb::k_avg_prepare<<<grid1(M + 1, batch), 256, 0, st>>>(S, s_stride, la.as<float>(), stride, M, log_avg);
        LAUNCHED();
        if (log_avg && fused && passes >= 1 && passes <= irb::kAvgMaxPasses && batch <= la_n) {
            const int smem = passes * irb::kAvgPassSmemBytes;
            CK(cudaFuncSetAttribute(irb::k_avg_passes, cudaFuncAttributeMaxDynamicSharedMemorySize, irb::kAvgMaxPasses * irb::kAvgPassSmemBytes));
            irb::k_avg_passes<<<batch, passes * irb::kAvgPassThreads, smem, st>>>(S, s_stride, la.as<float>(), stride, stride * la_n, ops.as<int>(), endq.as<int>(), kstart.as<int>(),
                                                                                 lo.as<int>(), hi.as<int>(), nchunks, n_ops, M, passes, include_phase, include_ampl);
            LAUNCHED();
            return 0;
        }
        if (fused) return fail(IRB_ERR_ARG, "averagingFilter: %d passes over %d spectra do not fit the plan made for %d", passes, batch, la_n);
        for (int i = 0; i < passes; ++i) {
            if (log_avg) irb::k_avg_scan<<<batch, 32 + irb::kAvgProducers, 0, st>>>(la.as<float>(), stride, ops.as<int>(), endq.as<int>(), kstart.as<int>(), nchunks, n_ops, rs.as<float>(), stride, M);
            else irb::k_avg_linear_sum<<<grid1(M + 1, batch), 256, 0, st>>>(la.as<float>(), stride, lo.as<int>(), hi.as<int>(), rs.as<float>(), stride, M);
            LAUNCHED();
            irb::k_avg_apply<<<grid1(M + 1, batch), 256, 0, st>>>(S, s_stride, rs.as<float>(), stride, lo.as<int>(), hi.as<int>(), M, log_avg, include_phase, include_ampl,
                                                                  i + 1 < passes ? la.as<float>() : nullptr, stride);
            LAUNCHED();
        }
        return 0;
    }
};

int fft_size_for(int len, int* N) {
    int n = irbh::next_pow2(len);
    if (n < 2 * kMinM) return fail(IRB_ERR_ARG, "length %d gives an FFT of %d points; the device transforms start at %d", len, n, 2 * kMinM);
    if (n > 2 * kMaxBigM) return fail(IRB_ERR_ARG, "length %d needs an FFT above 2^22 points", len);
    *N = n;
    return 0;
}

// fp::ir::IRchop (+ fp::tools::normalize) of rows of a batch (irb_chop.cuh); positions: [rows][2] device memory, or null
struct ChopSpec {
    int ir_length;
    float threshold_db;
    int consecutive, normalize;
    float goal_lin;               // tools::dBToLin(goal_db), computed here on the host as the facade does
    int* positions;               // the caller's [batch][2], or null
};

// every argument error of the chop, before any CUDA call; len: the samples of each row the chop reads
int chop_spec(int len, int ir_length, float threshold_db, int consecutive, int normalize, float goal_db, int* positions, ChopSpec* c) {
    if (ir_length < 1 || ir_length > len) return fail(IRB_ERR_ARG, "ir_length %d outside [1, %d]: the IR is cut from rows of %d samples", ir_length, len, len);
    *c = ChopSpec{ir_length, threshold_db, consecutive, normalize != 0, std::pow(10.0f, goal_db / 20.0f), positions};
    return 0;
}

// chunks per row of the peak pass: about 8 CTAs per SM over the batch, at least 8192 samples per chunk
int chop_chunks(int rows, long long len, long long* chunk_len) {
    constexpr long long kTargetCtas = 148 * 8, kMinChunk = 8192;
    long long chunks = std::max(1LL, std::min((kTargetCtas + rows - 1) / rows, (len + kMinChunk - 1) / kMinChunk));
    *chunk_len = ((len + chunks - 1) / chunks + 3) & ~3LL;
    return (int) ((len + *chunk_len - 1) / *chunk_len);
}

// bytes of the peak pass's partial results for rows x chunks
size_t chop_part_bytes(int rows, int chunks) { return (sizeof(long long) + sizeof(float)) * (size_t) rows * chunks; }

// rows of x[rows][len] (device) -> out[rows][c.ir_length] and pos[rows][2] (device, or null); chunks / chunk_len from chop_chunks,
// part: chop_part_bytes(rows, chunks)
int launch_chop(const float* x, int rows, long long len, int chunks, long long chunk_len, const ChopSpec& c, float* out, int* pos, void* part, cudaStream_t st) {
    long long* part_i = static_cast<long long*>(part);
    float* part_m = reinterpret_cast<float*>(part_i + (size_t) rows * chunks);
    const bool vec = (uintptr_t) x % 16 == 0 && len % 4 == 0;
    if (vec) irb::k_chop_peak<true><<<(unsigned) ((long long) rows * chunks), irb::kChopPeakThreads, 0, st>>>(x, len, chunks, chunk_len, part_m, part_i);
    else irb::k_chop_peak<false><<<(unsigned) ((long long) rows * chunks), irb::kChopPeakThreads, 0, st>>>(x, len, chunks, chunk_len, part_m, part_i);
    g_launches++;
    CK(cudaGetLastError());
    irb::ChopArgs a{x, len, chunks, part_m, part_i, c.ir_length, c.consecutive, c.normalize, c.threshold_db, c.goal_lin, out, pos};
    irb::k_chop_cut<<<(unsigned) rows, irb::kChopCutThreads, 0, st>>>(a);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}

}  // namespace

// One batched spectral product, the core of the batched division and of the (batched) linear convolution:
//   y_b = IFFT_N(FFT_N(x_b) op FFT_N(h_b)),  h_b = h[0] (h_batch == 1, one operand shared by every item) or h[b] (h_batch == batch),
// both signals zero-padded to N; op is the per-bin product, or the division tools::complexDivCartesian carried out as a product with
// the reciprocal spectrum.  win.len < 0: each row of out is the whole N-point result; else the rows hold win.len floats, the
// window [win.off, win.off + win.len) of each result (win.stride == win.len).
struct BatchJob {
    const float* x; int batch, len_x;
    const float* h; int h_batch, len_h;          // host or device memory
    int N;
    bool divide;
    OutWindow win;
    float* out;
    const ChopSpec* chop = nullptr;              // division only: out[batch][ir_length] holds each row cut by the chop
    long long out_row() const { return win.len >= 0 ? win.len : N; }
};

// The batch runs in sub-batches through a three-stage pipeline (upload i+1 | kernels i | download i-1) over
// double-buffered device memory; a sub-batch is small enough for its intermediate spectra to stay in the L2.
// Per-item operands are uploaded and transformed with their sub-batch.  The smoothing path (division only: a shared
// denominator, no window) is fp::convolution::deconvolve's averagingFilter between the division and the inverse transform.
// device_io: inputs and results lie in device memory, so the smoothed path reports irb_last_compute_ms() as the device span from its
// first to its last kernel (groups overlap); from host buffers it is the sum of the kernel sections' spans, copies excluded.
static int batch_staged(const BatchJob& J, double sample_rate, int smoothing, int include_phase, int include_amplitude, bool device_io) {
    const float* nums = J.x;
    const int batch = J.batch, len_num = J.len_x, len_den = J.len_h, N = J.N, M = N / 2, dev = irbh::current_device();
    const bool per_item = J.h_batch > 1;
    const long long out_row = J.out_row();
    int rc;
    CK(cudaSetDevice(dev));
    Plan plan;
    if ((rc = plan.init(dev, M))) return rc;
    struct Slot { DevBuf dn, Zn, dy, dy2, tmp, dh, Zh, Bh, dc, dpos, dpart; cudaEvent_t ev_in = nullptr, ev_done = nullptr, ev_out = nullptr, t0 = nullptr, t1 = nullptr;
                  bool dn_busy = false, dy_busy = false, timed = false;
                  ~Slot() { for (cudaEvent_t e : {ev_in, ev_done, ev_out, t0, t1}) if (e) cudaEventDestroy(e); } } slot[4];   // [2], [3]: the smoothing path's last phase
    // smoothing runs in up to kLanes groups of captures at once, each on its own compute stream with its own spectrum array and
    // smoother, so that one group's transforms and copies run under another group's running sums
    constexpr int kLanes = 8, kLanesDefault = 4;
    struct Lane { DevBuf Sall; Smoother sm; } lane[kLanes];
    struct Spans {                                       // one pair of timing events per kernel section, read back when everything has drained
        std::vector<cudaEvent_t> ev;
        ~Spans() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
        int open(cudaStream_t s) { cudaEvent_t e0 = nullptr, e1 = nullptr; CK(cudaEventCreate(&e0)); ev.push_back(e0); CK(cudaEventCreate(&e1)); ev.push_back(e1); CK(cudaEventRecord(e0, s)); return 0; }
        int close(cudaStream_t s) { CK(cudaEventRecord(ev.back(), s)); return 0; }
        int total(double* ms) { *ms = 0.0; for (size_t i = 0; i + 1 < ev.size(); i += 2) { float t = 0.f; CK(cudaEventElapsedTime(&t, ev[i], ev[i + 1])); *ms += t; } return 0; }
    } spans;
    DevBuf dd, Zd, Bd, Sd, dtmp;
    irbh::StreamGuard sg, sg_in, sg_out, sg_lane[kLanes - 1];   // after every buffer: an early return drains the streams before the buffers return to the pool
    if ((rc = sg.create()) || (rc = sg_in.create()) || (rc = sg_out.create())) return rc;
    cudaStream_t st = sg.s;
    const long long lne = (len_num + 1) & ~1LL, lde = (len_den + 1) & ~1LL;
    const bool fused = plan.big() && !smoothing;
    // items per sub-batch: about 48 MB of spectra (IRB_DECONV_SUB overrides), never more than the batch; per-item operands add
    // their spectrum (and, on the fused path, its split copy).  The per-item kernels run one item per grid.y slice, so a sub-batch
    // also stays within the 65 535 slices a launch can have (many short signals).
    const int spectra = per_item ? (fused ? 3 : 2) : 1;
    const int sub_pref = irbh::g_tuning.deconv_sub;
    int sub = sub_pref > 0 ? sub_pref : (int) std::max<long long>(1, (48LL << 20) / ((long long) sizeof(float2) * M * spectra));
    sub = std::min(std::min(sub, batch), kMaxGridY);
    // smoothing: the running sum is one sequential chain per capture and costs the same few milliseconds for 1 or 500 captures,
    // so a whole GROUP of captures is smoothed at once, between a first phase (upload | forward transform, split, divide) and a
    // last phase (merge, inverse transform | download) that both run in sub-batches with their copies overlapped; the batch is
    // cut into kLanes groups (more, in rounds, when a group would exceed about 1.5 GB of spectra and sums) that run side by side.
    const int lanes_pref = irbh::g_tuning.deconv_groups > 0 ? std::min(irbh::g_tuning.deconv_groups, kLanes) : kLanesDefault;
    const long long grp_cap = irbh::g_tuning.deconv_group_cap > 0 ? irbh::g_tuning.deconv_group_cap : (3LL << 29) / (20LL * (M + 1));
    const int grp = smoothing ? (int) std::min<long long>(batch, std::max<long long>(sub, std::min<long long>((batch + lanes_pref - 1) / lanes_pref, grp_cap))) : batch;
    const int ngroups = (batch + grp - 1) / grp, nlanes = std::min(ngroups, lanes_pref);
    const float smooth_per_avg = 1.0 / 13.0;                                          // fp/convolution.cpp:390 (a float there)
    const int nslots = batch > sub ? 2 : 1;
    long long chop_chunk_len = 0;
    const int chop_chunks_n = J.chop ? chop_chunks(sub, N, &chop_chunk_len) : 0;
    for (int i = 0; i < (smoothing ? 2 * nslots : nslots); ++i) {
        Slot& q = slot[i < nslots ? i : 2 + (i - nslots)];
        const bool first = i < nslots, last = !smoothing || !first;                // which phase(s) of the pipeline the slot serves
        if ((first && (rc = q.dn.alloc(sizeof(float) * lne * sub, true))) || (rc = q.Zn.alloc(sizeof(float2) * (size_t) M * sub, false)) ||
            (last && (rc = q.dy.alloc(sizeof(float) * (size_t) out_row * sub, false))))
            return rc;
        if (!fused && (rc = q.tmp.alloc(sizeof(float2) * (size_t) M * sub, false))) return rc;
        if (last && !include_phase && (rc = q.dy2.alloc(sizeof(float) * (size_t) N * sub, false))) return rc;
        if (last && J.chop && ((rc = q.dc.alloc(sizeof(float) * (size_t) J.chop->ir_length * sub, false)) || (rc = q.dpos.alloc(sizeof(int) * 2 * (size_t) sub, false)) ||
                               (rc = q.dpart.alloc(chop_part_bytes(sub, chop_chunks_n), false))))
            return rc;
        if (per_item && ((rc = q.dh.alloc(sizeof(float) * lde * sub, true)) || (rc = q.Zh.alloc(sizeof(float2) * (size_t) M * sub, false)) ||
                         (fused && (rc = q.Bh.alloc(sizeof(float2) * (size_t) M * sub, false)))))
            return rc;
        CK(cudaEventCreateWithFlags(&q.ev_in, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&q.ev_done, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&q.ev_out, cudaEventDisableTiming)); CK(cudaEventCreate(&q.t0)); CK(cudaEventCreate(&q.t1));
    }
    if (!per_item) {
        if ((rc = dd.alloc(sizeof(float) * lde, true)) || (rc = Zd.alloc(sizeof(float2) * (size_t) M, false)) || (rc = dtmp.alloc(sizeof(float2) * (size_t) M, false))) return rc;
        if (fused && (rc = Bd.alloc(sizeof(float2) * (size_t) M, false))) return rc;
    }
    cudaStream_t lst[kLanes];
    for (int l = 0; l < kLanes; ++l) lst[l] = st;
    cudaEvent_t ev_den = nullptr, ev_join[kLanes] = {};
    struct EvGuard { cudaEvent_t& d; cudaEvent_t* j; ~EvGuard() { if (d) cudaEventDestroy(d); for (int i = 0; i < kLanes; ++i) if (j[i]) cudaEventDestroy(j[i]); } } evg{ev_den, ev_join};
    if (smoothing) {
        if ((rc = Sd.alloc(sizeof(float2) * (size_t) (M + 1), false))) return rc;
        CK(cudaEventCreateWithFlags(&ev_den, cudaEventDisableTiming));
        for (int l = 0; l < nlanes; ++l) {
            if (l && (rc = sg_lane[l - 1].create())) return rc;
            if (l) lst[l] = sg_lane[l - 1].s;
            if ((rc = lane[l].Sall.alloc(sizeof(float2) * (size_t) (M + 1) * grp, false)) || (rc = lane[l].sm.init(M, grp, (double) smooth_per_avg, sample_rate, 1, lst[l]))) return rc;
            CK(cudaEventCreateWithFlags(&ev_join[l], cudaEventDisableTiming));
        }
    }
    irbh::set_last_compute_ms(0.0);
    // a shared operand's spectrum, once (the reciprocal for a division)
    if (!per_item) {
        CK(cudaMemcpyAsync(dd.p, J.h, sizeof(float) * len_den, cudaMemcpyDefault, st));
        if (fused) {
            if ((rc = plan.cols_fwd(dd.p, lde / 2, len_den, Zd.as<float2>(), 1, st)) || (rc = plan.rows_to_split_spectrum(Zd.as<float2>(), Bd.as<float2>(), 1, J.divide, st))) return rc;
        } else {
            if ((rc = plan.run(dd.p, lde / 2, len_den, Zd.as<float2>(), M, dtmp.as<float2>(), 1, false, 1.0f, st))) return rc;
            if (smoothing) {
                irb::k_spec_split<<<grid1(M + 1, 1), 256, 0, st>>>(Zd.as<float2>(), M, Sd.as<float2>(), M + 1, M, 0, plan.WN);
                LAUNCHED();
            }
        }
    }
    double total_ms = 0.0;
    auto collect = [&](Slot& q) -> int {          // kernel time of the section that last used this slot
        if (!q.timed) return 0;
        CK(cudaEventSynchronize(q.t1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, q.t0, q.t1));
        total_ms += ms;
        q.timed = false;
        return 0;
    };
    // upload of a sub-batch into q.dn (and its per-item operands into q.dh) after the kernels that last used the slot, and the
    // compute stream cs waiting for it
    auto upload = [&](Slot& q, int b0, int nb, cudaStream_t cs) -> int {
        if (q.dn_busy) CK(cudaStreamWaitEvent(sg_in.s, q.ev_done, 0));
        CK(cudaMemcpy2DAsync(q.dn.p, sizeof(float) * lne, nums + (size_t) b0 * len_num, sizeof(float) * len_num, sizeof(float) * len_num, nb, cudaMemcpyDefault, sg_in.s));
        if (per_item)
            CK(cudaMemcpy2DAsync(q.dh.p, sizeof(float) * lde, J.h + (size_t) b0 * len_den, sizeof(float) * len_den, sizeof(float) * len_den, nb, cudaMemcpyDefault, sg_in.s));
        CK(cudaEventRecord(q.ev_in, sg_in.s));
        CK(cudaStreamWaitEvent(cs, q.ev_in, 0));
        return 0;
    };
    // inverse-transformed sub-batch in q.dy -> (half swap) -> (chop) -> host
    auto download = [&](Slot& q, int b0, int nb, cudaStream_t cs) -> int {
        const float* res = q.dy.as<float>();
        if (!include_phase) {                                                        // ir::shifteroo, fp/convolution.cpp:400
            irb::k_shifteroo<<<grid1(N, nb), 256, 0, cs>>>(q.dy.as<float>(), q.dy2.as<float>(), N, N);
            LAUNCHED();
            res = q.dy2.as<float>();
        }
        if (J.chop) { int rc2 = launch_chop(res, nb, N, chop_chunks_n, chop_chunk_len, *J.chop, q.dc.as<float>(), q.dpos.as<int>(), q.dpart.p, cs); if (rc2) return rc2; }
        if (smoothing) { int rc2 = spans.close(cs); if (rc2) return rc2; }
        else CK(cudaEventRecord(q.t1, cs));
        CK(cudaEventRecord(q.ev_done, cs));
        CK(cudaStreamWaitEvent(sg_out.s, q.ev_done, 0));
        if (J.chop) {                                                                // only the IRs (and their positions) leave the device
            const long long Lw = J.chop->ir_length;
            CK(cudaMemcpyAsync(J.out + (size_t) b0 * Lw, q.dc.p, sizeof(float) * (size_t) Lw * nb, cudaMemcpyDefault, sg_out.s));
            if (J.chop->positions) CK(cudaMemcpyAsync(J.chop->positions + 2 * (size_t) b0, q.dpos.p, sizeof(int) * 2 * (size_t) nb, cudaMemcpyDefault, sg_out.s));
        } else {
            CK(cudaMemcpyAsync(J.out + (size_t) b0 * out_row, res, sizeof(float) * (size_t) out_row * nb, cudaMemcpyDefault, sg_out.s));
        }
        CK(cudaEventRecord(q.ev_out, sg_out.s));
        q.dy_busy = true;
        return 0;
    };
    int it = 0;
    if (!smoothing) {
        const float inv_n = 1.0f / (float) N;
        const OutWindow win{J.win.off, out_row, J.win.len};
        for (int b0 = 0; b0 < batch; b0 += sub, ++it) {
            Slot& q = slot[it % nslots];
            const int nb = std::min(sub, batch - b0);
            if ((rc = collect(q)) || (rc = upload(q, b0, nb, st))) return rc;
            if (q.dy_busy) CK(cudaStreamWaitEvent(st, q.ev_out, 0));                  // the previous download has drained q.dy
            CK(cudaEventRecord(q.t0, st));
            q.timed = true;
            if (fused) {
                const float2* B = Bd.as<float2>();
                if (per_item) {
                    if ((rc = plan.cols_fwd(q.dh.p, lde / 2, len_den, q.Zh.as<float2>(), nb, st)) ||
                        (rc = plan.rows_to_split_spectrum(q.Zh.as<float2>(), q.Bh.as<float2>(), nb, J.divide, st)))
                        return rc;
                    B = q.Bh.as<float2>();
                }
                if ((rc = plan.cols_fwd(q.dn.p, lne / 2, len_num, q.Zn.as<float2>(), nb, st)) || (rc = plan.rows_binop(q.Zn.as<float2>(), B, per_item ? M : 0, nb, st)) ||
                    (rc = plan.cols_inv(q.Zn.as<float2>(), q.dy.as<float2>(), M, nb, inv_n, st, win)))
                    return rc;
            } else {
                const float2* B = Zd.as<float2>();
                if (per_item) {
                    if ((rc = plan.run(q.dh.p, lde / 2, len_den, q.Zh.as<float2>(), M, q.tmp.as<float2>(), nb, false, 1.0f, st))) return rc;
                    B = q.Zh.as<float2>();
                }
                if ((rc = plan.run(q.dn.p, lne / 2, len_num, q.Zn.as<float2>(), M, q.tmp.as<float2>(), nb, false, 1.0f, st))) return rc;
                const long long bs = per_item ? M : 0;
                if (J.divide) irb::k_spec_fused<true><<<grid1(M / 2 + 1, nb), 256, 0, st>>>(q.Zn.as<float2>(), M, B, bs, q.Zn.as<float2>(), M, M, plan.WN);
                else irb::k_spec_fused<false><<<grid1(M / 2 + 1, nb), 256, 0, st>>>(q.Zn.as<float2>(), M, B, bs, q.Zn.as<float2>(), M, M, plan.WN);
                LAUNCHED();
                if ((rc = plan.run(q.Zn.p, M, -1, q.dy.as<float2>(), M, q.tmp.as<float2>(), nb, true, inv_n, st, win))) return rc;
            }
            if ((rc = download(q, b0, nb, st))) return rc;
            q.dn_busy = true;
        }
        CK(cudaStreamSynchronize(sg_out.s));
        CK(cudaStreamSynchronize(st));
        for (int i = 0; i < nslots; ++i) if ((rc = collect(slot[i]))) return rc;
        irbh::set_last_compute_ms(total_ms);
        return 0;
    }
    // ---- smoothing: groups of captures side by side, one lane (stream, spectrum array, smoother) each; rounds of nlanes groups.
    // Nothing below blocks the host: the first phase and the last phase have their own staging slots, slot and lane reuse is ordered by
    // events on the device, and the kernel sections' timing events are read when everything has drained -- so the downloads of the first
    // group start as soon as its running sums are done, under the uploads of the later groups. ----
    bool slot_used[4] = {false, false, false, false};
    cudaEvent_t w0 = nullptr, w1 = nullptr;
    struct WallGuard { cudaEvent_t& a; cudaEvent_t& b; ~WallGuard() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); } } wall_guard{w0, w1};
    CK(cudaEventCreate(&w0)); CK(cudaEventCreate(&w1));
    CK(cudaEventRecord(w0, st));
    CK(cudaEventRecord(ev_den, st));
    for (int l = 1; l < nlanes; ++l) CK(cudaStreamWaitEvent(lst[l], ev_den, 0));     // the denominator's spectrum
    int it_last = 0;
    for (int r0 = 0; r0 < ngroups; r0 += nlanes) {
        const int rn = std::min(nlanes, ngroups - r0);
        for (int l = 0; l < rn; ++l) {                                               // first phase and the running sums of every group of the round
            const int g0 = (r0 + l) * grp, gn = std::min(grp, batch - g0);
            cudaStream_t cs = lst[l];
            for (int b0 = g0; b0 < g0 + gn; b0 += sub, ++it) {
                const int qi = it % nslots;
                Slot& q = slot[qi];
                const int nb = std::min(sub, g0 + gn - b0);
                if (slot_used[qi]) CK(cudaStreamWaitEvent(cs, q.ev_done, 0));          // another lane's kernels may have used the slot last
                if ((rc = upload(q, b0, nb, cs)) || (rc = spans.open(cs))) return rc;
                if ((rc = plan.run(q.dn.p, lne / 2, len_num, q.Zn.as<float2>(), M, q.tmp.as<float2>(), nb, false, 1.0f, cs))) return rc;
                float2* Sg = lane[l].Sall.as<float2>() + (size_t) (b0 - g0) * (M + 1);
                irb::k_spec_split<<<grid1(M + 1, nb), 256, 0, cs>>>(q.Zn.as<float2>(), M, Sg, M + 1, M, 0, plan.WN);
                LAUNCHED();
                irb::k_spec_binop<true><<<grid1(M + 1, nb), 256, 0, cs>>>(Sg, M + 1, Sd.as<float2>(), 0, M);
                LAUNCHED();
                if ((rc = spans.close(cs))) return rc;
                CK(cudaEventRecord(q.ev_done, cs));
                q.dn_busy = true;
                slot_used[qi] = true;
            }
            if ((rc = spans.open(cs)) || (rc = lane[l].sm.run(lane[l].Sall.as<float2>(), M + 1, gn, 3, 1, include_phase, include_amplitude, cs)) || (rc = spans.close(cs))) return rc;
        }
        for (int l = 0; l < rn; ++l) {                                               // last phase
            const int g0 = (r0 + l) * grp, gn = std::min(grp, batch - g0);
            cudaStream_t cs = lst[l];
            for (int b0 = g0; b0 < g0 + gn; b0 += sub, ++it_last) {
                const int qi = 2 + it_last % nslots;
                Slot& q = slot[qi];
                const int nb = std::min(sub, g0 + gn - b0);
                if (slot_used[qi]) CK(cudaStreamWaitEvent(cs, q.ev_done, 0));
                if (q.dy_busy) CK(cudaStreamWaitEvent(cs, q.ev_out, 0));
                if ((rc = spans.open(cs))) return rc;
                irb::k_spec_merge<<<grid1(M, nb), 256, 0, cs>>>(lane[l].Sall.as<float2>() + (size_t) (b0 - g0) * (M + 1), M + 1, q.Zn.as<float2>(), M, M, plan.WN);
                LAUNCHED();
                if ((rc = plan.run(q.Zn.p, M, -1, q.dy.as<float2>(), M, q.tmp.as<float2>(), nb, true, 1.0f / (float) N, cs))) return rc;
                if ((rc = download(q, b0, nb, cs))) return rc;                        // closes the section
                slot_used[qi] = true;
            }
        }
    }
    for (int l = 1; l < nlanes; ++l) { CK(cudaEventRecord(ev_join[l], lst[l])); CK(cudaStreamWaitEvent(st, ev_join[l], 0)); }
    CK(cudaEventRecord(ev_join[0], sg_out.s)); CK(cudaStreamWaitEvent(st, ev_join[0], 0));
    CK(cudaEventRecord(w1, st));
    CK(cudaStreamSynchronize(sg_out.s));
    for (int l = 0; l < nlanes; ++l) CK(cudaStreamSynchronize(lst[l]));
    if (device_io) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, w0, w1));
        irbh::set_last_compute_ms((double) ms);
        return 0;
    }
    if ((rc = spans.total(&total_ms))) return rc;
    irbh::set_last_compute_ms(total_ms);
    return 0;
}

// The same on DEVICE-resident inputs and results with no staging at all: every sub-batch's column pass reads the signals (and
// per-item operands) where they lie, the inverse column pass writes the results (or their windows) where they belong, and
// consecutive sub-batches alternate between compute streams so that one sub-batch's row kernels fill the SMs another one's column
// pass leaves idle.  Needs the fused four-step plan, float2-aligned rows of x (and of a per-item h, which must be in device memory)
// and, without a window, of out.  irb_last_compute_ms() is the device time of the whole call.
static int batch_direct(const BatchJob& J, const Plan& plan) {
    const int batch = J.batch, len_num = J.len_x, len_den = J.len_h, N = J.N, M = N / 2;
    const bool per_item = J.h_batch > 1;
    const long long out_row = J.out_row();
    constexpr int kStreams = 3;
    const int spectra = per_item ? 3 : 1;
    const int sub_pref = irbh::g_tuning.deconv_sub;
    int sub = sub_pref > 0 ? sub_pref : (int) std::max<long long>(1, (32LL << 20) / ((long long) sizeof(float2) * M * spectra));      // about 32 MB of spectra per sub-batch
    sub = std::min(sub, batch);
    const int ncs = std::max(1, std::min(std::min(kStreams, irbh::g_tuning.deconv_streams > 0 ? irbh::g_tuning.deconv_streams : 2), (batch + sub - 1) / sub));
    const long long lde = (len_den + 1) & ~1LL;
    int rc;
    DevBuf Zn[kStreams], Zh[kStreams], Bh[kStreams], dd, Zd, Bd;
    cudaEvent_t e0 = nullptr, e1 = nullptr, ev_den = nullptr, ev_end[kStreams] = {nullptr, nullptr, nullptr};
    struct EvGuard { cudaEvent_t *a, *b, *c, *d; ~EvGuard() { for (cudaEvent_t* e : {a, b, c}) if (*e) cudaEventDestroy(*e); for (int i = 0; i < kStreams; ++i) if (d[i]) cudaEventDestroy(d[i]); } } evg{&e0, &e1, &ev_den, ev_end};
    irbh::StreamGuard cs[kStreams];                      // after the buffers and events: drained first on an early return
    for (int i = 0; i < ncs; ++i) {
        if ((rc = cs[i].create()) || (rc = Zn[i].alloc(sizeof(float2) * (size_t) M * sub, false))) return rc;
        if (per_item && ((rc = Zh[i].alloc(sizeof(float2) * (size_t) M * sub, false)) || (rc = Bh[i].alloc(sizeof(float2) * (size_t) M * sub, false)))) return rc;
        CK(cudaEventCreateWithFlags(&ev_end[i], cudaEventDisableTiming));
    }
    if (!per_item && ((rc = dd.alloc(sizeof(float) * lde, true)) || (rc = Zd.alloc(sizeof(float2) * (size_t) M, false)) || (rc = Bd.alloc(sizeof(float2) * (size_t) M, false)))) return rc;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1)); CK(cudaEventCreateWithFlags(&ev_den, cudaEventDisableTiming));
    cudaStream_t st = cs[0].s;
    if (!per_item) {
        CK(cudaMemcpyAsync(dd.p, J.h, sizeof(float) * len_den, cudaMemcpyDefault, st));
        CK(cudaEventRecord(e0, st));
        // the shared operand's spectrum (the reciprocal for a division) in row layout, once
        if ((rc = plan.cols_fwd(dd.p, lde / 2, len_den, Zd.as<float2>(), 1, st)) || (rc = plan.rows_to_split_spectrum(Zd.as<float2>(), Bd.as<float2>(), 1, J.divide, st))) return rc;
    } else {
        CK(cudaEventRecord(e0, st));
    }
    CK(cudaEventRecord(ev_den, st));
    for (int i = 1; i < ncs; ++i) CK(cudaStreamWaitEvent(cs[i].s, ev_den, 0));
    const OutWindow win{J.win.off, out_row, J.win.len};
    int it = 0;
    for (int b0 = 0; b0 < batch; b0 += sub, ++it) {
        const int k = it % ncs, nb = std::min(sub, batch - b0);
        cudaStream_t s = cs[k].s;
        const float2* B = Bd.as<float2>();
        if (per_item) {
            if ((rc = plan.cols_fwd(J.h + (size_t) b0 * len_den, len_den / 2, len_den, Zh[k].as<float2>(), nb, s)) ||
                (rc = plan.rows_to_split_spectrum(Zh[k].as<float2>(), Bh[k].as<float2>(), nb, J.divide, s)))
                return rc;
            B = Bh[k].as<float2>();
        }
        if ((rc = plan.cols_fwd(J.x + (size_t) b0 * len_num, len_num / 2, len_num, Zn[k].as<float2>(), nb, s)) ||
            (rc = plan.rows_binop(Zn[k].as<float2>(), B, per_item ? M : 0, nb, s)) ||
            (rc = plan.cols_inv(Zn[k].as<float2>(), reinterpret_cast<float2*>(J.out + (size_t) b0 * out_row), M, nb, 1.0f / (float) N, s, win)))
            return rc;
    }
    for (int i = 1; i < ncs; ++i) { CK(cudaEventRecord(ev_end[i], cs[i].s)); CK(cudaStreamWaitEvent(st, ev_end[i], 0)); }
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    irbh::set_last_compute_ms((double) ms);
    return 0;
}

// the division's job: nums[batch][len_num] / den[len_den] -> out[batch][N], N = nextPowerOfTwo(max(len_num, len_den))
static int deconvolve_job(const float* nums, int batch, int len_num, const float* den, int len_den, float* out, BatchJob* J) {
    if (!nums || !den || !out) return fail(IRB_ERR_ARG, "null argument");
    if (batch < 1 || len_num < 1 || len_den < 1) return fail(IRB_ERR_ARG, "empty input");
    int N = 0, rc;
    if ((rc = fft_size_for(len_num > len_den ? len_num : len_den, &N))) return rc;
    *J = BatchJob{nums, batch, len_num, den, 1, len_den, N, true, OutWindow{}, out};
    return 0;
}

// the convolution's job (include/irb_b200.h, irb_convolve_batch); every argument error is found here, before any CUDA call
static int convolve_job(const float* x, int batch, int len_x, const float* h, int h_batch, int len_h, int out_offset, int out_len, float* out, BatchJob* J) {
    if (!x || !h || !out) return fail(IRB_ERR_ARG, "null argument");
    if (batch < 1 || len_x < 1 || len_h < 1) return fail(IRB_ERR_ARG, "empty input");
    if (h_batch != 1 && h_batch != batch) return fail(IRB_ERR_ARG, "h_batch %d: one IR for every signal (1) or one per signal (%d)", h_batch, batch);
    const long long Lout = (long long) len_x + len_h - 1;
    if (out_offset < 0 || out_len < 1 || (long long) out_offset + out_len > Lout)
        return fail(IRB_ERR_ARG, "window [%d, %lld) is empty or outside the %lld samples of the result", out_offset, (long long) out_offset + out_len, Lout);
    if (Lout > 2LL * kMaxBigM) return fail(IRB_ERR_ARG, "result of %lld samples needs an FFT above 2^22 points", Lout);
    int N = 2 * kMinM;                                   // a longer zero-padded transform yields the same linear convolution
    while (N < Lout) N *= 2;
    *J = BatchJob{x, batch, len_x, h, h_batch, len_h, N, false, OutWindow{out_offset, out_len, out_len}, out};
    return 0;
}

// memory a pointer lies in: device (or managed) memory can be read in place by the kernels
static bool on_device(const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

extern "C" {

// fp::convolution::convolveNonPeriodic (fp/convolution.cpp:246-347): each channel of the audio is one item of the batched
// convolution, with the IR channel of its own (stereo / stereo, :320-323) or the one IR (stereo audio, mono IR); a stereo IR
// for mono audio is folded to mono first (IRStereoAudioMono -> sumToMono, :302)
int irb_convolve_nonperiodic(const float* x, int ch_x, int len_x, const float* h, int ch_h, int len_h, float* out) {
    if (!x || !h || !out) return fail(IRB_ERR_ARG, "null argument");
    if (len_x < 1 || len_h < 1 || ch_x < 1 || ch_h < 1) return fail(IRB_ERR_ARG, "empty input");
    if (!((ch_x == 1 || ch_x == 2) && (ch_h == 1 || ch_h == 2)))
        return fail(IRB_ERR_LAYOUT, "audio has %d channels and the IR %d: only mono/stereo layouts exist (fp/convolution.cpp:259-275)", ch_x, ch_h);
    const long long Lout = (long long) len_x + len_h - 1;
    if (Lout > 2LL * kMaxBigM) return fail(IRB_ERR_ARG, "result of %lld samples needs an FFT above 2^22 points", Lout);
    if (!(ch_h == 2 && ch_x == 1)) return irb_convolve_batch(x, ch_x, len_x, h, ch_h, len_h, 0, (int) Lout, out);
    DevBuf dh, dhf;
    irbh::StreamGuard sg;
    int rc;
    CK(cudaSetDevice(irbh::current_device()));
    if ((rc = sg.create())) return rc;
    const long long lhe = (len_h + 1) & ~1LL;
    if ((rc = dh.alloc(sizeof(float) * lhe * 2, false)) || (rc = dhf.alloc(sizeof(float) * lhe, false))) return rc;
    for (int c = 0; c < 2; ++c) CK(cudaMemcpyAsync(dh.as<float>() + c * lhe, h + (size_t) c * len_h, sizeof(float) * len_h, cudaMemcpyHostToDevice, sg.s));
    cudaEvent_t f0 = nullptr, f1 = nullptr;
    struct EvGuard { cudaEvent_t &a, &b; ~EvGuard() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); } } evg{f0, f1};
    CK(cudaEventCreate(&f0)); CK(cudaEventCreate(&f1));
    CK(cudaEventRecord(f0, sg.s));
    irb::k_fold_mono<<<grid1(len_h, 1), 256, 0, sg.s>>>(dh.as<float>(), dh.as<float>() + lhe, dhf.as<float>(), len_h);
    LAUNCHED();
    CK(cudaEventRecord(f1, sg.s));
    // the batch core runs on streams of its own and reads the folded IR as device memory: it has to be complete first
    CK(cudaEventSynchronize(f1));
    if ((rc = irb_convolve_batch(x, 1, len_x, dhf.as<float>(), 1, len_h, 0, (int) Lout, out))) return rc;
    float fold_ms = 0.f;                                 // irb_last_compute_ms() covers the fold too
    CK(cudaEventElapsedTime(&fold_ms, f0, f1));
    irbh::set_last_compute_ms(irb_last_compute_ms() + fold_ms);
    return 0;
}

int irb_convolve_batch(const float* x, int batch, int len_x, const float* h, int h_batch, int len_h, int out_offset, int out_len, float* out) {
    BatchJob J;
    const int rc = convolve_job(x, batch, len_x, h, h_batch, len_h, out_offset, out_len, out, &J);
    return rc ? rc : batch_staged(J, 0.0, 0, 1, 1, false);
}

// Staging-free when the transform is a four-step one, x_dev is float2-aligned with an even len_x, and a per-item h lies in device
// memory, float2-aligned with an even len_h (a shared h is copied once from wherever it is); any other case goes through the staged
// pipeline with device-to-device copies.  The windowed store is scalar, so out_dev needs no more than float alignment either way.
int irb_convolve_batch_device(const float* x_dev, int batch, int len_x, const float* h, int h_batch, int len_h, int out_offset, int out_len, float* out_dev) {
    BatchJob J;
    int rc;
    if ((rc = convolve_job(x_dev, batch, len_x, h, h_batch, len_h, out_offset, out_len, out_dev, &J))) return rc;
    const int dev = irbh::current_device();
    CK(cudaSetDevice(dev));
    Plan plan;
    if ((rc = plan.init(dev, J.N / 2))) return rc;
    const bool x_direct = (uintptr_t) x_dev % alignof(float2) == 0 && len_x % 2 == 0;
    const bool h_direct = h_batch == 1 || ((uintptr_t) h % alignof(float2) == 0 && len_h % 2 == 0 && on_device(h));
    if (!(plan.big() && x_direct && h_direct)) return batch_staged(J, 0.0, 0, 1, 1, true);
    return batch_direct(J, plan);
}

int irb_deconvolve_batch(const float* nums, int batch, int len_num, const float* den, int len_den, double sample_rate, int smoothing, int include_phase,
                         int include_amplitude, float* out) {
    BatchJob J;
    const int rc = deconvolve_job(nums, batch, len_num, den, len_den, out, &J);
    return rc ? rc : batch_staged(J, sample_rate, smoothing, include_phase, include_amplitude, false);
}

// The same with DEVICE-resident captures and results (den: host or device).  Large plain divisions (no smoothing, phase kept, an
// even capture length) run with no staging at all (batch_direct).  The column passes read the captures and write the results as
// float2, so that path also needs both pointers 8-byte aligned (a float view at an odd offset is only 4-byte aligned).  Everything
// else goes through the staged pipeline with device-to-device copies, which take any alignment.  irb_last_compute_ms() is the
// device time of the whole call.
int irb_deconvolve_batch_device(const float* nums_dev, int batch, int len_num, const float* den, int len_den, double sample_rate, int smoothing, int include_phase,
                                int include_amplitude, float* out_dev) {
    BatchJob J;
    int rc;
    if ((rc = deconvolve_job(nums_dev, batch, len_num, den, len_den, out_dev, &J))) return rc;
    const int dev = irbh::current_device();
    CK(cudaSetDevice(dev));
    Plan plan;
    if ((rc = plan.init(dev, J.N / 2))) return rc;
    const bool aligned = (((uintptr_t) nums_dev | (uintptr_t) out_dev) % alignof(float2)) == 0;
    if (!(plan.big() && !smoothing && include_phase && len_num % 2 == 0 && aligned))
        return batch_staged(J, sample_rate, smoothing, include_phase, include_amplitude, true);
    return batch_direct(J, plan);
}

int irb_deconvolve_chop_batch(const float* nums, int batch, int len_num, const float* den, int len_den, double sample_rate, int smoothing, int include_phase,
                              int include_amplitude, int ir_length, float threshold_db, int consecutive, int normalize, float goal_db, float* out, int* positions) {
    BatchJob J;
    ChopSpec c;
    int rc;
    if ((rc = deconvolve_job(nums, batch, len_num, den, len_den, out, &J)) || (rc = chop_spec(J.N, ir_length, threshold_db, consecutive, normalize, goal_db, positions, &c)))
        return rc;
    J.chop = &c;
    return batch_staged(J, sample_rate, smoothing, include_phase, include_amplitude, false);
}

int irb_ir_chop_batch_device(const float* x_dev, int batch, int len, int ir_length, float threshold_db, int consecutive, int normalize, float goal_db, float* out_dev,
                             int* positions) {
    if (!x_dev || !out_dev) return fail(IRB_ERR_ARG, "null argument");
    if (batch < 1 || len < 1) return fail(IRB_ERR_ARG, "empty input");
    ChopSpec c;
    int rc;
    if ((rc = chop_spec(len, ir_length, threshold_db, consecutive, normalize, goal_db, positions, &c))) return rc;
    CK(cudaSetDevice(irbh::current_device()));
    long long chunk_len = 0;
    const int chunks = chop_chunks(batch, len, &chunk_len);
    DevBuf part;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    struct EvGuard { cudaEvent_t &a, &b; ~EvGuard() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); } } evg{e0, e1};
    irbh::StreamGuard sg;
    if ((rc = sg.create()) || (rc = part.alloc(chop_part_bytes(batch, chunks), false))) return rc;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0, sg.s));
    if ((rc = launch_chop(x_dev, batch, len, chunks, chunk_len, c, out_dev, positions, part.p, sg.s))) return rc;
    CK(cudaEventRecord(e1, sg.s));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    irbh::set_last_compute_ms((double) ms);
    return 0;
}

int irb_deconvolve(const float* num, int len_num, const float* den, int len_den, double sample_rate, int smoothing, int include_phase, int include_amplitude,
                   float* out) {
    return irb_deconvolve_batch(num, 1, len_num, den, len_den, sample_rate, smoothing, include_phase, include_amplitude, out);
}

// fp::ir::invertFilter (fp/ir.cpp:13-18): deconvolve(generatePulse(len), x, sr) with the default flags
int irb_invert_filter(const float* x, int len, int sample_rate, float* out) {
    if (!x || !out || len < 1) return fail(IRB_ERR_ARG, "bad argument");
    std::vector<float> pulse((size_t) len, 0.0f);
    pulse[0] = 1.0f;                                                                 // tools::generatePulse, fp/tools.cpp:235-241
    return irb_deconvolve_batch(pulse.data(), 1, len, x, len, (double) sample_rate, 1, 1, 1, out);
}

// fp::tools::fftTransform (fp/tools.cpp:321-346): x[ch][len] -> out[ch][2N]; only channel 0 carries data (:328)
int irb_fft_transform(const float* x, int ch, int len, int format_ampl_phase, float* out) {
    if (!x || !out || ch < 1 || len < 1) return fail(IRB_ERR_ARG, "bad argument");
    int N = 0, rc;
    if ((rc = fft_size_for(len, &N))) return rc;
    const int M = N / 2, dev = irbh::current_device();
    CK(cudaSetDevice(dev));
    Plan plan;
    if ((rc = plan.init(dev, M))) return rc;
    DevBuf dx, Z, tmp, S;
    irbh::StreamGuard sg;
    if ((rc = sg.create())) return rc;
    cudaStream_t st = sg.s;
    if ((rc = dx.alloc(sizeof(float) * ((size_t) len + 1), true)) || (rc = Z.alloc(sizeof(float2) * (size_t) M, false)) || (rc = tmp.alloc(sizeof(float2) * (size_t) M, false)) ||
        (rc = S.alloc(sizeof(float2) * (size_t) N, true)))
        return rc;
    CK(cudaMemcpyAsync(dx.p, x, sizeof(float) * len, cudaMemcpyHostToDevice, st));
    if ((rc = plan.run(dx.p, 0, len, Z.as<float2>(), M, tmp.as<float2>(), 1, false, 1.0f, st))) return rc;
    irb::k_spec_split<<<grid1(M + 1, 1), 256, 0, st>>>(Z.as<float2>(), M, S.as<float2>(), N, M, 1, plan.WN);
    LAUNCHED();
    if (format_ampl_phase) { irb::k_spec_ampl_phase<<<grid1(M + 1, 1), 256, 0, st>>>(S.as<float2>(), N, M); LAUNCHED(); }
    memset(out, 0, sizeof(float) * 2 * (size_t) N * ch);                              // channels >= 1 transform silence
    CK(cudaMemcpyAsync(out, S.p, sizeof(float) * 2 * (size_t) N, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// fp::tools::fftInvTransform (fp/tools.cpp:351-369): spec[ch][fft_size] (interleaved, bins 0..N/2 used) -> out[ch][N], N = fft_size/2
int irb_fft_inv_transform(const float* spec, int ch, int fft_size, float* out) {
    if (!spec || !out || ch < 1 || fft_size < 2) return fail(IRB_ERR_ARG, "bad argument");
    const int N = fft_size / 2, M = N / 2, dev = irbh::current_device();
    int rc;
    if (N != irbh::next_pow2(N) || M < kMinM) return fail(IRB_ERR_ARG, "fft_size %d: N must be a power of two >= %d", fft_size, 2 * kMinM);
    CK(cudaSetDevice(dev));
    Plan plan;
    if ((rc = plan.init(dev, M))) return rc;
    DevBuf S, Z, tmp, dy;
    irbh::StreamGuard sg;
    if ((rc = sg.create())) return rc;
    cudaStream_t st = sg.s;
    if ((rc = S.alloc(sizeof(float) * (size_t) fft_size * ch, false)) || (rc = Z.alloc(sizeof(float2) * (size_t) M * ch, false)) ||
        (rc = tmp.alloc(sizeof(float2) * (size_t) M * ch, false)) || (rc = dy.alloc(sizeof(float2) * (size_t) M * ch, false)))
        return rc;
    CK(cudaMemcpyAsync(S.p, spec, sizeof(float) * (size_t) fft_size * ch, cudaMemcpyHostToDevice, st));
    irb::k_spec_merge<<<grid1(M, ch), 256, 0, st>>>(S.as<float2>(), N, Z.as<float2>(), M, M, plan.WN);
    LAUNCHED();
    if ((rc = plan.run(Z.p, M, -1, dy.as<float2>(), M, tmp.as<float2>(), ch, true, 1.0f / (float) N, st))) return rc;
    CK(cudaMemcpyAsync(out, dy.p, sizeof(float) * (size_t) N * ch, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// fp::convolution::averagingFilter (fp/convolution.cpp:406-546), in place on spec[ch][fft_size]
int irb_averaging_filter(float* spec, int ch, int fft_size, double octave_fraction, double sample_rate, int log_avg, int include_phase, int include_amplitude) {
    if (!spec || ch < 1 || fft_size < 4) return fail(IRB_ERR_ARG, "bad argument");
    if (fft_size & (fft_size - 1)) return 0;                                          // not a power of two: untouched (:412-415)
    const int N = fft_size / 2, M = N / 2, dev = irbh::current_device();
    CK(cudaSetDevice(dev));
    DevBuf S;
    Smoother sm;
    irbh::StreamGuard sg;
    int rc;
    if ((rc = sg.create())) return rc;
    cudaStream_t st = sg.s;
    if ((rc = S.alloc(sizeof(float) * (size_t) fft_size * ch, false)) || (rc = sm.init(M, ch, octave_fraction, sample_rate, log_avg, st))) return rc;
    CK(cudaMemcpyAsync(S.p, spec, sizeof(float) * (size_t) fft_size * ch, cudaMemcpyHostToDevice, st));
    if ((rc = sm.run(S.as<float2>(), N, ch, 1, log_avg, include_phase, include_amplitude, st))) return rc;
    CK(cudaMemcpyAsync(spec, S.p, sizeof(float) * (size_t) fft_size * ch, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// fp::ExpSineSweep::generate / generateInv (fp/ExpSineSweep.cpp:26-41,59-79,212-220) in FP64 on the device.
// Returns the sweep length (int) (sample_rate * duration); writes min(length, capacity) doubles when out != NULL.
int irb_ess_generate(double duration_s, double sample_rate, double f1, double f2, double gain_db, int inverse, double* out, int capacity) {
    const double T = sample_rate * duration_s;
    const double w1 = f1 / sample_rate * 2 * M_PI, w2 = f2 / sample_rate * 2 * M_PI;
    if (!(T >= 1.0) || !(f1 > 0) || !(f2 > f1) || T > 2147483647.0) return fail(IRB_ERR_ARG, "bad sweep parameters");
    const double K = T * w1 / log(w2 / w1), L = T / log(w2 / w1);
    const int n = (int) T;
    if (!out) return n;
    const int m = std::min(n, capacity);
    if (m <= 0) return n;
    const double g = pow(10.0, gain_db / 20.0);                                       // tools::dBToLin(double), fp/tools.cpp:93-95
    const double kdecay = pow(10.0, (-6.0 * log2(w2 / w1)) / 20.0 / T);               // fp/ExpSineSweep.cpp:70
    CK(cudaSetDevice(irbh::current_device()));
    DevBuf d;
    irbh::StreamGuard sg;
    int rc;
    if ((rc = sg.create())) return rc;
    if ((rc = d.alloc(sizeof(double) * (size_t) n, false))) return rc;
    irb::k_ess<<<grid1(n, 1), 256, 0, sg.s>>>(d.as<double>(), n, g, K, L, inverse, kdecay);
    LAUNCHED();
    CK(cudaMemcpyAsync(out, d.p, sizeof(double) * (size_t) m, cudaMemcpyDeviceToHost, sg.s));
    CK(cudaStreamSynchronize(sg.s));
    return n;
}

}  // extern "C"
