/*
 * irb_b200.h -- C ABI of the B200-native partitioned-convolution engine (libirb_b200.so).
 *
 * This is the drop-in boundary for ONE path of Flixor/IRBaboon: the uniformly partitioned FFT
 * convolution engine and the spectral-division deconvolution that reuses its kernels.  The reference
 * has no FFI of its own (it is a C++14 JUCE plugin); what a maintainer binds is its fp:: header surface,
 * so each entry point below names the reference interface it stands behind (paths relative to the
 * reference tree).  The C++ facade in irbaboon_b200/fp/ (same namespaces, names, defaults as the
 * reference's fp/ headers) is a thin wrapper over these calls -- see INTEGRATION.md.
 *
 * Conventions: plain pointers and sizes, no C++/torch types.  All audio is float32, except that the streaming engine's
 * _pcm entry points also take and return 16- and 24-bit integer PCM (irb_sample_format).  Every function
 * returns 0 on success or a negative irb_status; irb_last_error() gives the message of the calling
 * thread's most recent failure.  No exception crosses this boundary.  There is NO CPU fallback: if no
 * sm_100 device is usable every compute entry point fails with IRB_ERR_CUDA.
 *
 * Threading: one thread drives a given irb_engine at a time (the audio callback, as in the reference);
 * different engines are independent.  The offline functions are re-entrant.
 */
#ifndef IRB_B200_H
#define IRB_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum irb_status {
    IRB_OK = 0,
    IRB_ERR_ARG = -1,      /* bad argument (size, null pointer, unsupported block size) */
    IRB_ERR_LAYOUT = -2,   /* channel layout the reference rejects (fp/convolution.cpp:39-42): outputs are zeroed */
    IRB_ERR_CUDA = -3,     /* CUDA runtime failure / no usable device */
    IRB_ERR_STATE = -4     /* call not valid in the engine's current state */
} irb_status;

typedef struct irb_engine irb_engine;

/* Sample format of the block arrays of the streaming engine's _pcm entry points.  The layout does not change with the format:
 * [n_blocks][channels][block_size] elements.  S16 is an int16_t; S24 is 3 bytes, little-endian and packed as in a WAV file
 * (element k at bytes 3k .. 3k+2).  Any pointer aligned to its element works (2 bytes for S16, any byte for S24).
 *   integer in  -> float: value / 2^(bits-1), exact (so a PCM input gives the same delay line as the float engine fed the
 *                  dequantised block);
 *   float out -> integer: the integer-WAV writer's rule (JUCE 6's AudioFormatWriter, as fp::formats::writeWav), in double:
 *                  y <= -1 gives INT32_MIN, y >= 1 gives INT32_MAX, NaN gives 0, otherwise lrint(2147483647.0 * y) rounding
 *                  half to even; then an arithmetic shift right by 32 - bits, which rounds toward minus infinity.  No dither.
 * An integer output block is therefore exactly what writeWav writes for the float output block.  The engine applies no gain and
 * no limiting: outputs at or beyond full scale clip to the extreme codes; to avoid clipping, scale the IR. */
typedef enum irb_sample_format { IRB_SAMPLE_F32 = 0, IRB_SAMPLE_S16 = 1, IRB_SAMPLE_S24 = 2 } irb_sample_format;

/* ---- library ------------------------------------------------------------------------------------ */
const char* irb_last_error(void);
int irb_version(void);                       /* 100 * major + minor */
int irb_device_count(void);                  /* CUDA devices visible; < 0 on failure */
int irb_set_device(int device);              /* device used by the offline functions on this thread */
int irb_max_block_size(void);                /* largest processBlockSize the block kernels take (2048) */

/* pinned host buffers for the engine's host-side entry points (plain malloc'ed memory also works, slower) */
void* irb_host_alloc(size_t bytes);
/* the same, write-combined: for buffers the host only WRITES, front to back (audio input).  The device's reads then skip the
 * CPU cache snoop, which matters when several GPUs pull from one host; reading such memory from the CPU is very slow. */
void* irb_host_alloc_write_combined(size_t bytes);
void irb_host_free(void* p);

/* ---- streaming engine -----------------------------------------------------------------------------
 * Replaces the real-time UPOLA engine inlined in IRBaboonAudioProcessor::processBlock
 * (Source/PluginProcessor.cpp:403-562; state PluginProcessor.h:194-217; setup :57-82,164-234) and its
 * fp::CircularBufferArray rings (fp/CircularBufferArray.hpp:18-64), batched over n_channels independent
 * stream-channels.  Device state per channel: a ring of max_partitions packed spectra (the frequency
 * domain delay line, FDL), its head index, and block_size overlap samples.
 */
int irb_engine_create(irb_engine** out, int device, int block_size, int max_partitions, int n_channels, int n_irs);
int irb_engine_destroy(irb_engine* e);
/* run on a caller-owned CUDA stream (cudaStream_t / CUstream; NULL is the legacy default stream);
 * IRB_OWN_STREAM restores the engine's own non-blocking stream */
#define IRB_OWN_STREAM ((void*) (~(size_t) 0))
int irb_engine_set_stream(irb_engine* e, void* cuda_stream);

/* Partition, zero-pad and transform an impulse response (fp/convolution.cpp:106-125 /
 * PluginProcessor.cpp:455-461, done for all partitions at once).  n_taps <= block_size*max_partitions.
 * right != NULL folds a stereo IR to (left+right)/2 first (tools::sumToMono, fp/tools.cpp:13-30). */
int irb_engine_set_ir(irb_engine* e, int ir_id, const float* left, const float* right, int n_taps);
/* Switch an IR the way the plug-in does (IRtoConvolve, PluginProcessor.cpp:411-414): nothing is transformed here; each
 * following block step re-transforms ONE partition of the staged taps, round-robin (:455-461), inside the step's own
 * forward-FFT launch, so the new IR replaces the old one partition by partition over `partitions` blocks.  The first
 * call for an ir_id fixes its partition count (n_partitions, or ceil(n_taps/block_size) when 0; later calls with 0
 * keep it) and, if nothing was loaded before, starts from cleared spectra as prepareToPlay does (:225-226).  Taps beyond
 * n_partitions*block_size are never read; shorter IRs are zero-extended. */
int irb_engine_stage_ir(irb_engine* e, int ir_id, const float* left, const float* right, int n_taps, int n_partitions);
/* n IRs in one call.  Row j (taps + j*ld, and right + j*ld when right != NULL, folded to (L+R)/2) holds n_taps[j] taps
 * (n_taps == NULL: ld taps each) for IR ir_ids[j].  taps/right: host memory (pageable or pinned) or device memory of the
 * engine's device, any 4-byte alignment (both of one kind).  Row j's result is exactly what irb_engine_set_ir / _stage_ir of
 * that row gives, and rows are applied in order j = 0, 1, ....  Returns when the spectra are in place (one sync of the engine's
 * stream).  Device taps are read on the engine's stream (irb_engine_set_stream): a writer on another stream orders its write
 * before the call, as for _process_device.  Host taps go through a bounded staging area (at most 64 MB per side and chunk, two
 * chunks in flight, from the workspace pool when the rows exceed the engine's own buffer), the upload of one chunk overlapping
 * the transform of the previous one.
 * One kernel (k_ir_load) per chunk transforms every partition of every row, writes every copy of the spectra, clears the ring
 * partitions past each IR's last and, for staged IRs, writes the zero-extended taps into their round-robin buffers.
 * All or nothing: every argument error is IRB_ERR_ARG, returned before any CUDA call and before anything is loaded -- a null
 * engine, ir_ids or taps; n < 1; an id outside [0, n_irs) or repeated; n_taps[j] < 1; ld < n_taps[j]; for _set_irs
 * n_taps[j] > block_size * max_partitions; for _stage_irs more partitions than max_partitions by stage_ir's rule per row.  Then
 * the pointers are classified: device memory of another device, or taps and right of different kinds, are IRB_ERR_ARG too.
 * irb_engine_set_ir / _stage_ir are the one-row calls of these. */
int irb_engine_set_irs(irb_engine* e, int n, const int* ir_ids, const float* taps, const float* right, long long ld, const int* n_taps);
int irb_engine_stage_irs(irb_engine* e, int n, const int* ir_ids, const float* taps, const float* right, long long ld, const int* n_taps,
                         int n_partitions);
/* channels [chan_begin, chan_end) convolve with ir_id.  When every kernel tile (irb_engine_tile_channels()
 * consecutive channels) is bound to one IR the tile shares the staged IR spectra; otherwise every channel stages its own
 * partitions (twice the memory traffic).  Either way a block step is one launch of the persistent kernel. */
int irb_engine_bind(irb_engine* e, int chan_begin, int chan_end, int ir_id);
int irb_engine_tile_channels(const irb_engine* e);
/* How the next block step will launch the MAC: *slots_kernel = 1 when every row stages its own IR partitions (mixed IRs in
 * a tile, or few rows), *split_in = tile slots sharing a row, *cluster = CTAs per cluster splitting the partitions further
 * (both 1 unless there are so few rows that a row's partitions are spread over the GPU). */
int irb_engine_mac_plan(irb_engine* e, int* slots_kernel, int* split_in, int* cluster);
/* Force the split (powers of two; clamped to what the tile allows; 1,1 = one CTA per tile) or return to automatic (0,0). */
int irb_engine_set_mac_split(irb_engine* e, int split_in, int cluster);
/* A block step is ONE launch: the forward transform of the new block runs in the MAC kernel's prologue (default).
 * 0 restores the two-launch form (k_fwd, then the MAC kernel) -- same results bit for bit; kept for verification. */
int irb_engine_set_fused_step(irb_engine* e, int enable);
/* Streams come and go: only channels [0, n_active) take part in the following block steps (their FDL rings advance, the
 * others keep their state); the in/out arrays of the process calls are then [n_blocks][n_active][block_size].  n_active is a
 * whole number of kernel tiles (irb_engine_tile_channels()) or n_channels (the default). */
int irb_engine_set_active_channels(irb_engine* e, int n_active);
int irb_engine_active_channels(const irb_engine* e);
/* clear FDL rings, overlap buffers and heads (prepareToPlay, PluginProcessor.cpp:164-234) */
int irb_engine_reset(irb_engine* e);

/* One UPOLA step per block for every channel: forward FFT into the FDL, MAC over all partitions,
 * inverse FFT, overlap-add.  in/out are [n_blocks][n_channels][block_size] float32.
 *   _process        : HOST buffers; copies in, runs, copies out, returns when out is complete.
 *   _process_device : DEVICE buffers on the engine's stream; asynchronous. */
int irb_engine_process(irb_engine* e, const float* in_host, float* out_host, int n_blocks);
int irb_engine_process_device(irb_engine* e, const float* in_dev, float* out_dev, int n_blocks);
/* The block order of ONE plug-in callback (PluginProcessor.cpp:421-518): all n_blocks blocks are transformed into the
 * FDL first, then convolved one after the other, each preceded by one round-robin IR refresh.  Identical to
 * _process for n_blocks == 1; for n_blocks > 1 it reproduces the reference when the host block exceeds
 * processBlockSize (its oldest partitions then meet FDL slots already overwritten by the callback's later blocks
 * unless max_partitions >= partitions + n_blocks - 1).  HOST buffers [n_blocks][n_channels][block_size]. */
int irb_engine_process_callback(irb_engine* e, const float* in_host, float* out_host, int n_blocks);
int irb_engine_synchronize(irb_engine* e);
/* Asynchronous host path for a continuous feed: _submit returns once the copies and kernels of n_blocks (>= 2) blocks are
 * enqueued -- the host arrays must be pinned (irb_host_alloc) and stay valid until _wait; consecutive submits keep the
 * upload | kernels | download pipeline full instead of draining it at every call.  _wait returns when everything
 * submitted so far is back in host memory. */
int irb_engine_submit(irb_engine* e, const float* in_host, float* out_host, int n_blocks);
int irb_engine_wait(irb_engine* e);
/* The same block steps with the input and the output in any irb_sample_format each (all nine pairs; in and out sized over the
 * input and output channels, as above, on a matrix engine too).  The formats are arguments of each call, not engine state;
 * _process, _submit and _process_device are the (F32, F32) case.  A format outside the enum gives IRB_ERR_ARG without touching
 * a device; _submit_pcm takes n_blocks >= 2 like _submit and is completed by irb_engine_wait.  Blocks of different formats may
 * follow each other on one engine.  _process_callback stays float only. */
int irb_engine_process_pcm(irb_engine* e, const void* in_host, int in_format, void* out_host, int out_format, int n_blocks);
int irb_engine_submit_pcm(irb_engine* e, const void* in_host, int in_format, void* out_host, int out_format, int n_blocks);
int irb_engine_process_device_pcm(irb_engine* e, const void* in_dev, int in_format, void* out_dev, int out_format, int n_blocks);

/* Per-step device timing with CUDA events on the engine's stream: whole block step (k_fwd + k_mac) and the
 * FDL-MAC kernel alone (on a one-launch block step the two are the same pair of events: no event is recorded in between).
 * set_timing(1) clears the record; get_timings returns the number of steps copied. */
int irb_engine_set_timing(irb_engine* e, int enable);
int irb_engine_get_timings(irb_engine* e, float* step_ms, float* mac_ms, int max_steps);

/* introspection (tests, benchmarks) */
size_t irb_engine_state_bytes(const irb_engine* e);            /* device bytes held */
int irb_engine_fft_size(const irb_engine* e);                  /* N = 2M actually used */
int irb_engine_partitions(const irb_engine* e, int ir_id);     /* partitions of a loaded IR */
/* copy one packed spectrum (M complex: bin 0 = {Re X[0], Re X[N/2]}) to the host:
 * the IR partition `part` of ir_id, or the FDL slot `age` blocks old (0 = newest) of a channel */
int irb_engine_read_ir_spectrum(irb_engine* e, int ir_id, int part, float* out_packed);
int irb_engine_read_fdl_spectrum(irb_engine* e, int chan, int age, float* out_packed);
/* kernel launches issued by this engine so far, and by the whole library */
long long irb_engine_launch_count(const irb_engine* e);
long long irb_launch_count(void);
/* The offline functions recycle their device scratch buffers through a process-wide pool (at most 12 GB of free blocks) so
 * that repeated calls do not pay cudaMalloc / cudaFree of gigabytes each time; this returns the pool to the driver and
 * reports how many bytes it held.  Engines do not use the pool. */
size_t irb_release_workspace(void);
/* device time (CUDA events, ms) of the kernels of the calling thread's most recent offline call
 * (irb_convolve_periodic / _nonperiodic / irb_deconvolve*), host<->device copies excluded */
double irb_last_compute_ms(void);
/* ---- IR matrix engine ---------------------------------------------------------------------------------
 * n_groups groups of `ins` consecutive input channels, each producing `outs` consecutive output channels:
 *   out[g*outs + o] = sum_i conv(in[g*ins + i], IR ir_ids[i*outs + o])
 * Supported (ins, outs): (1, 2) mono -> stereo, (2, 2) true stereo (IRs LL, LR, RL, RR).  Block sizes whose FFT half size is
 * 256..1024 (129 <= block_size <= 1024).  Each input channel keeps ONE FDL ring (advanced once per block, read once per block
 * step for all the IRs it feeds); each output channel keeps its overlap.  n_irs >= ins*outs; until bound, every group uses
 * ir_ids = {0, 1, ..., ins*outs-1}.  For (1, 2) output o is bit-identical to a plain engine channel bound to ir_ids[o].
 * in: [n_blocks][n_groups*ins][block_size], out: [n_blocks][n_groups*outs][block_size].
 * The other irb_engine_* calls keep their meaning on a matrix engine (read_fdl_spectrum: `chan` is an input channel;
 * mac_plan: slots_kernel = 1 when some kernel unit mixes matrices and every group stages its own IR partitions), except
 * irb_engine_bind, _process_callback, _set_active_channels, _set_mac_split and _set_fused_step(0): IRB_ERR_STATE. */
int irb_engine_create_matrix(irb_engine** out, int device, int block_size, int max_partitions, int n_groups, int ins, int outs, int n_irs);
int irb_engine_bind_matrix(irb_engine* e, int group_begin, int group_end, const int* ir_ids /* [ins*outs] */);

/* ---- several GPUs from one process ---------------------------------------------------------------------
 * Streams never interact (fp/convolution.cpp:160-215 has no cross-channel term), so n_channels are cut into contiguous
 * ranges of whole kernel tiles, one irb_engine per device.  n_irs > 0: shared IRs, replicated on every device, bound with
 * irb_group_bind.  n_irs == 0: every channel owns an IR that lives on the channel's device; ir_id then means the channel.
 * No device-to-device traffic and no collective: each device reads its channel range of the caller's
 * [n_blocks][n_channels][block_size] arrays and writes its range of the output (the "host-side gather").  One host thread
 * feeds all devices: every device's copies and kernels are enqueued before the first is waited for. */
typedef struct irb_group irb_group;
int irb_group_create(irb_group** out, const int* devices, int n_devices, int block_size, int max_partitions, int n_channels, int n_irs);
int irb_group_destroy(irb_group* g);
int irb_group_device_count(const irb_group* g);
int irb_group_channel_range(const irb_group* g, int index, int* begin, int* end);
int irb_group_set_ir(irb_group* g, int ir_id, const float* left, const float* right, int n_taps);
int irb_group_stage_ir(irb_group* g, int ir_id, const float* left, const float* right, int n_taps, int n_partitions);
/* host memory only; private-IR groups (n_irs == 0) send each row to the device that owns channel ir_ids[j], shared-IR groups
 * send every row to every device; every device's copies and kernels are enqueued before the first wait (as irb_group_process).
 * Arguments as irb_engine_set_irs / _stage_irs; device memory is IRB_ERR_ARG.  irb_group_set_ir / _stage_ir are their one-row calls. */
int irb_group_set_irs(irb_group* g, int n, const int* ir_ids, const float* taps, const float* right, long long ld, const int* n_taps);
int irb_group_stage_irs(irb_group* g, int n, const int* ir_ids, const float* taps, const float* right, long long ld, const int* n_taps,
                        int n_partitions);
int irb_group_bind(irb_group* g, int chan_begin, int chan_end, int ir_id);
int irb_group_reset(irb_group* g);
int irb_group_process(irb_group* g, const float* in_host, float* out_host, int n_blocks);
/* irb_group_process with the input and output in any irb_sample_format (see irb_engine_process_pcm) */
int irb_group_process_pcm(irb_group* g, const void* in_host, int in_format, void* out_host, int out_format, int n_blocks);
size_t irb_group_state_bytes(const irb_group* g);

/* ---- offline functions ------------------------------------------------------------------------------
 * fp::convolution::convolvePeriodic (fp/convolution.hpp:31, fp/convolution.cpp:14-242): planar
 * x[ch_x][len_x], h[ch_h][len_h] -> out[ch_x][len_x+len_h-1].  Same channel layouts (mono/stereo x
 * mono/stereo), partition count, iteration count and unflushed tail as the reference.  Any block_size >= 1: sizes above
 * irb_max_block_size() are computed with the largest block the kernels take and cut at the reference's output length. */
int irb_convolve_periodic(const float* x, int ch_x, int len_x, const float* h, int ch_h, int len_h, int block_size, float* out);


/* fp::convolution::convolveNonPeriodic (fp/convolution.hpp:32, fp/convolution.cpp:246-347): one real FFT of
 * N = pow2 >= len_x+len_h-1 per signal, per-bin product, inverse; out[ch_x][len_x+len_h-1].  IRB_ERR_LAYOUT for the
 * layouts the reference rejects (it returns a cleared copy of the input there, :271-275). */
int irb_convolve_nonperiodic(const float* x, int ch_x, int len_x, const float* h, int ch_h, int len_h, float* out);

/* `batch` signals x[batch][len_x], each linearly convolved with an IR h[h_batch][len_h], h_batch = 1 (one IR shared by every
 * signal) or batch (signal b with IR b).  N = nextPowerOfTwo(len_x + len_h - 1), at least 16, at most 2^22, as irb_convolve_nonperiodic.
 * Only the window [out_offset, out_offset + out_len) of each full result is written: out[batch][out_len].
 * Requires 0 <= out_offset and out_offset + out_len <= len_x + len_h - 1.
 * With out_offset = 0 and out_len = len_x + len_h - 1, row b is bit-identical to irb_convolve_nonperiodic(x[b], 1, len_x, h[b or 0], 1, len_h).
 * Every argument error (null pointer, batch < 1, h_batch not 1 or batch, an empty signal, out_len < 1, a window outside the
 * result, a result above 2^22 points) is IRB_ERR_ARG, returned before any CUDA call.  The batch runs in sub-batches with uploads,
 * kernels and downloads overlapped; only the window's samples are written to device memory and copied back. */
int irb_convolve_batch(const float* x, int batch, int len_x, const float* h, int h_batch, int len_h, int out_offset, int out_len, float* out);
/* The same on DEVICE-resident x_dev and out_dev.  h may be in host or device memory, as `den` of irb_deconvolve_batch_device.
 * No staging copies when N > 4096, x_dev is 8-byte aligned and len_x even, and a per-signal h (h_batch = batch) is device memory,
 * 8-byte aligned, with len_h even; any other float alignment is accepted and goes through staged device-to-device copies. */
int irb_convolve_batch_device(const float* x_dev, int batch, int len_x, const float* h, int h_batch, int len_h, int out_offset, int out_len, float* out_dev);

/* fp::convolution::deconvolve (fp/convolution.hpp:38, fp/convolution.cpp:351-403): spectral division
 * FFT(num)/FFT(den) at N = nextPowerOfTwo(max(len_num, len_den)) (circular), optional 3x 1/13-octave
 * averagingFilter, inverse FFT, ir::shifteroo when the phase is dropped.  out[N] (or [batch][N]).
 * _batch divides `batch` numerators [batch][len_num] by one denominator: the batched ESS IR capture. */
int irb_deconvolve(const float* num, int len_num, const float* den, int len_den, double sample_rate, int smoothing, int include_phase, int include_amplitude,
                   float* out);
int irb_deconvolve_batch(const float* nums, int batch, int len_num, const float* den, int len_den, double sample_rate, int smoothing, int include_phase,
                         int include_amplitude, float* out);
/* _batch with DEVICE-resident captures nums_dev[batch][len_num] and results out_dev[batch][N] (den: host or device memory):
 * the batched capture when the recordings already live in HBM.  No staging copies for large plain divisions (no smoothing,
 * phase kept, even len_num) when nums_dev and out_dev are both 8-byte aligned; any other alignment of a float pointer is
 * accepted too, and goes through staged device-to-device copies. */
int irb_deconvolve_batch_device(const float* nums_dev, int batch, int len_num, const float* den, int len_den, double sample_rate, int smoothing,
                                int include_phase, int include_amplitude, float* out_dev);
/* fp::ir::IRchop followed, when `normalize`, by fp::tools::normalize(goal_db) on each row x[0, len) of x_dev[batch][len]
 * (device memory) -> out_dev[batch][ir_length] (device memory); positions (null, or device memory) [batch][2] = {q, start}:
 * the peak's index (the system delay of a capture) and the first sample of the cut.  The rule, the facade's (fp_b200.cpp):
 *   peak = max |x_i| accumulated as std::max(m, fabs(x_i)) from m = 0 (NaN samples are ignored, an Inf makes the peak Inf);
 *   q = the first index with fabs(x_q) == peak, 0 when there is none (every sample NaN);
 *   below(i) := linTodB(fabs(x_i)) - linTodB(peak) < threshold_db in float, linTodB(v) = v == 0 ? -333 : 20 * ln(v) / ln(10)
 *   evaluated left to right in float, ln(v) = (float) log((double) v) (the correctly rounded float log; see below);
 *   walked = 0 when consecutive <= 0, else the smallest k >= consecutive such that below(s_{k-consecutive}) .. below(s_{k-1})
 *   all hold, s_j = (q - j) mod len, capped at ir_length; start = (q - walked) mod len;
 *   out = the ir_length samples from start (wrapping past len - 1 to 0); samples [ir_length-1-ir_length/4, ir_length-1) times
 *   (float) (1.0 - (double) (float(i') * step)) (the last sample is not faded, as in the reference), then samples [0, walked/4)
 *   times float(i') * step; i' is the offset in the fade, step = (float) (1.0 / fade length) (tools::linearFade);
 *   normalize: every sample times goal / max|out|, goal = dBToLin(goal_db) in float (a silent row gives NaN, as the facade).
 * The log: glibc's logf is not correctly rounded (on about 417 000 of the 2^31 positive floats it differs from the correctly
 * rounded result; linTodB then differs on about 326 000), and the device's own logf has a different error set, so the device
 * uses the correctly rounded float log, computed as log((double) v) rounded to float (with glibc's double log that formula is the
 * nearest float to ln(v) on every positive float except five hard cases, 0x3c413d3a, 0x41178feb, 0x4c5d65a5, 0x65d890d3 and
 * 0x6f31a8ec).  A row's cut can therefore differ from the host facade's only when the level of one of its walked samples, or of
 * its peak, is one of those inputs AND that 1-ulp difference flips a threshold decision.  Everything else (the peak, the cut,
 * the fades, the gain) is the facade's arithmetic bit for bit (NaN samples stay NaN; the payload is the device's).
 * IRB_ERR_ARG before any CUDA call: a null x_dev or out_dev, batch < 1, len < 1, ir_length < 1 or > len.  Any 4-byte aligned
 * pointers; irb_last_compute_ms() is the device time of the call. */
int irb_ir_chop_batch_device(const float* x_dev, int batch, int len, int ir_length, float threshold_db, int consecutive, int normalize, float goal_db,
                             float* out_dev, int* positions);
/* irb_deconvolve_batch followed by the chop above, inside the sub-batch pipeline: host (or pinned) nums in, out[batch][ir_length]
 * and positions (null, or host memory [batch][2]) back; the [batch][N] results never leave the device.  Row b is bit-identical to
 * irb_deconvolve_batch's row b chopped by irb_ir_chop_batch_device.  IRB_ERR_ARG before any CUDA call for the division's own
 * rejections and ir_length < 1 or > N.  irb_last_compute_ms() covers the chop as part of the kernel sections. */
int irb_deconvolve_chop_batch(const float* nums, int batch, int len_num, const float* den, int len_den, double sample_rate, int smoothing, int include_phase,
                              int include_amplitude, int ir_length, float threshold_db, int consecutive, int normalize, float goal_db, float* out, int* positions);
/* fp::ir::invertFilter (fp/ir.hpp:20, fp/ir.cpp:13-18); out[nextPowerOfTwo(len)] */
int irb_invert_filter(const float* x, int len, int sample_rate, float* out);
/* fp::convolution::averagingFilter (fp/convolution.hpp:44, fp/convolution.cpp:406-546), in place on an interleaved
 * spectrum spec[ch][fft_size]; a fft_size that is not a power of two leaves it untouched (:412-415).  The last two
 * flags are INCLUDE flags, as the reference's body treats them. */
int irb_averaging_filter(float* spec, int ch, int fft_size, double octave_fraction, double sample_rate, int log_avg, int include_phase, int include_amplitude);
/* fp::tools::fftTransform / fftInvTransform (fp/tools.hpp:88-89, fp/tools.cpp:321-369) */
int irb_fft_transform(const float* x, int ch, int len, int format_ampl_phase, float* out /* [ch][2N] */);
int irb_fft_inv_transform(const float* spec, int ch, int fft_size, float* out /* [ch][fft_size/2] */);
/* fp::ir::IRtoRealFFTRaw (fp/ir.hpp:36, fp/ir.cpp:106-147): partitioned packed spectra of an IR, the engine's own
 * FDL/IR wire format; out[(len/part_size + 1) * 2*part_size] */
int irb_ir_to_real_fft_raw(const float* x, int len, int part_size, float* out);
/* fp::ExpSineSweep::generate / generateInv (fp/ExpSineSweep.hpp:27-33, fp/ExpSineSweep.cpp:26-41,59-79), FP64.
 * Returns the sweep length (int)(sample_rate*duration); out == NULL only queries it. */
int irb_ess_generate(double duration_s, double sample_rate, double f1, double f2, double gain_db, int inverse, double* out, int capacity);

#ifdef __cplusplus
}
#endif
#endif /* IRB_B200_H */
