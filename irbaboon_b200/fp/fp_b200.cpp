// fp_b200.cpp -- implementation of the fp:: facade over the C ABI (include/irb_b200.h).
// Host code only marshals buffers; every transform / multiply-accumulate runs in libirb_b200.so on the GPU.
// A failing CUDA call throws std::runtime_error: there is no host fallback to hide behind.
#include <cmath>
#include <cstdlib>
#include <stdexcept>
#include <string>

#include "../../include/irb_b200.h"
#include "CircularBufferArray.hpp"
#include "PluginConvolver.hpp"
#include "StreamingConvolver.hpp"
#include "convolution.hpp"
#include "tools.hpp"

namespace {

[[noreturn]] void raise(const char* what) {
    throw std::runtime_error(std::string(what) + ": " + irb_last_error());
}

// planar AudioBuffer -> one dense [channels][samples] array (JUCE channels need not be adjacent in memory)
std::vector<float> pack(const AudioBuffer<float>& b) {
    const int ch = b.getNumChannels(), n = b.getNumSamples();
    std::vector<float> v((size_t) ch * (size_t) n);
    for (int c = 0; c < ch; ++c) std::copy_n(b.getReadPointer(c), n, v.begin() + (size_t) c * n);
    return v;
}

// the channels of an IR file as the rows [channels][ld] of irb_*_set_irs: in place when they are evenly spaced, else packed
struct IrRows {
    std::vector<float> packed;
    std::vector<int> ids, taps;
    const float* data = nullptr;
    long long ld = 0;
    IrRows(const AudioBuffer<float>& b, int firstId) {
        const int ch = b.getNumChannels(), n = b.getNumSamples();
        for (int c = 0; c < ch; ++c) { ids.push_back(firstId + c); taps.push_back(n); }
        data = b.getReadPointer(0);
        ld = ch > 1 ? (long long) (b.getReadPointer(1) - data) : n;
        bool even = ld >= n;
        for (int c = 2; c < ch && even; ++c) even = b.getReadPointer(c) - b.getReadPointer(c - 1) == ld;
        if (!even) { packed = pack(b); data = packed.data(); ld = n; }
    }
};

}  // namespace

namespace fp {

// ---- convolution ---------------------------------------------------------------------------------
AudioBuffer<float> convolution::convolvePeriodic(AudioBuffer<float>& buffer1, AudioBuffer<float>& buffer2, int processBlockSize) {
    const int chx = buffer1.getNumChannels(), lx = buffer1.getNumSamples();
    const int chh = buffer2.getNumChannels(), lh = buffer2.getNumSamples();
    AudioBuffer<float> out(chx, lx + lh - 1);
    out.clear();
    if (out.getNumSamples() <= 0 || chx <= 0) return out;
    std::vector<float> x = pack(buffer1), h = pack(buffer2), y((size_t) chx * out.getNumSamples());
    const int rc = irb_convolve_periodic(x.data(), chx, lx, h.data(), chh, lh, processBlockSize, y.data());
    if (rc == IRB_ERR_LAYOUT) {
        DBG("Either buffer1 or buffer2 is not mono nor stereo. Abort abort \n");
        return out;
    }
    if (rc != IRB_OK) raise("fp::convolution::convolvePeriodic");
    for (int c = 0; c < chx; ++c) out.copyFrom(c, 0, y.data() + (size_t) c * out.getNumSamples(), out.getNumSamples());
    return out;
}

// ---- CircularBufferArray (fp/CircularBufferArray.cpp:12-205) ---------------------------------------
CircularBufferArray::CircularBufferArray() {}
CircularBufferArray::CircularBufferArray(int amountOfBuffers, int bufferChannelSize, int bufferSampleSize) {
    initBuffers(amountOfBuffers, bufferChannelSize, bufferSampleSize);
}
CircularBufferArray::~CircularBufferArray() {}

void CircularBufferArray::initBuffers(int amountOfBuffers, int bufferChannelSize, int bufferSampleSize) {
    channelsPerBuffer = bufferChannelSize;
    samplesPerBuffer = bufferSampleSize;
    arraySize = amountOfBuffers;
    readIndex = writeIndex = 0;
    bufferArray.assign((size_t) std::max(0, amountOfBuffers), AudioBuffer<float>());
    for (auto& b : bufferArray) { b.setSize(bufferChannelSize, bufferSampleSize); b.clear(); }
}
void CircularBufferArray::clearAndResize(int amountOfBuffers, int bufferChannelSize, int bufferSampleSize) {
    initBuffers(amountOfBuffers, bufferChannelSize, bufferSampleSize);
}
void CircularBufferArray::changeArraySize(int amountOfBuffers) {
    if (amountOfBuffers == arraySize) return;
    if (amountOfBuffers == 0) {
        bufferArray.clear();
        readIndex = writeIndex = arraySize = 0;
        return;
    }
    if (amountOfBuffers > arraySize) {
        const int extra = amountOfBuffers - arraySize;
        for (int i = 0; i < extra; ++i) {
            AudioBuffer<float> b(channelsPerBuffer, samplesPerBuffer);
            b.clear();
            bufferArray.push_back(b);
            // the reference clears slot i here -- an OLD front slot, not the new one (CircularBufferArray.cpp:49-52);
            // observable, so kept
            if (i < (int) bufferArray.size()) bufferArray[(size_t) i].clear();
        }
        arraySize = (int) bufferArray.size();
        return;
    }
    // shrinking
    if (lastWrittenIndex == -1) {          // never written: plain truncation
        bufferArray.resize((size_t) amountOfBuffers);
        return;                            // (arraySize is left untouched by the reference on this path, :84-86)
    }
    const int readBack = lastWrittenIndex - readIndex, writeBack = lastWrittenIndex - writeIndex;
    std::vector<AudioBuffer<float>> kept((size_t) amountOfBuffers);
    int src = lastWrittenIndex;
    for (int i = amountOfBuffers - 1; i >= 0; --i) {      // newest ends up last
        kept[(size_t) i] = bufferArray[(size_t) src];
        src = src == 0 ? arraySize - 1 : src - 1;
    }
    bufferArray.swap(kept);
    arraySize = amountOfBuffers;
    const int last = arraySize - 1;
    auto remap = [&](int back) { return back > last ? 0 : (back < 0 ? last - (arraySize + back) : last - back); };
    readIndex = remap(readBack);
    writeIndex = remap(writeBack);
}
AudioBuffer<float>* CircularBufferArray::getReadBufferPtr() { return &bufferArray[(size_t) readIndex]; }
AudioBuffer<float>* CircularBufferArray::getWriteBufferPtr() { lastWrittenIndex = writeIndex; return &bufferArray[(size_t) writeIndex]; }
AudioBuffer<float>* CircularBufferArray::getBufferPtrAtIndex(int index) { return &bufferArray[(size_t) index]; }
void CircularBufferArray::incrReadIndex() { if (++readIndex >= arraySize) readIndex = 0; }
void CircularBufferArray::decrReadIndex() { if (--readIndex < 0) readIndex = arraySize - 1; }
void CircularBufferArray::incrWriteIndex() { if (++writeIndex >= arraySize) writeIndex = 0; }
AudioBuffer<float> CircularBufferArray::consolidate(int bufOffset) {
    AudioBuffer<float> all(channelsPerBuffer, samplesPerBuffer * arraySize);
    int start = bufOffset < 0 ? arraySize - 1 - std::abs(bufOffset) : bufOffset;
    for (int k = 0; k < arraySize; ++k) {
        const int slot = (start + k) % std::max(1, arraySize);
        for (int c = 0; c < channelsPerBuffer; ++c)
            all.copyFrom(c, k * samplesPerBuffer, bufferArray[(size_t) slot], c, 0, samplesPerBuffer);
    }
    return all;
}
int CircularBufferArray::getReadIndex() { return readIndex; }
void CircularBufferArray::setReadIndex(int index) { readIndex = index; }
int CircularBufferArray::getWriteIndex() { return writeIndex; }
void CircularBufferArray::setWriteIndex(int index) { writeIndex = index; }
int CircularBufferArray::getArraySize() { return arraySize; }
int CircularBufferArray::getChannelsPerBuffer() { return channelsPerBuffer; }
int CircularBufferArray::getSamplesPerBuffer() { return samplesPerBuffer; }

// ---- StreamingConvolver ----------------------------------------------------------------------------
namespace b200 {

StreamingConvolver::StreamingConvolver(int blockSize_, int maxPartitions, int channels_, int numIRs, int device)
    : blockSize(blockSize_), channels(channels_) {
    if (irb_engine_create(&engine, device, blockSize, maxPartitions, channels, numIRs) != IRB_OK) raise("irb_engine_create");
    stageIn.resize((size_t) blockSize * channels);
    stageOut.resize((size_t) blockSize * channels);
}
StreamingConvolver::~StreamingConvolver() { irb_engine_destroy(engine); }
void StreamingConvolver::setIR(int irId, const AudioBuffer<float>& ir, bool foldStereo) {
    const float* r = (foldStereo && ir.getNumChannels() == 2) ? ir.getReadPointer(1) : nullptr;
    if (irb_engine_set_ir(engine, irId, ir.getReadPointer(0), r, ir.getNumSamples()) != IRB_OK) raise("irb_engine_set_ir");
}
void StreamingConvolver::setIRs(int firstId, const AudioBuffer<float>& irs) {
    const IrRows r(irs, firstId);
    if (irb_engine_set_irs(engine, (int) r.ids.size(), r.ids.data(), r.data, nullptr, r.ld, r.taps.data()) != IRB_OK) raise("irb_engine_set_irs");
}
void StreamingConvolver::bind(int channelBegin, int channelEnd, int irId) {
    if (irb_engine_bind(engine, channelBegin, channelEnd, irId) != IRB_OK) raise("irb_engine_bind");
}
void StreamingConvolver::reset() {
    if (irb_engine_reset(engine) != IRB_OK) raise("irb_engine_reset");
}
void StreamingConvolver::processBlock(AudioBuffer<float>& buffer) {
    if (buffer.getNumChannels() != channels || buffer.getNumSamples() != blockSize)
        throw std::invalid_argument("StreamingConvolver::processBlock: buffer must be channels x blockSize");
    for (int c = 0; c < channels; ++c) std::copy_n(buffer.getReadPointer(c), blockSize, stageIn.begin() + (size_t) c * blockSize);
    if (irb_engine_process(engine, stageIn.data(), stageOut.data(), 1) != IRB_OK) raise("irb_engine_process");
    for (int c = 0; c < channels; ++c) buffer.copyFrom(c, 0, stageOut.data() + (size_t) c * blockSize, blockSize);
}
void StreamingConvolver::process(const float* in, float* out, int nBlocks) {
    if (irb_engine_process(engine, in, out, nBlocks) != IRB_OK) raise("irb_engine_process");
}
void StreamingConvolver::process(const void* in, irb_sample_format inFormat, void* out, irb_sample_format outFormat, int nBlocks) {
    if (irb_engine_process_pcm(engine, in, inFormat, out, outFormat, nBlocks) != IRB_OK) raise("irb_engine_process_pcm");
}

// ---- MatrixConvolver ------------------------------------------------------------------------------------
MatrixConvolver::MatrixConvolver(int blockSize_, int maxPartitions, int groups_, int ins_, int outs_, int numIRs, int device)
    : blockSize(blockSize_), groups(groups_), ins(ins_), outs(outs_) {
    if (irb_engine_create_matrix(&engine, device, blockSize, maxPartitions, groups, ins, outs, numIRs > 0 ? numIRs : ins * outs) != IRB_OK)
        raise("irb_engine_create_matrix");
    stageIn.resize((size_t) blockSize * groups * ins);
    stageOut.resize((size_t) blockSize * groups * outs);
}
MatrixConvolver::~MatrixConvolver() { irb_engine_destroy(engine); }
void MatrixConvolver::setIR(int irId, const AudioBuffer<float>& ir) {
    const int ch = ir.getNumChannels();
    if (ch != 1 && ch != ins * outs)
        throw std::invalid_argument("MatrixConvolver::setIR: an IR file has 1 channel or one per IR of the matrix (" + std::to_string(ins * outs) + ")");
    const IrRows r(ir, irId);
    if (irb_engine_set_irs(engine, ch, r.ids.data(), r.data, nullptr, r.ld, r.taps.data()) != IRB_OK) raise("irb_engine_set_irs");
}
void MatrixConvolver::bindMatrix(int groupBegin, int groupEnd, const std::vector<int>& irIds) {
    if ((int) irIds.size() != ins * outs) throw std::invalid_argument("MatrixConvolver::bindMatrix: one IR id per input and output (ins*outs)");
    if (irb_engine_bind_matrix(engine, groupBegin, groupEnd, irIds.data()) != IRB_OK) raise("irb_engine_bind_matrix");
}
void MatrixConvolver::reset() {
    if (irb_engine_reset(engine) != IRB_OK) raise("irb_engine_reset");
}
void MatrixConvolver::processBlock(const AudioBuffer<float>& in, AudioBuffer<float>& out) {
    if (in.getNumChannels() != groups * ins || in.getNumSamples() != blockSize || out.getNumChannels() != groups * outs || out.getNumSamples() != blockSize)
        throw std::invalid_argument("MatrixConvolver::processBlock: in must be groups*ins x blockSize, out groups*outs x blockSize");
    for (int c = 0; c < groups * ins; ++c) std::copy_n(in.getReadPointer(c), blockSize, stageIn.begin() + (size_t) c * blockSize);
    if (irb_engine_process(engine, stageIn.data(), stageOut.data(), 1) != IRB_OK) raise("irb_engine_process");
    for (int c = 0; c < groups * outs; ++c) out.copyFrom(c, 0, stageOut.data() + (size_t) c * blockSize, blockSize);
}
void MatrixConvolver::process(const float* in, float* out, int nBlocks) {
    if (irb_engine_process(engine, in, out, nBlocks) != IRB_OK) raise("irb_engine_process");
}
void MatrixConvolver::process(const void* in, irb_sample_format inFormat, void* out, irb_sample_format outFormat, int nBlocks) {
    if (irb_engine_process_pcm(engine, in, inFormat, out, outFormat, nBlocks) != IRB_OK) raise("irb_engine_process_pcm");
}

// ---- MultiGpuConvolver ----------------------------------------------------------------------------------
MultiGpuConvolver::MultiGpuConvolver(const std::vector<int>& devices, int blockSize, int maxPartitions, int channels, int numIRs) {
    if (irb_group_create(&group, devices.data(), (int) devices.size(), blockSize, maxPartitions, channels, numIRs) != IRB_OK) raise("irb_group_create");
}
MultiGpuConvolver::~MultiGpuConvolver() { irb_group_destroy(group); }
void MultiGpuConvolver::setIR(int irId, const AudioBuffer<float>& ir, bool foldStereo) {
    const float* r = (foldStereo && ir.getNumChannels() == 2) ? ir.getReadPointer(1) : nullptr;
    if (irb_group_set_ir(group, irId, ir.getReadPointer(0), r, ir.getNumSamples()) != IRB_OK) raise("irb_group_set_ir");
}
void MultiGpuConvolver::setIRs(int firstId, const AudioBuffer<float>& irs) {
    const IrRows r(irs, firstId);
    if (irb_group_set_irs(group, (int) r.ids.size(), r.ids.data(), r.data, nullptr, r.ld, r.taps.data()) != IRB_OK) raise("irb_group_set_irs");
}
void MultiGpuConvolver::bind(int channelBegin, int channelEnd, int irId) {
    if (irb_group_bind(group, channelBegin, channelEnd, irId) != IRB_OK) raise("irb_group_bind");
}
void MultiGpuConvolver::reset() {
    if (irb_group_reset(group) != IRB_OK) raise("irb_group_reset");
}
void MultiGpuConvolver::process(const float* in, float* out, int nBlocks) {
    if (irb_group_process(group, in, out, nBlocks) != IRB_OK) raise("irb_group_process");
}
void MultiGpuConvolver::process(const void* in, irb_sample_format inFormat, void* out, irb_sample_format outFormat, int nBlocks) {
    if (irb_group_process_pcm(group, in, inFormat, out, outFormat, nBlocks) != IRB_OK) raise("irb_group_process_pcm");
}

// ---- PluginConvolver ------------------------------------------------------------------------------------
PluginConvolver::PluginConvolver(int processBlockSize, int channels_, int device_) : B(processBlockSize), channels(channels_), device(device_) {
    latency = B;                                                                      // PluginProcessor.cpp:59
}
PluginConvolver::~PluginConvolver() { destroyEngine(); }
void PluginConvolver::destroyEngine() {
    if (engine) irb_engine_destroy(engine);
    engine = nullptr;
}
void PluginConvolver::prepareToPlay(double, int samplesPerBlock, const AudioBuffer<float>& ir) {
    if (samplesPerBlock < 1 || ir.getNumSamples() < 1 || ir.getNumChannels() < 1) throw std::invalid_argument("PluginConvolver::prepareToPlay: empty host block or IR");
    hostBlock = samplesPerBlock;
    latency = hostBlock > B ? hostBlock : B;                                          // :166-171
    inArray = (int) std::ceil((float) hostBlock / (float) B);                         // :203
    outArray = tools::nextPowerOfTwo((int) (std::ceil((float) B / (float) hostBlock) + 1));   // :205
    partitions = (int) std::ceil((float) ir.getNumSamples() / (float) B);             // :225
    // FDL ring: the reference's max(partitions, inArray) slots (:229-230), or room for every spectrum a callback needs
    const int ring = exactOrder ? std::max(partitions, inArray) : partitions + inArray - 1;
    destroyEngine();
    if (irb_set_device(device) != IRB_OK) raise("irb_set_device");
    if (irb_engine_create(&engine, device, B, ring, channels, 1) != IRB_OK) raise("irb_engine_create");
    if (irb_engine_stage_ir(engine, 0, ir.getReadPointer(0), nullptr, ir.getNumSamples(), partitions) != IRB_OK) raise("irb_engine_stage_ir");
    inBlocks.assign((size_t) (inArray + 1) * channels * B, 0.0f);        // + the block still being collected
    outBlocks.assign((size_t) (inArray + 1) * channels * B, 0.0f);
    outRing.assign((size_t) outArray * channels * hostBlock, 0.0f);
    bypassRing.assign((size_t) outArray * channels * hostBlock, 0.0f);
    inSample = 0; blocksToProcess = 0;
    outWrite = 0; outRead = 1; outWriteSample = 0; outReadSample = 0;                 // :218
    bypassWrite = 0; bypassRead = 0;
}
void PluginConvolver::setIR(const AudioBuffer<float>& ir) {
    if (!engine) throw std::logic_error("PluginConvolver::setIR before prepareToPlay");
    if (irb_engine_stage_ir(engine, 0, ir.getReadPointer(0), nullptr, ir.getNumSamples(), 0) != IRB_OK) raise("irb_engine_stage_ir");
}
void PluginConvolver::processBlock(AudioBuffer<float>& buffer) {
    if (!engine) throw std::logic_error("PluginConvolver::processBlock before prepareToPlay");
    const int n = buffer.getNumSamples();
    if (n == 0) return;                                                               // :279-281
    if (buffer.getNumChannels() < channels || n > hostBlock) throw std::invalid_argument("PluginConvolver::processBlock: buffer smaller than the channel count or longer than samplesPerBlock");
    // collect samples into processBlockSize blocks (:421-445); a callback completes at most inArray of them
    for (int s = 0; s < n; ++s) {
        for (int c = 0; c < channels; ++c) inBlocks[((size_t) blocksToProcess * channels + c) * B + inSample] = buffer.getSample(c, s);
        if (++inSample >= B) { inSample = 0; ++blocksToProcess; }
    }
    if (blocksToProcess > 0) {
        // forward FFTs of all completed blocks, then per block: IR refresh, MAC, inverse FFT, overlap-add (:452-518) -- on the GPU
        if (irb_engine_process_callback(engine, inBlocks.data(), outBlocks.data(), blocksToProcess) != IRB_OK) raise("irb_engine_process_callback");
        // the samples of a block still being collected sit at the front of the next callback's first block
        if (inSample > 0)
            for (int c = 0; c < channels; ++c)
                std::copy_n(&inBlocks[((size_t) blocksToProcess * channels + c) * B], inSample, &inBlocks[(size_t) c * B]);
        // completed blocks -> host-sized output buffers (:525-545); a buffer is cleared when its first sample is written
        for (int b = 0; b < blocksToProcess; ++b) {
            for (int s = 0; s < B; ++s) {
                float* ob = &outRing[(size_t) outWrite * channels * hostBlock];
                if (outWriteSample == 0) std::fill_n(ob, (size_t) channels * hostBlock, 0.0f);
                for (int c = 0; c < channels; ++c) ob[(size_t) c * hostBlock + outWriteSample] = outBlocks[((size_t) b * channels + c) * B + s];
                if (++outWriteSample >= hostBlock) { outWriteSample = 0; if (++outWrite >= outArray) outWrite = 0; }
            }
        }
        blocksToProcess = 0;
    }
    // output buffers -> the host's buffer (:552-560)
    for (int s = 0; s < n; ++s) {
        const float* ob = &outRing[(size_t) outRead * channels * hostBlock];
        for (int c = 0; c < channels; ++c) buffer.setSample(c, s, ob[(size_t) c * hostBlock + outReadSample]);
        if (++outReadSample >= hostBlock) { outReadSample = 0; if (++outRead >= outArray) outRead = 0; }
    }
    // standard attenuation, then the limiter: normalise to 0 dB when channel 0 peaks above it (:567-574)
    buffer.applyGain(tools::dBToLin(outputVolumedB));
    if (tools::linTodB(buffer.getMagnitude(0, 0, std::min(hostBlock, n))) > 0.0) tools::normalize(&buffer, 0.0f, false);
}
void PluginConvolver::processBlockBypassed(AudioBuffer<float>& buffer) {
    if (!engine) throw std::logic_error("PluginConvolver::processBlockBypassed before prepareToPlay");
    const int n = std::min(buffer.getNumSamples(), hostBlock);
    float* wb = &bypassRing[(size_t) bypassWrite * channels * hostBlock];
    for (int c = 0; c < channels; ++c) { std::fill_n(wb + (size_t) c * hostBlock, hostBlock, 0.0f); std::copy_n(buffer.getReadPointer(c), n, wb + (size_t) c * hostBlock); }
    if (++bypassWrite >= outArray) bypassWrite = 0;
    if (++bypassRead >= outArray) bypassRead = 0;
    const float* rb = &bypassRing[(size_t) bypassRead * channels * hostBlock];
    for (int c = 0; c < channels; ++c) buffer.copyFrom(c, 0, rb + (size_t) c * hostBlock, n);
}

}  // namespace b200
}  // namespace fp

// =====================================================================================================
// tools / ir / ExpSineSweep / remaining convolution functions
// =====================================================================================================
#include "ExpSineSweep.hpp"
#include "ir.hpp"
#include "tools.hpp"

namespace fp {

// ---- tools (fp/tools.cpp) -- small host helpers kept for source compatibility ---------------------------
void tools::sumToMono(AudioBuffer<float>* buffer) {
    if (buffer->getNumChannels() != 2) { DBG("sumToMono() error: input is not stereo\n"); return; }
    float* l = buffer->getWritePointer(0);
    float* r = buffer->getWritePointer(1);
    for (int i = 0; i < buffer->getNumSamples(); ++i) { l[i] += r[i]; l[i] /= 2.0f; r[i] = 0.0f; }
}
void tools::makeStereo(AudioBuffer<float>* buffer) {
    if (buffer->getNumChannels() != 1) { DBG("makeStereo() error: input is not mono\n"); return; }
    buffer->setSize(2, buffer->getNumSamples(), true);
    buffer->copyFrom(1, 0, *buffer, 0, 0, buffer->getNumSamples());
}
void tools::complexDivPolar(float* a, float* b, float c, float d) {
    float amplA = std::sqrt((*a) * (*a) + (*b) * (*b)), phaseA = std::atan2(*b, *a);
    const float amplB = std::sqrt(c * c + d * d), phaseB = std::atan2(d, c);
    amplA /= amplB;
    phaseA -= phaseB;
    *a = amplA * std::cos(phaseA);
    *b = amplA * std::sin(phaseA);
}
float tools::dBToLin(float dB) { return std::pow(10.0f, dB / 20.0f); }
double tools::dBToLin(double dB) { return std::pow(10.0, dB / 20.0); }
float tools::linTodB(float lin) { return lin == 0.0f ? -333.0f : 20.0f * std::log(lin) / std::log(10.0f); }
double tools::linTodB(double lin) { return lin == 0.0 ? -333.0 : 20.0 * std::log(lin) / std::log(10.0); }
void tools::normalize(AudioBuffer<float>* buffer, float dBGoalLevel, bool printGain) {
    const float gain = dBToLin(dBGoalLevel) / buffer->getMagnitude(0, buffer->getNumSamples());
    buffer->applyGain(gain);
    if (printGain) std::printf("normalize gain: %g, dB: %9.6f\n", gain, linTodB(gain));
}
bool tools::isPowerOfTwo(int x) { return x != 0 && (x & (x - 1)) == 0; }
int tools::nextPowerOfTwo(int x, int result) {
    if (!isPowerOfTwo(result)) result = 1;
    if (isPowerOfTwo(x)) return x;
    while (result <= x) result *= 2;
    return result;
}
void tools::roundToZero(float* x, float threshold) {
    if (threshold < 0.0f) { DBG("tools::roundToZero error: threshold should be positive\n"); return; }
    if (!std::signbit(*x) && *x < threshold) *x = 0.0f;
    if (std::signbit(*x) && *x > -threshold) *x = 0.0f;
}
void tools::roundTo1TenQuadrillionth(float* x) {
    if (!std::signbit(*x) && *x < 1e-16) *x = 1e-16;
    if (std::signbit(*x) && *x > -1e-16) *x = -1e-16;
}
float tools::binAmpl(float* binPtr) { return (float) std::sqrt(std::pow((double) binPtr[0], 2.0) + std::pow((double) binPtr[1], 2.0)); }
float tools::binPhase(float* binPtr) { return std::atan2(binPtr[1], binPtr[0]); }
AudioBuffer<float> tools::generatePulse(int numSamples, int pulseOffset) {
    AudioBuffer<float> pulse(1, numSamples);
    pulse.clear();
    if (pulseOffset >= numSamples || pulseOffset < 0) pulseOffset = 0;
    pulse.setSample(0, pulseOffset, 1.0f);
    return pulse;
}
void tools::linearFade(AudioBuffer<float>* buffer, bool fadeIn, int startSample, int numSamples) {
    if (startSample + numSamples > buffer->getNumSamples()) { DBG("linearFade: startSample + numSamples exceeds buffer size.\n"); return; }
    const float step = 1.0 / numSamples;
    for (int c = 0; c < buffer->getNumChannels(); ++c)
        for (int i = startSample; i < startSample + numSamples; ++i) {
            const float gain = fadeIn ? (i - startSample) * step : 1.0 - (i - startSample) * step;
            buffer->setSample(c, i, buffer->getSample(c, i) * gain);
        }
}
void tools::sineFill(AudioBuffer<float>* buffer, float freq, float sampleRate, float ampl) {
    if (ampl > 1.0 || ampl <= 0.0) ampl = 1.0;
    for (int c = 0; c < buffer->getNumChannels(); ++c)
        for (int i = 0; i < buffer->getNumSamples(); ++i) buffer->setSample(c, i, ampl * std::cos(M_PI * 2 * freq * i / sampleRate));
}
AudioBuffer<float> tools::fftTransform(AudioBuffer<float>& buffer, bool formatAmplPhase) {
    const int ch = buffer.getNumChannels(), n = buffer.getNumSamples(), N = nextPowerOfTwo(n);
    AudioBuffer<float> out(ch, 2 * N);
    out.clear();
    std::vector<float> x = pack(buffer), y((size_t) ch * 2 * N);
    if (irb_fft_transform(x.data(), ch, n, formatAmplPhase ? 1 : 0, y.data()) != IRB_OK) raise("fp::tools::fftTransform");
    for (int c = 0; c < ch; ++c) out.copyFrom(c, 0, y.data() + (size_t) c * 2 * N, 2 * N);
    return out;
}
AudioBuffer<float> tools::fftInvTransform(AudioBuffer<float>& buffer) {
    const int ch = buffer.getNumChannels(), fftSize = buffer.getNumSamples(), N = fftSize / 2;
    AudioBuffer<float> out(ch, N);
    std::vector<float> s = pack(buffer), y((size_t) ch * N);
    if (irb_fft_inv_transform(s.data(), ch, fftSize, y.data()) != IRB_OK) raise("fp::tools::fftInvTransform");
    for (int c = 0; c < ch; ++c) out.copyFrom(c, 0, y.data() + (size_t) c * N, N);
    return out;
}

// ---- convolution (rest) -------------------------------------------------------------------------------
AudioBuffer<float> convolution::convolveNonPeriodic(AudioBuffer<float>& buffer1, AudioBuffer<float>& buffer2) {
    const int chx = buffer1.getNumChannels(), lx = buffer1.getNumSamples(), chh = buffer2.getNumChannels(), lh = buffer2.getNumSamples();
    const int lout = lx + lh - 1;
    std::vector<float> x = pack(buffer1), h = pack(buffer2), y((size_t) std::max(chx, 1) * std::max(lout, 1));
    const int rc = irb_convolve_nonperiodic(x.data(), chx, lx, h.data(), chh, lh, y.data());
    if (rc == IRB_ERR_LAYOUT) {
        std::printf("Either buffer1 or buffer2 is not mono nor stereo. Abort abort \n");
        AudioBuffer<float> cleared(buffer1);
        cleared.clear();
        return cleared;
    }
    if (rc != IRB_OK) raise("fp::convolution::convolveNonPeriodic");
    AudioBuffer<float> out(chx, lout);
    for (int c = 0; c < chx; ++c) out.copyFrom(c, 0, y.data() + (size_t) c * lout, lout);
    return out;
}
AudioBuffer<float> convolution::deconvolve(AudioBuffer<float>* numeratorBuffer, AudioBuffer<float>* denominatorBuffer, double sampleRate, bool smoothing,
                                           bool includePhase, bool includeAmplitude) {
    const int ln = numeratorBuffer->getNumSamples(), ld = denominatorBuffer->getNumSamples();
    const int N = tools::nextPowerOfTwo(std::max(ln, ld));
    AudioBuffer<float> out(1, N);
    if (irb_deconvolve(numeratorBuffer->getReadPointer(0), ln, denominatorBuffer->getReadPointer(0), ld, sampleRate, smoothing, includePhase, includeAmplitude,
                       out.getWritePointer(0)) != IRB_OK)
        raise("fp::convolution::deconvolve");
    return out;
}
void convolution::averagingFilter(AudioBuffer<float>* buffer, double octaveFraction, double sampleRate, bool logAvg, bool includePhase, bool includeAmplitude) {
    const int ch = buffer->getNumChannels(), fftSize = buffer->getNumSamples();
    if (!tools::isPowerOfTwo(fftSize)) { DBG("applyBucket() error: input buffer size is not power of 2.\n"); return; }
    std::vector<float> s = pack(*buffer);
    if (irb_averaging_filter(s.data(), ch, fftSize, octaveFraction, sampleRate, logAvg, includePhase, includeAmplitude) != IRB_OK) raise("fp::convolution::averagingFilter");
    for (int c = 0; c < ch; ++c) buffer->copyFrom(c, 0, s.data() + (size_t) c * fftSize, fftSize);
}

// ---- ir (fp/ir.cpp) ----------------------------------------------------------------------------------------
AudioBuffer<float> ir::invertFilter(AudioBuffer<float>& buffer, int samplerate) {
    const int n = buffer.getNumSamples();
    AudioBuffer<float> out(1, tools::nextPowerOfTwo(n));
    if (irb_invert_filter(buffer.getReadPointer(0), n, samplerate, out.getWritePointer(0)) != IRB_OK) raise("fp::ir::invertFilter");
    return out;
}
void ir::shifteroo(AudioBuffer<float>* buffer) {
    const int n = buffer->getNumSamples();
    if (n < 2) return;
    const int second = n / 2, first = n - second;
    AudioBuffer<float> moved(buffer->getNumChannels(), n);
    for (int c = 0; c < buffer->getNumChannels(); ++c) {
        moved.copyFrom(c, 0, *buffer, c, first, second);
        moved.copyFrom(c, second, *buffer, c, 0, first);
    }
    *buffer = moved;
}
AudioBuffer<float> ir::IRchop(AudioBuffer<float>& buffer, int IRlength, float thresholdLeveldB, int consecutiveSamplesBelowThreshold) {
    const int n = buffer.getNumSamples();
    const float* p = buffer.getReadPointer(0);
    const float peak = buffer.getMagnitude(0, n);
    int cursor = 0;
    while (cursor < n && std::fabs(p[cursor]) != peak) ++cursor;          // first sample carrying the peak magnitude
    if (cursor == n) cursor = 0;
    const float peakdB = tools::linTodB(std::fabs(peak));
    int below = 0, walked = 0;
    while (below < consecutiveSamplesBelowThreshold) {                       // walk backwards (with wrap) to a quiet run
        below = (tools::linTodB(std::fabs(p[cursor])) - peakdB < thresholdLeveldB) ? below + 1 : 0;
        if (--cursor < 0) cursor = n - 1;
        if (++walked == IRlength) break;
    }
    const int start = cursor;
    const int head = (IRlength + start > n - 1) ? n - start : IRlength;
    AudioBuffer<float> IR(1, IRlength);
    IR.clear();
    IR.copyFrom(0, 0, buffer, 0, start, head);
    if (head < IRlength) IR.copyFrom(0, head, buffer, 0, 0, IRlength - head);  // the part folded around the end
    const int fadeOut = IRlength / 4;
    tools::linearFade(&IR, false, IRlength - 1 - fadeOut, fadeOut);
    tools::linearFade(&IR, true, 0, walked / 4);
    return IR;
}
AudioBuffer<float> ir::IRtoRealFFTRaw(AudioBuffer<float>& buffer, int irPartSize) {
    const int n = buffer.getNumSamples(), parts = n / irPartSize + 1;
    AudioBuffer<float> out(1, parts * 2 * irPartSize);
    if (irb_ir_to_real_fft_raw(buffer.getReadPointer(0), n, irPartSize, out.getWritePointer(0)) != IRB_OK) raise("fp::ir::IRtoRealFFTRaw");
    return out;
}

// ---- ExpSineSweep (fp/ExpSineSweep.cpp) ---------------------------------------------------------------------
ExpSineSweep::ExpSineSweep() {}
ExpSineSweep::~ExpSineSweep() {}
void ExpSineSweep::assignParameters(double durationSecs, double sampleRate, double lowFreq, double highFreq) {
    SR = sampleRate;
    T = SR * durationSecs;
    w1 = lowFreq / SR * 2 * M_PI;
    w2 = highFreq / SR * 2 * M_PI;
    K = T * w1 / std::log(w2 / w1);
    L = T / std::log(w2 / w1);
}
void ExpSineSweep::generate(double durationSecs, double sampleRate, double lowFreq, double highFreq, double dBGain) {
    assignParameters(durationSecs, sampleRate, lowFreq, highFreq);
    genDuration = durationSecs; genLow = lowFreq; genHigh = highFreq; gendB = dBGain;
    const int n = (int) T;
    sweep.setSize(1, n);
    if (n > 0 && irb_ess_generate(durationSecs, sampleRate, lowFreq, highFreq, dBGain, 0, sweep.getWritePointer(0), n) < 0) raise("fp::ExpSineSweep::generate");
}
AudioBuffer<double> ExpSineSweep::getSweep() { return sweep; }
AudioBuffer<float> ExpSineSweep::getSweepFloat() { AudioBuffer<float> f; f.makeCopyOf(sweep); return f; }
void ExpSineSweep::generateInv() {
    if (sweep.getNumSamples() == 0) { DBG("ExpSineSweep::generateInv(): seems like generate() has not been used first to create sweep attribute. \n"); return; }
    // the reference reverses the CURRENT sweep buffer (fades included) and applies -6 dB/oct sample by sample
    sweepInv.makeCopyOf(sweep);
    sweepInv.reverse(0, sweepInv.getNumSamples());
    k = std::pow(10.0, (-6.0 * std::log2(w2 / w1)) / 20.0 / T);
    kend = std::pow(k, T);
    double* p = sweepInv.getWritePointer(0);
    double gain = k;
    for (int i = 0; i < sweepInv.getNumSamples(); ++i) { p[i] *= gain; gain *= k; }
}
void ExpSineSweep::generateInv(double durationSecs, double sampleRate, double lowFreq, double highFreq, double dBGain) {
    generate(durationSecs, sampleRate, lowFreq, highFreq, dBGain);
    generateInv();
}
AudioBuffer<double> ExpSineSweep::getSweepInv() { return sweepInv; }
AudioBuffer<float> ExpSineSweep::getSweepInvFloat() { AudioBuffer<float> f; f.makeCopyOf(sweepInv); return f; }
double ExpSineSweep::getFreqAtSampleIndexHelper(int index) {
    if (index < 0 || index >= (int) T) { DBG("index out of bounds. \n"); return -1; }
    const double lowFreq = w1 * SR / (2 * M_PI), totalOct = std::log(w2 / w1) / std::log(2);
    return lowFreq * std::pow(2.0, (double) index / T * totalOct);
}
int ExpSineSweep::getSampleHelper(double freq) {
    const double lowFreq = w1 * SR / (2 * M_PI);
    const double oct = std::log(freq / lowFreq) / std::log(2), totalOct = std::log(w2 / w1) / std::log(2);
    const int t = (int) std::round(oct / totalOct * T);
    if (t < 0 || t >= T) { DBG("Specified frequency is out of bounds for this sweep. \n"); return -1; }
    return t;
}
int ExpSineSweep::getSampleIndexAtFreq(double freq) {
    if (sweep.getNumSamples() == 0) { DBG("sweep has not been generated yet. Try overloaded function? \n"); return -1; }
    return getSampleHelper(freq);
}
int ExpSineSweep::getSampleIndexAtFreq(double freq, double durationSecs, double sampleRate, double lowFreq, double highFreq) {
    assignParameters(durationSecs, sampleRate, lowFreq, highFreq);
    return getSampleHelper(freq);
}
double ExpSineSweep::getFreqAtSampleIndex(int index) {
    if (sweep.getNumSamples() == 0) { DBG("sweep has not been generated yet. Try overloaded function? \n"); return -1; }
    return getFreqAtSampleIndexHelper(index);
}
double ExpSineSweep::getFreqAtSampleIndex(int index, double durationSecs, double sampleRate, double lowFreq, double highFreq) {
    assignParameters(durationSecs, sampleRate, lowFreq, highFreq);
    return getFreqAtSampleIndexHelper(index);
}
void ExpSineSweep::linFadeout(double freq) {
    if (sweep.getNumSamples() == 0) { DBG("Sweep has not been generated yet. \n"); return; }
    const int index = getSampleIndexAtFreq(freq), len = sweep.getNumSamples() - index;
    for (int i = index; i < sweep.getNumSamples(); ++i) sweep.setSample(0, i, sweep.getSample(0, i) * (len - (i - index)) / len);
}
void ExpSineSweep::dBFadeout(double freq) {
    if (sweep.getNumSamples() == 0) { DBG("Sweep has not been generated yet. \n"); return; }
    const int index = getSampleIndexAtFreq(freq), len = sweep.getNumSamples() - index;
    const double perSample = tools::dBToLin(-80.0 / len);
    double g = perSample;
    for (int i = index; i < sweep.getNumSamples(); ++i) { sweep.setSample(0, i, sweep.getSample(0, i) * g); g *= perSample; }
}
void ExpSineSweep::brickwallFadeout(double freq) {
    if (sweep.getNumSamples() == 0) { DBG("Sweep has not been generated yet. \n"); return; }
    const int index = getSampleIndexAtFreq(freq);
    sweep.clear(index, sweep.getNumSamples() - index);
}

}  // namespace fp

// =====================================================================================================
// Formats (N4) and the capture -> filter chain (N3): host I/O and composition only
// =====================================================================================================
#include <cstdint>
#include <fstream>
#include <iomanip>

#include "CaptureChain.hpp"
#include "Formats.hpp"

namespace fp {
namespace b200 {
namespace formats {

namespace {
void put16(std::vector<unsigned char>& v, uint32_t x) { v.push_back(x & 0xff); v.push_back((x >> 8) & 0xff); }
void put32(std::vector<unsigned char>& v, uint32_t x) { put16(v, x & 0xffff); put16(v, x >> 16); }
uint32_t get32(const unsigned char* p) { return (uint32_t) p[0] | ((uint32_t) p[1] << 8) | ((uint32_t) p[2] << 16) | ((uint32_t) p[3] << 24); }
uint32_t get16(const unsigned char* p) { return (uint32_t) p[0] | ((uint32_t) p[1] << 8); }
}  // namespace

bool writeWav(const std::string& path, const AudioBuffer<float>& buffer, int sampleRate, int bitsPerSample) {
    if (bitsPerSample != 16 && bitsPerSample != 24) return false;
    const int ch = buffer.getNumChannels(), n = buffer.getNumSamples(), bytes = bitsPerSample / 8;
    if (ch < 1) return false;
    const uint32_t dataBytes = (uint32_t) ((size_t) ch * (size_t) n * (size_t) bytes);
    std::vector<unsigned char> out;
    out.reserve(44 + (size_t) dataBytes + 1);
    out.insert(out.end(), {'R', 'I', 'F', 'F'});
    put32(out, 36 + dataBytes + (dataBytes & 1));
    out.insert(out.end(), {'W', 'A', 'V', 'E', 'f', 'm', 't', ' '});
    put32(out, 16); put16(out, 1); put16(out, (uint32_t) ch); put32(out, (uint32_t) sampleRate);
    put32(out, (uint32_t) (sampleRate * ch * bytes)); put16(out, (uint32_t) (ch * bytes)); put16(out, (uint32_t) bitsPerSample);
    out.insert(out.end(), {'d', 'a', 't', 'a'});
    put32(out, dataBytes);
    // Sample quantisation = what juce::AudioFormatWriter does for an integer WAV (JUCE 6.0.1, the version the reference pins;
    // JUCE is not vendored by the reference, so this restates two of its functions):
    //   1. AudioFormatWriter::convertFloatsToInts (juce_audio_formats/format/juce_AudioFormatWriter.cpp): every float goes to a
    //      LEFT-JUSTIFIED 32-bit integer in double arithmetic:  samp <= -1.0 -> INT_MIN;  samp >= 1.0 -> INT_MAX;
    //      otherwise roundToInt (INT_MAX * samp), round-half-to-even (a NaN fails both comparisons and its conversion is
    //      undefined there; here it becomes 0);
    //   2. WavAudioFormatWriter::write converts Int32 -> Int24 / Int16 with AudioData::Int24::setAsInt32LE =
    //      littleEndian24BitToChars (value >> 8) and Int16::setAsInt32LE = (value >> 16): an ARITHMETIC shift, i.e. the top
    //      bits of the 32-bit value, rounding toward minus infinity (no dither).
    // So +1.0 -> 0x7fffff, -1.0 -> -0x800000, and anything of magnitude below 2^-32 (every denormal) -> 0.
    for (int i = 0; i < n; ++i)
        for (int c = 0; c < ch; ++c) {
            const double samp = (double) buffer.getSample(c, i);
            int32_t q;
            if (samp <= -1.0) q = INT32_MIN;
            else if (samp >= 1.0) q = INT32_MAX;
            else if (samp != samp) q = 0;
            else q = (int32_t) std::lrint(2147483647.0 * samp);
            const uint32_t u = (uint32_t) (q >> (32 - bitsPerSample));
            for (int b = 0; b < bytes; ++b) out.push_back((u >> (8 * b)) & 0xff);
        }
    if (dataBytes & 1) out.push_back(0);
    std::ofstream f(path, std::ios::binary | std::ios::trunc);
    if (!f) return false;
    f.write((const char*) out.data(), (std::streamsize) out.size());
    return (bool) f;
}

AudioBuffer<float> readWav(const std::string& path, int* sampleRate) {
    AudioBuffer<float> empty;
    std::ifstream f(path, std::ios::binary);
    if (!f) return empty;
    std::vector<unsigned char> d((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    if (d.size() < 12 || std::memcmp(d.data(), "RIFF", 4) != 0 || std::memcmp(d.data() + 8, "WAVE", 4) != 0) return empty;
    int fmt = 0, ch = 0, bits = 0, rate = 0;
    size_t pos = 12;
    while (pos + 8 <= d.size()) {
        const uint32_t len = get32(&d[pos + 4]);
        const unsigned char* body = &d[pos + 8];
        if (pos + 8 + len > d.size() && std::memcmp(&d[pos], "data", 4) != 0) return empty;
        if (std::memcmp(&d[pos], "fmt ", 4) == 0 && len >= 16) {
            fmt = (int) get16(body); ch = (int) get16(body + 2); rate = (int) get32(body + 4); bits = (int) get16(body + 14);
            if (fmt == 0xfffe && len >= 26) fmt = (int) get16(body + 24);      // WAVE_FORMAT_EXTENSIBLE: the sub-format's first two bytes
        } else if (std::memcmp(&d[pos], "data", 4) == 0) {
            if (ch < 1 || !((fmt == 1 && (bits == 16 || bits == 24 || bits == 32)) || (fmt == 3 && bits == 32))) return empty;
            const size_t avail = std::min<size_t>(len, d.size() - pos - 8), bytes = (size_t) bits / 8;
            const int n = (int) (avail / (bytes * (size_t) ch));
            AudioBuffer<float> out(ch, n);
            for (int i = 0; i < n; ++i)
                for (int c = 0; c < ch; ++c) {
                    const unsigned char* p = body + ((size_t) i * ch + c) * bytes;
                    float v;
                    if (fmt == 3) { uint32_t u = get32(p); std::memcpy(&v, &u, 4); }
                    else {
                        uint32_t u = 0;
                        for (size_t b = 0; b < bytes; ++b) u |= (uint32_t) p[b] << (8 * b);
                        const int32_t s = (int32_t) (u << (32 - bits)) >> (32 - bits);      // sign extension
                        v = (float) ((double) s / (double) (1u << (bits - 1)));
                    }
                    out.setSample(c, i, v);
                }
            if (sampleRate) *sampleRate = rate;
            return out;
        }
        pos += 8 + (size_t) len + (len & 1);
    }
    return empty;
}

bool writeSweepAndIR(const std::string& path, const AudioBuffer<float>& sweepRecording, const AudioBuffer<float>& ir, int sampleRate, int numSamples) {
    if (sweepRecording.getNumChannels() < 1 || ir.getNumChannels() < 1 || numSamples < 1) return false;
    AudioBuffer<float> save(2, numSamples);                                       // PluginProcessor.cpp:664-682
    save.clear();
    save.copyFrom(0, 0, sweepRecording, 0, 0, std::min(numSamples, sweepRecording.getNumSamples()));
    save.copyFrom(1, 0, ir, 0, 0, std::min(numSamples, ir.getNumSamples()));
    return writeWav(path, save, sampleRate, 24);
}
bool readSweepAndIR(const std::string& path, AudioBuffer<float>& sweepRecording, AudioBuffer<float>& ir, int numSamples) {
    AudioBuffer<float> both = readWav(path);
    if (both.getNumChannels() < 2) return false;
    sweepRecording.setSize(1, numSamples); ir.setSize(1, numSamples);             // PluginProcessor.cpp:909-917
    sweepRecording.clear(); ir.clear();
    const int n = std::min(numSamples, both.getNumSamples());
    sweepRecording.copyFrom(0, 0, both, 0, 0, n);
    ir.copyFrom(0, 0, both, 1, 0, n);
    return true;
}

bool writeSpectrumTsv(const std::string& path, const std::string& name, const AudioBuffer<float>& spectrum, int sampleRate) {
    const int fftSize = spectrum.getNumSamples();
    if (spectrum.getNumChannels() < 1 || !tools::isPowerOfTwo(fftSize)) return false;          // ParallelBufferPrinter.cpp:289-293
    const int N = fftSize / 2;
    const double nyquist = sampleRate / 2;
    const double freqPerBin = nyquist / (double) (N / 2);
    std::ofstream fout(path, std::ofstream::out | std::ofstream::trunc);
    if (!fout.is_open()) return false;
    std::vector<float> bins(spectrum.getReadPointer(0), spectrum.getReadPointer(0) + fftSize);
    fout << "freq\t" << name << "[lin]\t" << name << "[dB]\t" << "bin\t" << name << " phase[rad]\n";
    for (int bin = 0; bin <= N; bin += 2) {                                       // the first column keeps the stream's precision of the
        fout << freqPerBin * bin / 2 << "\t";                                     // previous row (8 after row 0), as in the reference
        fout << std::setprecision(8) << tools::binAmpl(&bins[(size_t) bin]) << "\t";
        fout << std::setprecision(8) << tools::linTodB(std::fabs(tools::binAmpl(&bins[(size_t) bin]))) << "\t";
        fout << bin / 2 << "\t";
        fout << std::setprecision(8) << tools::binPhase(&bins[(size_t) bin]) << "\n";
    }
    return (bool) fout;
}

bool writeRawSpectraText(const std::string& path, const AudioBuffer<float>& packed, int irPartSize) {
    if (packed.getNumChannels() < 1 || irPartSize < 1) return false;
    const int N = 2 * irPartSize;
    std::ofstream fout(path, std::ofstream::out | std::ofstream::trunc);
    if (!fout.is_open()) return false;
    for (int i = 0; i < packed.getNumSamples(); ++i) {                             // fp/ir.cpp:137-142
        if (i % 8 == 0) fout << '\n';
        if (i % N == 0) fout << '\n';
        fout << packed.getSample(0, i) << ", ";
    }
    return (bool) fout;
}

}  // namespace formats

// ---- capture -> filter chain ---------------------------------------------------------------------------
AudioBuffer<float> captureToIR(CircularBufferArray& capturedBlocks, AudioBuffer<float>& sweepForDeconv, double sampleRate, AudioBuffer<float>* recordingOut) {
    AudioBuffer<float> recording = capturedBlocks.consolidate(0);                 // PluginProcessor.cpp:305,311
    if (recordingOut) recordingOut->makeCopyOf(recording);
    return convolution::deconvolve(&recording, &sweepForDeconv, sampleRate);      // :306,312 (smoothing, phase, amplitude: defaults)
}
AudioBuffer<float> createIRFilt(AudioBuffer<float>& irTarget, AudioBuffer<float>& irBase, double sampleRate, bool includePhase, bool includeAmplitude) {
    return convolution::deconvolve(&irTarget, &irBase, sampleRate, true, includePhase, includeAmplitude);      // :606-615
}
AudioBuffer<float> chopAndNormalize(AudioBuffer<float>& ir, int irLength, float thresholdLeveldB, int consecutiveSamplesBelowThreshold) {
    AudioBuffer<float> out = ir::IRchop(ir, irLength, thresholdLeveldB, consecutiveSamplesBelowThreshold);
    tools::normalize(&out, 0.0f, false);
    return out;
}
AudioBuffer<float> capturesToIRs(AudioBuffer<float>& captures, AudioBuffer<float>& sweepForDeconv, double sampleRate, int irLength, float thresholdLeveldB,
                                 int consecutiveSamplesBelowThreshold, bool smoothing) {
    const int batch = captures.getNumChannels(), n = captures.getNumSamples();
    std::vector<float> x = pack(captures);
    AudioBuffer<float> out(batch, irLength);
    if (irb_deconvolve_chop_batch(x.data(), batch, n, sweepForDeconv.getReadPointer(0), sweepForDeconv.getNumSamples(), sampleRate, smoothing, 1, 1, irLength,
                                  thresholdLeveldB, consecutiveSamplesBelowThreshold, 1, 0.0f, out.getWritePointer(0), nullptr) != IRB_OK)
        raise("fp::b200::capturesToIRs");
    return out;
}

}  // namespace b200
}  // namespace fp
