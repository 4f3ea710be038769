// fp/StreamingConvolver.hpp -- C++ RAII handle over irb_engine (include/irb_b200.h): the batched,
// device-resident replacement of the real-time UPOLA engine the reference inlines in
// IRBaboonAudioProcessor::processBlock (Source/PluginProcessor.cpp:403-562).  The reference has no
// class for this (SURVEY D2); this is the object a processBlock replacement or a headless harness owns.
#pragma once
#ifdef IRB_USE_REAL_JUCE
#include <JuceHeader.h>
#else
#include "juce_stub/JuceHeader.h"
#endif
#include <vector>

#include "../../include/irb_b200.h"

namespace fp {
namespace b200 {

class StreamingConvolver {
public:
    // channels = independent stream-channels processed per block; maxPartitions = ceil(longest IR / blockSize)
    StreamingConvolver(int blockSize, int maxPartitions, int channels, int numIRs = 1, int device = 0);
    ~StreamingConvolver();
    StreamingConvolver(const StreamingConvolver&) = delete;
    StreamingConvolver& operator=(const StreamingConvolver&) = delete;

    // mono IR (channel 0) or stereo IR folded to (L+R)/2, as convolvePeriodic does for mono audio
    void setIR(int irId, const AudioBuffer<float>& ir, bool foldStereo = false);
    // many IRs in one call (irb_engine_set_irs): channel c of irs becomes IR firstId + c, each mono
    void setIRs(int firstId, const AudioBuffer<float>& irs);
    void bind(int channelBegin, int channelEnd, int irId);
    void reset();
    // one block per call: buffer holds `channels` channels of exactly blockSize samples, processed in place
    void processBlock(AudioBuffer<float>& buffer);
    // dense [nBlocks][channels][blockSize] host arrays (pinned memory from irb_host_alloc is fastest)
    void process(const float* in, float* out, int nBlocks);
    // the same with 16- or 24-bit integer PCM (or float) in and out, converted on the device (irb_engine_process_pcm)
    void process(const void* in, irb_sample_format inFormat, void* out, irb_sample_format outFormat, int nBlocks);

    int getBlockSize() const { return blockSize; }
    int getNumChannels() const { return channels; }
    int getLatencySamples() const { return blockSize; }      // PluginProcessor.cpp:59,169-174 with hostBlock <= B
    irb_engine* handle() const { return engine; }

private:
    irb_engine* engine = nullptr;
    int blockSize, channels;
    std::vector<float> stageIn, stageOut;
};

// IR-matrix streaming convolution (irb_engine_create_matrix): `groups` groups of `ins` input channels, each producing `outs`
// output channels, out[g*outs + o] = sum_i conv(in[g*ins + i], IR ids[i*outs + o]).  (1, 2) is mono -> stereo (a binaural or
// spatial source), (2, 2) true stereo with the IRs LL, LR, RL, RR.  Every input keeps one delay line, read once per block for
// all the IRs it feeds.
class MatrixConvolver {
public:
    // numIRs = 0: one matrix, ins*outs IRs; until bindMatrix every group uses IRs 0 .. ins*outs-1
    MatrixConvolver(int blockSize, int maxPartitions, int groups, int ins, int outs, int numIRs = 0, int device = 0);
    ~MatrixConvolver();
    MatrixConvolver(const MatrixConvolver&) = delete;
    MatrixConvolver& operator=(const MatrixConvolver&) = delete;

    // An IR file: a mono one sets IR irId; one with ins*outs channels sets IRs irId .. irId + ins*outs - 1 from its channels
    // (a stereo file is the {L, R} pair of a (1, 2) matrix, a four-channel file the LL, LR, RL, RR of a (2, 2) matrix), in one
    // irb_engine_set_irs call
    void setIR(int irId, const AudioBuffer<float>& ir);
    void bindMatrix(int groupBegin, int groupEnd, const std::vector<int>& irIds);    // irIds[i*outs + o]
    void reset();
    // one block per call: `in` holds groups*ins channels, `out` groups*outs channels, of exactly blockSize samples
    void processBlock(const AudioBuffer<float>& in, AudioBuffer<float>& out);
    // dense host arrays: in [nBlocks][groups*ins][blockSize], out [nBlocks][groups*outs][blockSize]
    void process(const float* in, float* out, int nBlocks);
    // the same in any irb_sample_format each (irb_engine_process_pcm)
    void process(const void* in, irb_sample_format inFormat, void* out, irb_sample_format outFormat, int nBlocks);

    int getBlockSize() const { return blockSize; }
    int getNumInputs() const { return groups * ins; }
    int getNumOutputs() const { return groups * outs; }
    int getLatencySamples() const { return blockSize; }
    irb_engine* handle() const { return engine; }

private:
    irb_engine* engine = nullptr;
    int blockSize, groups, ins, outs;
    std::vector<float> stageIn, stageOut;
};

// The same over several GPUs driven from this process (irb_group_*): channels are sharded by contiguous ranges, shared IRs are
// replicated on every device (numIRs > 0) or every channel owns the IR with its own number (numIRs == 0).
class MultiGpuConvolver {
public:
    MultiGpuConvolver(const std::vector<int>& devices, int blockSize, int maxPartitions, int channels, int numIRs = 1);
    ~MultiGpuConvolver();
    MultiGpuConvolver(const MultiGpuConvolver&) = delete;
    MultiGpuConvolver& operator=(const MultiGpuConvolver&) = delete;
    void setIR(int irId, const AudioBuffer<float>& ir, bool foldStereo = false);
    // many IRs in one call (irb_group_set_irs): channel c of irs becomes IR (or, with numIRs == 0, channel) firstId + c, each mono
    void setIRs(int firstId, const AudioBuffer<float>& irs);
    void bind(int channelBegin, int channelEnd, int irId);
    void reset();
    void process(const float* in, float* out, int nBlocks);   // dense [nBlocks][channels][blockSize] host arrays
    // the same in any irb_sample_format each (irb_group_process_pcm)
    void process(const void* in, irb_sample_format inFormat, void* out, irb_sample_format outFormat, int nBlocks);
    irb_group* handle() const { return group; }

private:
    irb_group* group = nullptr;
};

}  // namespace b200
}  // namespace fp
