// fp/CaptureChain.hpp -- the capture -> filter chain around the deconvolution kernels (SURVEY 8f, N3), i.e. what
// IRBaboonAudioProcessor does once a sweep capture is complete (Source/PluginProcessor.cpp:291-332,606-615) and what its
// editor does to the result for display (ir::IRchop, tools::normalize).  Every step is one of the fp:: functions; the
// transforms, the division and the smoothing run on the GPU (convolution.hpp), the rest is sample shuffling.
#pragma once
#include "CircularBufferArray.hpp"
#include "convolution.hpp"
#include "ir.hpp"
#include "tools.hpp"

namespace fp {
namespace b200 {

// inputCaptureArray.consolidate(0) -> deconvolve(recording, sweepForDeconv, sampleRate) with the plug-in's defaults
// (smoothing, phase and amplitude kept): PluginProcessor.cpp:305-306,311-312.  recordingOut receives the consolidated capture.
AudioBuffer<float> captureToIR(CircularBufferArray& capturedBlocks, AudioBuffer<float>& sweepForDeconv, double sampleRate, AudioBuffer<float>* recordingOut = nullptr);
// createIRFilt (PluginProcessor.cpp:606-615): deconvolve(IRTarget, IRBase, sampleRate, true, includePhase, includeAmplitude)
AudioBuffer<float> createIRFilt(AudioBuffer<float>& irTarget, AudioBuffer<float>& irBase, double sampleRate, bool includePhase = true, bool includeAmplitude = true);
// an IR cut to irLength around its peak (ir::IRchop) and normalised to 0 dB (tools::normalize): library functions of
// fp/ir.hpp and fp/tools.hpp composed for convenience -- the plug-in itself never calls IRchop
AudioBuffer<float> chopAndNormalize(AudioBuffer<float>& ir, int irLength, float thresholdLeveldB, int consecutiveSamplesBelowThreshold);
// the batched form of captureToIR + chopAndNormalize: one capture per channel of `captures`, all divided by sweepForDeconv, cut and
// normalised on the GPU (irb_deconvolve_chop_batch) -> one IR of irLength samples per channel; only the IRs leave the device.
// smoothing = false skips the 1/13-octave smoothing the plug-in applies.
AudioBuffer<float> capturesToIRs(AudioBuffer<float>& captures, AudioBuffer<float>& sweepForDeconv, double sampleRate, int irLength, float thresholdLeveldB,
                                 int consecutiveSamplesBelowThreshold, bool smoothing = true);

}  // namespace b200
}  // namespace fp
