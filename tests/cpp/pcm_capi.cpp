// tests/cpp/pcm_capi.cpp -- TEST INFRASTRUCTURE: a flat C view of the raw-pointer PCM process() of the C++ facade
// (fp::b200::StreamingConvolver, MatrixConvolver, MultiGpuConvolver) so that a python test can drive it next to the python
// binding.  Compiled by the test itself (tests/test_gpu_pcm.py) into a temporary directory.
#include <cstdio>
#include <stdexcept>
#include <vector>

#include "../../irbaboon_b200/fp/StreamingConvolver.hpp"

using fp::b200::MatrixConvolver;
using fp::b200::MultiGpuConvolver;
using fp::b200::StreamingConvolver;

static AudioBuffer<float> mono(const float* ir, int n) {
    AudioBuffer<float> b(1, n);
    b.copyFrom(0, 0, ir, n);
    return b;
}

extern "C" {
// kind 0: StreamingConvolver(B, P, channels), 1: MatrixConvolver(B, P, channels = groups, ins, 2), 2: MultiGpuConvolver on devices 0 .. ndev-1
void* pc_create(int kind, int B, int P, int channels, int ins, int ndev) {
    try {
        if (kind == 0) return new StreamingConvolver(B, P, channels, 1, 0);
        if (kind == 1) return new MatrixConvolver(B, P, channels, ins, 2, 0, 0);
        std::vector<int> devs;
        for (int d = 0; d < ndev; ++d) devs.push_back(d);
        return new MultiGpuConvolver(devs, B, P, channels, 1);
    } catch (const std::exception& e) { std::fprintf(stderr, "pc_create: %s\n", e.what()); return nullptr; }
}
void pc_destroy(int kind, void* h) {
    if (kind == 0) delete (StreamingConvolver*) h;
    else if (kind == 1) delete (MatrixConvolver*) h;
    else delete (MultiGpuConvolver*) h;
}
// IR irId (a matrix engine: IR irId of its matrix) from n mono taps
int pc_set_ir(int kind, void* h, int irId, const float* ir, int n) {
    try {
        if (kind == 0) ((StreamingConvolver*) h)->setIR(irId, mono(ir, n));
        else if (kind == 1) ((MatrixConvolver*) h)->setIR(irId, mono(ir, n));
        else ((MultiGpuConvolver*) h)->setIR(irId, mono(ir, n));
        return 0;
    } catch (const std::exception&) { return -1; }
}
int pc_process(int kind, void* h, const void* in, int inFormat, void* out, int outFormat, int nBlocks) {
    const irb_sample_format fi = (irb_sample_format) inFormat, fo = (irb_sample_format) outFormat;
    try {
        if (kind == 0) ((StreamingConvolver*) h)->process(in, fi, out, fo, nBlocks);
        else if (kind == 1) ((MatrixConvolver*) h)->process(in, fi, out, fo, nBlocks);
        else ((MultiGpuConvolver*) h)->process(in, fi, out, fo, nBlocks);
        return 0;
    } catch (const std::exception&) { return -1; }
}
}
