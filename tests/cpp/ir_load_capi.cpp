// tests/cpp/ir_load_capi.cpp -- TEST INFRASTRUCTURE: a flat C view of fp::b200::StreamingConvolver and MultiGpuConvolver
// (irbaboon_b200/fp) for tests/test_gpu_ir_load.py: setIRs (one call for a whole IR file) next to a loop of setIR.  Compiled by
// the test itself into a temporary directory.
#include <cstdio>
#include <stdexcept>
#include <vector>

#include "../../irbaboon_b200/fp/StreamingConvolver.hpp"

static AudioBuffer<float> file(const float* data, int ch, int n) {
    AudioBuffer<float> b(ch, n);
    for (int c = 0; c < ch; ++c) b.copyFrom(c, 0, data + (size_t) c * n, n);
    return b;
}

extern "C" {
// multi = 0: StreamingConvolver on device 0; multi = n > 0: MultiGpuConvolver over devices 0 .. n-1 (modulo the device count)
void* il_create(int multi, int devices, int B, int P, int channels, int nIRs) {
    try {
        if (!multi) return new fp::b200::StreamingConvolver(B, P, channels, nIRs, 0);
        std::vector<int> d;
        for (int i = 0; i < multi; ++i) d.push_back(i % (devices > 0 ? devices : 1));
        return new fp::b200::MultiGpuConvolver(d, B, P, channels, nIRs);
    } catch (const std::exception& e) { std::fprintf(stderr, "il_create: %s\n", e.what()); return nullptr; }
}
void il_destroy(int multi, void* h) {
    if (multi) delete (fp::b200::MultiGpuConvolver*) h;
    else delete (fp::b200::StreamingConvolver*) h;
}
// irs: [ch][n] planar; loop = 1: one setIR per channel, 0: one setIRs
int il_set(int multi, void* h, int firstId, const float* irs, int ch, int n, int loop) {
    try {
        if (loop) {
            for (int c = 0; c < ch; ++c) {
                const AudioBuffer<float> b = file(irs + (size_t) c * n, 1, n);
                if (multi) ((fp::b200::MultiGpuConvolver*) h)->setIR(firstId + c, b);
                else ((fp::b200::StreamingConvolver*) h)->setIR(firstId + c, b);
            }
        } else {
            const AudioBuffer<float> b = file(irs, ch, n);
            if (multi) ((fp::b200::MultiGpuConvolver*) h)->setIRs(firstId, b);
            else ((fp::b200::StreamingConvolver*) h)->setIRs(firstId, b);
        }
        return 0;
    } catch (const std::exception& e) { std::fprintf(stderr, "il_set: %s\n", e.what()); return -1; }
}
int il_bind(int multi, void* h, int c0, int c1, int ir) {
    try {
        if (multi) ((fp::b200::MultiGpuConvolver*) h)->bind(c0, c1, ir);
        else ((fp::b200::StreamingConvolver*) h)->bind(c0, c1, ir);
        return 0;
    } catch (const std::exception&) { return -1; }
}
// dense [nBlocks][channels][B]
int il_process(int multi, void* h, const float* in, float* out, int nBlocks) {
    try {
        if (multi) ((fp::b200::MultiGpuConvolver*) h)->process(in, out, nBlocks);
        else ((fp::b200::StreamingConvolver*) h)->process(in, out, nBlocks);
        return 0;
    } catch (const std::exception&) { return -1; }
}
}
