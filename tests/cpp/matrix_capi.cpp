// tests/cpp/matrix_capi.cpp -- TEST INFRASTRUCTURE: a flat C view of fp::b200::MatrixConvolver (irbaboon_b200/fp) so that a
// python test can drive the C++ facade of the IR-matrix engine next to the python binding.  Compiled by the test itself
// (tests/test_gpu_matrix_facade.py) into a temporary directory.
#include <algorithm>
#include <cstdio>
#include <stdexcept>
#include <vector>

#include "../../irbaboon_b200/fp/StreamingConvolver.hpp"

static void fill(AudioBuffer<float>& b, const float* data) {
    for (int c = 0; c < b.getNumChannels(); ++c) b.copyFrom(c, 0, data + (size_t) c * b.getNumSamples(), b.getNumSamples());
}
static void dump(const AudioBuffer<float>& b, float* out) {
    for (int c = 0; c < b.getNumChannels(); ++c) std::copy_n(b.getReadPointer(c), b.getNumSamples(), out + (size_t) c * b.getNumSamples());
}

extern "C" {
void* mx_create(int B, int P, int groups, int ins, int outs, int nIRs) {
    try { return new fp::b200::MatrixConvolver(B, P, groups, ins, outs, nIRs, 0); }
    catch (const std::exception& e) { std::fprintf(stderr, "mx_create: %s\n", e.what()); return nullptr; }
}
void mx_destroy(void* h) { delete (fp::b200::MatrixConvolver*) h; }
// ir: [ch][n] planar, an IR file of 1 or ins*outs channels
int mx_set_ir(void* h, int irId, const float* ir, int ch, int n) {
    AudioBuffer<float> b(ch, n);
    fill(b, ir);
    try { ((fp::b200::MatrixConvolver*) h)->setIR(irId, b); return 0; } catch (const std::exception&) { return -1; }
}
int mx_bind(void* h, int g0, int g1, const int* ids, int n) {
    try { ((fp::b200::MatrixConvolver*) h)->bindMatrix(g0, g1, std::vector<int>(ids, ids + n)); return 0; } catch (const std::exception&) { return -1; }
}
int mx_reset(void* h) {
    try { ((fp::b200::MatrixConvolver*) h)->reset(); return 0; } catch (const std::exception&) { return -1; }
}
// dense [nBlocks][inputs][B] -> [nBlocks][outputs][B]
int mx_process(void* h, const float* in, float* out, int nBlocks) {
    try { ((fp::b200::MatrixConvolver*) h)->process(in, out, nBlocks); return 0; } catch (const std::exception&) { return -1; }
}
// one block through AudioBuffers: in [inputs][B], out [outputs][B] planar
int mx_process_block(void* h, const float* in, float* out) {
    auto* m = (fp::b200::MatrixConvolver*) h;
    AudioBuffer<float> bi(m->getNumInputs(), m->getBlockSize()), bo(m->getNumOutputs(), m->getBlockSize());
    fill(bi, in);
    try { m->processBlock(bi, bo); dump(bo, out); return 0; } catch (const std::exception&) { return -1; }
}
}
