// tests/cpp/chop_rule.cpp -- host side of the tests of the batched IR chop (irb_ir_chop_batch_device, irb_deconvolve_chop_batch):
// the level rule's log on the host, the facade's own levels, and the facade's capturesToIRs, as a flat C API for ctypes.
// Built by tests/chop_rule.py (g++ -fopenmp) against the facade library.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <exception>

#include "../../irbaboon_b200/fp/fp_include_all.hpp"

namespace {

float from_bits(uint32_t b) { float v; std::memcpy(&v, &b, 4); return v; }

// the device's level rule (irb_chop.cuh, chop_level_db) compiled for the host: without FMA contraction (x86-64, no -mfma)
// every float operation here is the device's __fmul_rn / __fdiv_rn
constexpr float kLn10f = 2.302585092994045684f;
float rule_log(float v) { return (float) std::log((double) v); }
float rule_db(float v) { return v == 0.0f ? -333.0f : 20.0f * rule_log(v) / kLn10f; }

}  // namespace

extern "C" {

float chop_ln10f() { return kLn10f; }
float chop_glibc_ln10f() { return std::log(10.0f); }

// levels of |x_i| in dB: the facade's tools::linTodB (glibc logf) and the device rule
void chop_levels_facade(const float* x, long long n, float* db) { for (long long i = 0; i < n; ++i) db[i] = fp::tools::linTodB(std::fabs(x[i])); }
void chop_levels_rule(const float* x, long long n, float* db) { for (long long i = 0; i < n; ++i) db[i] = rule_db(std::fabs(x[i])); }

// Every positive finite float v: is rule_log(v) the float nearest ln(v)?  The reference is ln(v) in x87 extended precision (64-bit
// significand, logl); a float that is no farther from it than both its neighbours is the correctly rounded result.
// counts = {inputs, rule not nearest, glibc logf != rule, facade linTodB != rule_db}; bad[0, max_bad) receives the first misses.
void chop_log_sweep(long long* counts, uint32_t* bad, int max_bad) {
    long long n = 0, miss = 0, dlog = 0, ddb = 0;
#pragma omp parallel for schedule(dynamic, 1 << 16) reduction(+ : n, miss, dlog, ddb)
    for (long long b = 1; b < 0x7f800000LL; ++b) {
        const float v = from_bits((uint32_t) b);
        const float r = rule_log(v);
        const long double ref = logl((long double) v);
        const long double e = fabsl((long double) r - ref);
        const float up = std::nextafter(r, INFINITY), dn = std::nextafter(r, -INFINITY);
        if (fabsl((long double) up - ref) < e || fabsl((long double) dn - ref) < e) {
            long long k;
#pragma omp atomic capture
            k = counts[1]++;
            if (k < max_bad) bad[k] = (uint32_t) b;
            ++miss;
        }
        ++n;
        if (std::log(v) != r) ++dlog;
        if (fp::tools::linTodB(v) != rule_db(v)) ++ddb;
    }
    counts[0] = n; counts[1] = miss; counts[2] = dlog; counts[3] = ddb;
}

// up to max_out positive floats from bits `from` upward whose facade level differs from the rule's, with the facade's below the rule's
int chop_find_level_flips(uint32_t from, float* out, int max_out) {
    int k = 0;
    for (uint32_t b = from; b < 0x7f800000u && k < max_out; ++b) {
        const float v = from_bits(b);
        if (fp::tools::linTodB(v) < rule_db(v)) out[k++] = v;
    }
    return k;
}

// fp::b200::capturesToIRs on captures[batch][n] -> out[batch][irLength]; 0, or -1 when the facade throws
int chop_captures_to_irs(const float* captures, int batch, int n, const float* sweep, int ns, double sr, int irLength, float thr, int cons, int smoothing, float* out) {
    try {
        AudioBuffer<float> c(batch, n), sw(1, ns);
        for (int b = 0; b < batch; ++b) c.copyFrom(b, 0, captures + (long long) b * n, n);
        sw.copyFrom(0, 0, sweep, ns);
        AudioBuffer<float> r = fp::b200::capturesToIRs(c, sw, sr, irLength, thr, cons, smoothing != 0);
        for (int b = 0; b < batch; ++b) std::memcpy(out + (long long) b * irLength, r.getReadPointer(b), sizeof(float) * irLength);
        return 0;
    } catch (const std::exception&) { return -1; }
}

}  // extern "C"
