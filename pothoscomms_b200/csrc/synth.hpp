// Host-side plan of one polyphase synthesis filter bank (b200c_synth, synth.cu).
#pragma once
#include <cstddef>
#include <cstdint>

#include "common.hpp"

namespace b200c {

constexpr size_t kSynthMaxChannels = 4096;
constexpr size_t kSynthMaxTapsPerPhase = 32;   // ntaps <= 32 D: at most 32 input frames per output sample
constexpr size_t kSynthMaxTapsPerChannel = 16; // ntaps <= 16 M

struct SynthPlan {
    int M = 0, logM = 0, D = 1, logD = 0;
    size_t ntaps = 1;
    int K = 1;                 // frames per output sample, ceil(ntaps / D)
    float *d_taps = nullptr;   // [K][D] prototype taps (float32): g zero-padded to K D
    size_t taps_capacity = 0;  // bytes
    void *d_tw = nullptr;      // [M] float2 exp(-2 pi i k / M)
    int P = 1;                 // frames per shared-memory chunk (power of two)
    int B = 1;                 // bins (= threads that own an output phase) per CTA
    int T = 1;                 // output frames per CTA
    size_t smem_bytes = 0;
};

// twiddle table and chunk shape; smem_optin = the device's opt-in shared memory per block
int synth_plan_create(SynthPlan &p, size_t nchan, size_t interp, size_t smem_optin);
void synth_plan_destroy(SynthPlan &p);
// uploads the taps (blocking) and sizes the tile for K; 1 <= ntaps <= min(16 M, 32 D) is checked by the caller
int synth_set_taps(SynthPlan &p, const double *taps, size_t ntaps);
// frames F >= 1 output frames (F D samples); stream_index = absolute stream index of d_out[0]
int synth_launch(const SynthPlan &p, const void *d_in, size_t in_stride, size_t frames, uint64_t stream_index, void *d_out,
                 cudaStream_t stream);

} // namespace b200c
