// Host side of the real-output polyphase synthesis filter bank (b200c_rsynth, rsynth.cu).  It keeps its state in a
// SynthPlan (synth.hpp): taps, twiddles and tile shape have the complex synthesizer's layout, so synth_plan_destroy
// serves both and rsynth_set_taps uploads through synth_set_taps.
#pragma once
#include <cstddef>
#include <cstdint>

#include "synth.hpp"

namespace b200c {

constexpr size_t kRSynthMaxBranches = 8192;   // M: an M/2 = 4096-point complex inverse transform per frame

// M-point twiddle table and chunk shape; smem_optin = the device's opt-in shared memory per block
int rsynth_plan_create(SynthPlan &p, size_t m, size_t interp, size_t smem_optin);
// uploads the taps (blocking) and sizes the tile and bin group for K; 1 <= ntaps <= min(16 M, 32 D) is checked by the
// caller
int rsynth_set_taps(SynthPlan &p, const double *taps, size_t ntaps);
// frames F >= 1 output frames (F D samples); dtype B200C_F32 or B200C_I16 (the output); d_in: rows 0 .. M/2;
// stream_index = absolute stream index of d_out[0]
int rsynth_launch(const SynthPlan &p, int dtype, const void *d_in, size_t in_stride, size_t frames, uint64_t stream_index,
                  void *d_out, cudaStream_t stream);

} // namespace b200c
