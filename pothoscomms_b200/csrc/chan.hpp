// Host-side plan of one polyphase filter-bank channelizer (b200c_chan, chan.cu).
#pragma once
#include <cstddef>
#include <cstdint>

#include "common.hpp"

namespace b200c {

constexpr size_t kChanMaxChannels = 4096;
constexpr size_t kChanMaxTapsPerBranch = 16;   // ntaps <= 16 * M: at most 16 prototype taps per polyphase branch

struct ChanPlan {
    int M = 0, logM = 0, D = 1;
    size_t ntaps = 1;
    int R = 1;                 // taps per branch, ceil(ntaps / M)
    float *d_taps = nullptr;   // [R][M] prototype taps (float32), zero beyond ntaps
    size_t taps_capacity = 0;  // bytes
    void *d_tw = nullptr;      // [M] float2 exp(-2 pi i k / M)
    int T = 4;                 // frames per CTA (power of two)
    size_t smem_bytes = 0;
};

// twiddle table and tile shape; smem_optin = the device's opt-in shared memory per block
int chan_plan_create(ChanPlan &p, size_t nchan, size_t decim, size_t smem_optin);
void chan_plan_destroy(ChanPlan &p);
// uploads the taps (blocking); 1 <= ntaps <= 16 M is checked by the caller
int chan_set_taps(ChanPlan &p, const double *taps, size_t ntaps);
// frames F >= 1 output frames; stream_index = absolute index of d_in[0]
int chan_launch(const ChanPlan &p, const void *d_in, size_t frames, uint64_t stream_index, void *d_out, size_t out_stride,
                cudaStream_t stream);

} // namespace b200c
