// Host side of the real-input polyphase filter-bank channelizer (b200c_rchan, rchan.cu).  It keeps its state in a
// ChanPlan (chan.hpp): taps, twiddles and tile shape have the complex channelizer's layout, so chan_set_taps and
// chan_plan_destroy serve both.
#pragma once
#include <cstddef>
#include <cstdint>

#include "chan.hpp"

namespace b200c {

constexpr size_t kRChanMaxBranches = 8192;   // M: an M/2 = 4096-point complex transform per frame

// M-point twiddle table and tile shape; smem_optin = the device's opt-in shared memory per block
int rchan_plan_create(ChanPlan &p, size_t m, size_t decim, size_t smem_optin);
// frames F >= 1; dtype B200C_F32 or B200C_I16; stream_index = absolute index of d_in[0]; rows 0 .. M/2 of d_out
int rchan_launch(const ChanPlan &p, int dtype, const void *d_in, size_t frames, uint64_t stream_index, void *d_out,
                 size_t out_stride, cudaStream_t stream);

} // namespace b200c
