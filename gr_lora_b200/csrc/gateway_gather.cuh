// gateway_gather.cuh -- how the gateway (gateway.cu) hands channelizer output to decoders that consume unequal amounts.
//
// Each SF's decoder owns two buffers B[n_ch][cap] and alternates between them.  After a call, stream ch of one SF has
// consumed `consumed` of its `len` items; the `pending = len - consumed` it left over (always < 2 sps unless the stream
// stopped at max_frames_per_call) must be presented again, followed by the channelizer's M new items:
//   next[ch][i] = prev[ch][consumed + i]   for i <  pending
//               = O[ch][i - pending]       for pending <= i < pending + M
// The index map and the bookkeeping are __host__ __device__ so that the CPU tests run the same code (host_emul.cu).
#pragma once
#include "lora_common.cuh"

namespace lb {

// where next[i] comes from: returns the index into prev (from_prev = 1) or into O (from_prev = 0)
LB_HD uint32_t gw_src(uint32_t i, uint32_t consumed, uint32_t pending, int *from_prev) {
    *from_prev = i < pending;
    return i < pending ? consumed + i : i - pending;
}

// After a call that consumed `consumed` of `len` items: the tail left over.  Then, before the next call brings m items:
// the length the stream will have, or 0 with *overflow = 1 when pending + m would not fit `cap` (nothing may be written).
LB_HD uint32_t gw_pending(uint32_t len, uint32_t consumed) { return consumed < len ? len - consumed : 0u; }
LB_HD uint32_t gw_next_len(uint32_t pending, uint32_t m, uint32_t cap, int *overflow) {
    const unsigned long long n = (unsigned long long)pending + m;
    *overflow = n > cap;
    return n > cap ? 0u : (uint32_t)n;
}

#ifdef __CUDACC__
// One launch for every SF (blockIdx.z) and channel (blockIdx.y): next = prev[consumed, len) ++ O[0, M), O read once per
// SF.  A thread writes one aligned pair of samples (float4; rows start 16-byte aligned because cap is even) and reads the
// two float2 it is made of, so a warp reads 512 contiguous bytes whatever the parity of `pending`.
struct GwGatherArgs {
    const float2 *out;                   // channelizer output [n_ch][o_stride]
    size_t o_stride;
    uint32_t m;                          // new items per channel
    uint32_t cap;                        // row stride of the decoder buffers (even)
    const float2 *prev[6];               // per SF slot: the buffer of the previous call [n_ch][cap]
    float2 *next[6];                     //              and the one for this call
    const uint32_t *consumed[6];         //              [n_ch] offsets of the pending tails in prev (device)
    const uint32_t *pending[6];          //              [n_ch]
};

__global__ void __launch_bounds__(256) gw_gather_kernel(GwGatherArgs a) {
    const uint32_t z = blockIdx.z, ch = blockIdx.y;
    const uint32_t consumed = a.consumed[z][ch], pending = a.pending[z][ch];
    const float2 *prev = a.prev[z] + (size_t)ch * a.cap;
    float2 *next = a.next[z] + (size_t)ch * a.cap;
    const float2 *o = a.out + (size_t)ch * a.o_stride;
    const uint32_t n = pending + a.m;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; 2 * j < n; j += gridDim.x * blockDim.x) {
        const uint32_t i = 2 * j;
        int fp;
        uint32_t s = gw_src(i, consumed, pending, &fp);
        const float2 v0 = fp ? prev[s] : o[s];
        if (i + 1 < n) {
            s = gw_src(i + 1, consumed, pending, &fp);
            const float2 v1 = fp ? prev[s] : o[s];
            reinterpret_cast<float4 *>(next)[j] = make_float4(v0.x, v0.y, v1.x, v1.y);
        } else {
            next[i] = v0;
        }
    }
}
#endif

}  // namespace lb
