// rx_internal.h -- what the gateway (gateway.cu) uses of a decoder beyond the public C ABI.  Internal to liblora_b200.so:
// none of this is declared in include/lora_b200.h.
#pragma once
#include "../../include/lora_b200.h"
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

// stores the message lora_b200_last_error() returns and gives back `code`
int lb_fail(int code, const char *fmt, ...);

// Launch step: the state machine of every stream of `d` over iq[stream][0, n_items_s[stream]) (row stride `stride_items`;
// n_items_s is a device array), on the decoder's own CUDA stream after `ready` has been reached; `done` is recorded
// behind it.  Asynchronous.
int lb_rx_launch_streams(lora_b200_decoder *d, const float2 *iq, size_t stride_items, const uint32_t *n_items_s,
                         cudaEvent_t ready, cudaEvent_t done);
// Finish step: waits for the launch, decodes the queued frames (K8), consumed[stream] = items consumed in this call; the
// frames are then what lora_b200_frames_last returns.
int lb_rx_finish_streams(lora_b200_decoder *d, size_t *consumed);
