// rx_stream.cuh -- the per-stream receive state machine on the GPU.
//
// One CTA walks one (channel, SF) stream through the reference's work() state machine
// (lib/decoder_impl.cc:740-903): DETECT -> SYNC -> FIND_SFD -> PAUSE -> DECODE_HEADER ->
// DECODE_PAYLOAD, consuming as many steps as the staged IQ allows (each step needs 2*sps
// items of look-ahead, the block's output_multiple :91).  Symbol n+1's window depends on
// symbol n's d_fine_sync, so the parallelism is across streams (grid) and inside a step
// (256 threads over the sps samples), not across the symbols of one frame.
//
// Phases (each restates one reference function, float stage A3-A11 of SURVEY.md 8a):
//   ifreq_block          instantaneous_frequency            :224-244
//   step DETECT          detect_preamble_autocorr           :340-366
//   step SYNC            sliding_norm_cross_correlate_upchirp :399-413
//   step FIND_SFD        detect_downchirp / cross_correlate_ifreq :385-390,:283-298
//   fine_sync_block      fine_sync                          :300-338
//   demod (gradient)     max_frequency_gradient_idx         :466-491
//   demod (FFT)          get_shift_fft via the K1 phase functions :430-464
// The integer tail (Gray, deinterleave, header parse) runs on thread 0 with int_chain.cuh;
// completed frames are queued for the follow-on K8 kernel.
#pragma once
#include "int_chain.cuh"
#include "k1_fft.cuh"
#include "../../include/lora_b200.h"

namespace lb {

constexpr int RX_THREADS = 256;
constexpr int RX_WARPS = RX_THREADS / 32;

struct RxStreamState {                 // members of decoder_impl, lib/decoder_impl.h:70-123
    int32_t state;
    int32_t payload_symbols;
    uint32_t payload_length;
    uint32_t corr_fails;
    float energy_threshold;
    float snr;
    float pwr_queue[4];                // boost::circular_buffer<float>(MAX_PWR_QUEUE_SIZE)
    int32_t pwr_n, pwr_head;
    uint32_t n_words;
    uint32_t words[8];
    uint32_t n_demod;
    uint32_t frame_seq;
    uint8_t phdr[3];
    uint8_t n_hdr_print;
    uint8_t hdr_print[4];
    uint8_t demodulated[LB_MAX_CW];
    float cfo_est;                     // experimental_determine_cfo at the last SYNC (Hz), only with cfo_estimate enabled
    uint32_t cfo_count;                // how many estimates this stream has produced
};

struct RxFrameRec {                    // one completed frame, input of the K8 kernel
    uint32_t stream, seq, n_cw, cr, payload_length;
    float snr;
    uint8_t phdr[3];
    uint8_t n_hdr_print;
    uint8_t hdr_print[4];
    uint8_t cw[LB_MAX_CW];
};

struct RxFrameOut {                    // output of K8: loratap | phy | payload (msg_lora_frame :588-609)
    uint32_t stream, seq, len;
    uint8_t n_hdr_print;
    uint8_t hdr_print[4];
    uint8_t pad[3];
    uint8_t bytes[LB_MAX_FRAME + 2];
};

struct RxParams {
    const float2 *iq;                  // [n_launch][stride_items]
    size_t stride_items;
    size_t n_items;
    uint32_t stream_base;
    uint32_t n_launch;                 // streams of this launch (rx_warp_kernel packs several per CTA)
    // tables
    const float2 *down;
    const float *down_ifreq, *up_ifreq, *up_ifreq_v;
    const float2 *tw;
    float down_ifreq_avg, down_ifreq_sd;      // over sps-1 entries (:287-289)
    // derived configuration (decoder_impl.cc:69-91)
    uint32_t sps, n_bins, n_bins_hdr, decim, sf;
    int implicit, reduced_rate, enable_fine_sync;
    int cfo_estimate;                  // 1: also run experimental_determine_cfo (:730-738) where the reference has its call commented out (:774)
    float samples_per_second;
    // state / outputs
    RxStreamState *states;
    float *scratch;                    // per stream 2*sps + n_bins floats
    unsigned long long *consumed;      // per stream
    RxFrameRec *frames;
    uint32_t *n_frames;                // global queue counter
    uint32_t frame_cap;
    uint32_t max_frames_per_stream;
    lora_b200_step *trace;
    uint32_t trace_cap;
    uint32_t *trace_n;                 // per stream
    const uint32_t *n_items_s;         // per-stream item counts [stream] (device); nullptr: every stream has n_items
};

// the items stream `stream` may read in this launch (read where it is used rather than held in a register: the kernels
// are at their register budget)
#define LB_RX_N_ITEMS(p, stream) ((p).n_items_s ? (unsigned long long)(p).n_items_s[stream] : (unsigned long long)(p).n_items)

#ifdef __CUDACC__

struct RxShared {
    float red[4][RX_WARPS];
    unsigned long long keys[RX_WARPS];
    float bcast[4];
    unsigned long long kbcast;
    int state;
    int flag;
    int consumed;
    int fine_sync;
    int bin;
    float metric;
    unsigned long long pos;
    unsigned int frames_here;
    unsigned int steps;
    unsigned int frame_slot;
};

LB_D float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// sum of up to 4 values over the CTA; result valid in every thread
template <int NV>
LB_D void block_sum(float (&v)[NV], RxShared &sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NV; k++) {
        const float s = warp_sum(v[k]);
        if (lane == 0) sh.red[k][warp] = s;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < NV; k++) {
            float s = lane < RX_WARPS ? sh.red[k][lane] : 0.0f;
            s = warp_sum(s);
            if (lane == 0) sh.bcast[k] = s;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NV; k++) v[k] = sh.bcast[k];
    __syncthreads();
}

LB_D unsigned long long block_max_key(unsigned long long k, RxShared &sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    k = warp_max_key(k);
    if (lane == 0) sh.keys[warp] = k;
    __syncthreads();
    if (warp == 0) {
        unsigned long long t = lane < RX_WARPS ? sh.keys[lane] : 0ull;
        t = warp_max_key(t);
        if (lane == 0) sh.kbcast = t;
    }
    __syncthreads();
    const unsigned long long r = sh.kbcast;
    __syncthreads();
    return r;
}

// candidate key for "c > max (initially 0), first maximum wins" loops (:311-314, :406-409)
LB_D unsigned long long corr_key(float c, uint32_t idx) { return c > 0.0f ? pack_key(c, idx) : 0ull; }

// A3 instantaneous_frequency (:224-244): out[i-1] = wrap(arg x[i] - arg x[i-1]), out[w-1] = out[w-2]
LB_D void ifreq_block(const float2 *__restrict__ x, float *__restrict__ out, int w) {
    const int lane = threadIdx.x & 31;
    for (int base = 1; base < w; base += RX_THREADS) {
        const int i = base + threadIdx.x;
        const bool active = i < w;
        float p2 = 0.0f;
        if (active) { const float2 s = x[i]; p2 = lb_atan2f(s.y, s.x); }
        float p1 = __shfl_up_sync(0xffffffffu, p2, 1);
        if (lane == 0 && active) { const float2 s = x[i - 1]; p1 = lb_atan2f(s.y, s.x); }
        if (active) {
            // :236-237, float difference against the double M_PI, correction in double
            while (p2 - p1 > LB_PI_BELOW) p2 = (float)((double)p2 - 6.283185307179586);
            while (p2 - p1 < -LB_PI_BELOW) p2 = (float)((double)p2 + 6.283185307179586);
            out[i - 1] = p2 - p1;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) out[w - 1] = out[w - 2];
    __syncthreads();
}

// A6 fine_sync (:300-338); ifreq of the window must already be in scr[0..sps)
// (scr is written earlier in this kernel: it must not be read through the non-coherent path)
LB_D int fine_sync_block(const RxParams &p, const float *scr, int bin_idx, int search, RxShared &sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sps = (int)p.sps;
    const int shift_ref = (bin_idx + 1) * (int)p.decim;           // :301
    const int last = 3 * sps - 1;
    unsigned long long best = 0ull;
    for (int li = warp; li < 2 * search - 1; li += RX_WARPS) {
        const int i = li - (search - 1);                          // lag in (-search, search)
        const int start = shift_ref + i + sps;                    // :310
        float c = 0.0f;
        for (int k = lane; k < sps; k += 32) {
            int idx = start + k;
            idx = idx < 0 ? 0 : (idx > last ? last : idx);        // defined over-read (oracle D1)
            c = fmaf(scr[k], __ldg(p.up_ifreq_v + idx), c);
        }
        c = warp_sum(c);
        const unsigned long long key = corr_key(c, (uint32_t)li);
        best = key > best ? key : best;
    }
    best = block_max_key(best, sh);
    const int lag = best ? (int)key_idx(best) - (search - 1) : 0;
    return -lag;                                                  // :321
}

template <int SF, bool FFT>
__global__ void __launch_bounds__(RX_THREADS)
rx_stream_kernel(RxParams p) {
    extern __shared__ float2 rx_dyn_smem[];
    __shared__ RxShared sh;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t stream = p.stream_base + blockIdx.x;
    const float2 *xs = p.iq + (size_t)blockIdx.x * p.stride_items;
    RxStreamState *st = p.states + stream;
    float *scr = p.scratch + (size_t)stream * (2 * (size_t)p.sps + p.n_bins);
    const int sps = (int)p.sps, N = (int)p.n_bins;
    lora_b200_step *trace = p.trace ? p.trace + (size_t)stream * p.trace_cap : nullptr;

    if (tid == 0) { sh.state = st->state; sh.pos = 0; sh.frames_here = 0; sh.steps = 0; }
    __syncthreads();

    while (true) {
        const unsigned long long pos = sh.pos;
        const int state = sh.state;
        if (pos + 2ull * (unsigned long long)sps > LB_RX_N_ITEMS(p, stream)) break;
        if (sh.frames_here >= p.max_frames_per_stream) break;
        const float2 *x = xs + pos;
        if (tid == 0) { sh.fine_sync = 0; sh.bin = -1; sh.metric = 0.0f; sh.flag = 0; sh.consumed = 0; }   // :749
        __syncthreads();

        switch (state) {
        case LORA_B200_DETECT: {                                  // :752-768, A8 :340-366
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            for (int i = tid; i < sps; i += RX_THREADS) {
                const float2 a = x[i], b = x[i + sps];
                v[0] += a.x * b.x + a.y * b.y;                    // a * conj(b)
                v[1] += a.y * b.x - a.x * b.y;
                v[2] += a.x * a.x + a.y * a.y;
                v[3] += b.x * b.x + b.y * b.y;
            }
            block_sum<4>(v, sh);
            if (tid == 0) {
                st->energy_threshold = v[3] / 2.0f;               // :357
                const float pw = v[2] / (float)p.sps;             // :360 push_back on the 4-deep ring
                if (st->pwr_n < 4) { st->pwr_queue[(st->pwr_head + st->pwr_n) & 3] = pw; st->pwr_n++; }
                else { st->pwr_queue[st->pwr_head] = pw; st->pwr_head = (st->pwr_head + 1) & 3; }
                const float s = sqrtf(v[2] * v[3]);
                const float corr = hypotf(v[0] / s, v[1] / s);    // :363
                sh.metric = corr;
                if (corr >= 0.90f) {                              // :755
                    if (st->pwr_n >= 2)                           // determine_snr :377-383
                        st->snr = st->pwr_queue[(st->pwr_head + st->pwr_n - 1) & 3] / st->pwr_queue[st->pwr_head];
                    st->corr_fails = 0u;
                    sh.state = LORA_B200_SYNC;
                } else {
                    sh.consumed = sps;
                }
            }
            break;
        }
        case LORA_B200_SYNC: {                                    // :770-783, A9 :392-413
            ifreq_block(x, scr, 2 * sps);
            unsigned long long best = 0ull;
            const int wlen = sps - 1;
            // each warp takes 4 consecutive lags at a time so every ideal-chirp value is reused 4x
            for (int i0 = warp * 4; i0 < sps; i0 += RX_WARPS * 4) {
                float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
                for (int k = lane; k < wlen; k += 32) {
                    const float u = __ldg(p.up_ifreq + k);
                    const float *f = scr + i0 + k;
                    c0 = fmaf(f[0], u, c0); c1 = fmaf(f[1], u, c1); c2 = fmaf(f[2], u, c2); c3 = fmaf(f[3], u, c3);
                }
                c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2); c3 = warp_sum(c3);
                unsigned long long k0 = corr_key(c0, i0), k1 = corr_key(c1, i0 + 1), k2 = corr_key(c2, i0 + 2), k3 = corr_key(c3, i0 + 3);
                k0 = k1 > k0 ? k1 : k0; k2 = k3 > k2 ? k3 : k2; k0 = k2 > k0 ? k2 : k0;
                best = k0 > best ? k0 : best;
            }
            best = block_max_key(best, sh);
            if (tid == 0) {
                sh.metric = best ? key_mag2(best) : 0.0f;
                sh.consumed = best ? (int)key_idx(best) : 0;      // :780 consume_each(i)
                sh.state = LORA_B200_FIND_SFD;
                if (p.cfo_estimate && sps > 257) {
                    // experimental_determine_cfo(&input[i], sps) (:730-738, call site :774 commented out in the reference):
                    // instantaneous frequency of samples * downchirp at the hard-coded index 256, in Hz
                    const float2 *xi = x + sh.consumed;
                    const float2 m0 = cmul(xi[256], __ldg(p.down + 256)), m1 = cmul(xi[257], __ldg(p.down + 257));
                    const float p1 = atan2f(m0.y, m0.x);
                    float p2 = atan2f(m1.y, m1.x);
                    while (p2 - p1 > LB_PI_BELOW) p2 = (float)((double)p2 - 6.283185307179586);
                    while (p2 - p1 < -LB_PI_BELOW) p2 = (float)((double)p2 + 6.283185307179586);
                    st->cfo_est = (float)((double)(p2 - p1) / (2.0 * 3.14159265358979323846) * (double)p.samples_per_second);
                    st->cfo_count++;
                }
            }
            break;
        }
        case LORA_B200_FIND_SFD: {                                // :785-818, A10
            ifreq_block(x, scr, sps);
            const int to_idx = sps - 1;
            float v1[1] = {0.f};
            for (int i = tid; i < to_idx; i += RX_THREADS) v1[0] += scr[i];
            block_sum<1>(v1, sh);
            const float average = v1[0] / (float)to_idx;          // :286
            float v2[2] = {0.f, 0.f};
            for (int i = tid; i < to_idx; i += RX_THREADS) {
                const float t = scr[i] - average;
                v2[0] = fmaf(t, t, v2[0]);                        // stddev :415-425
                v2[1] = fmaf(t, __ldg(p.down_ifreq + i) - p.down_ifreq_avg, v2[1]);
            }
            block_sum<2>(v2, sh);
            const float sd = sqrtf(v2[0] / (float)to_idx) * p.down_ifreq_sd;   // :288-289
            const float c = v2[1] / sd / (float)to_idx;           // :291-295
            int fs = 0;
            const bool up_again = !(c > 0.96f) && (c < -0.97f);
            if (up_again) fs = fine_sync_block(p, scr, -1, (int)p.decim * 4, sh);   // :803
            if (tid == 0) {
                sh.metric = c;
                if (c > 0.96f) {
                    sh.state = LORA_B200_PAUSE;                   // :799
                } else {
                    if (!up_again) st->corr_fails++;              // :805
                    if (st->corr_fails > 4u) sh.state = LORA_B200_DETECT;   // :808-813
                }
                sh.fine_sync = fs;
                sh.consumed = sps + fs;                           // :816
            }
            break;
        }
        case LORA_B200_PAUSE: {                                   // :820-824
            if (tid == 0) { sh.state = LORA_B200_DECODE_HEADER; sh.consumed = sps + sps / 4; }
            break;
        }
        case LORA_B200_DECODE_HEADER:
        case LORA_B200_DECODE_PAYLOAD: {                          // :826-886
            const bool is_first = state == LORA_B200_DECODE_HEADER;
            bool do_demod = true;
            if (!is_first && p.implicit) {                        // :861 determine_energy
                float e[1] = {0.f};
                for (int i = tid; i < sps; i += RX_THREADS) { const float2 a = x[i]; e[0] += a.x * a.x + a.y * a.y; }
                block_sum<1>(e, sh);
                if (e[0] < st->energy_threshold) do_demod = false;
            }
            int bin = -1, fs = 0;
            if (do_demod) {                                       // demodulate(), :493-529
                const bool need_ifreq = !FFT || p.enable_fine_sync;
                if (need_ifreq) ifreq_block(x, scr, sps);
                if (FFT) {
                    using C = K1Cfg<SF>;
                    K1Args a{x, p.down, p.tw, 1};
                    unsigned long long best = 0ull;
                    float2 wtab[C::NP / C::TPS];
                    k1_combine_twiddles<SF>(a, tid, wtab);
                    for (int s = 0; s < C::S; s++) {
                        k1_pass0<SF, false>(a, 0, s, tid, rx_dyn_smem);
                        __syncthreads();
                        k1_pass<SF, C::R1, C::SIG1>(a, tid, rx_dyn_smem);
                        __syncthreads();
                        if (C::R2 > 1) { k1_pass<SF, (C::R2 > 1 ? C::R2 : 2), 1>(a, tid, rx_dyn_smem); __syncthreads(); }
                        unsigned long long k = tid < C::TPS ? k1_combine<SF>(a, s, tid, rx_dyn_smem, wtab) : 0ull;
                        best = k > best ? k : best;
                        __syncthreads();
                    }
                    best = block_max_key(best, sh);
                    bin = ((int)key_idx(best) + N - 1) % N;       // gradient-index convention (SURVEY A7)
                } else {                                          // A5 :466-491
                    float *avg = scr + 2 * sps;
                    const int decim = (int)p.decim;
                    for (int i = tid; i < N; i += RX_THREADS) {
                        float acc = 0.0f;
                        for (int k = 0; k < decim; k++) acc += scr[i * decim + k];   // :475
                        avg[i] = acc / (float)decim;              // :476
                    }
                    __syncthreads();
                    unsigned long long best = 0ull;
                    for (int i = 1 + tid; i < N; i += RX_THREADS) {
                        const float g = avg[i - 1] - avg[i];      // :483
                        if (g > 0.1f) { const unsigned long long k = pack_key(g, (uint32_t)i); best = k > best ? k : best; }
                    }
                    best = block_max_key(best, sh);
                    const int max_index = best ? (int)key_idx(best) + 1 : 0;   // :486
                    bin = (N - max_index) % N;                    // :490
                }
                if (p.enable_fine_sync) {                         // :501-502
                    int s = (int)p.decim / 4; if (s < 2) s = 2;
                    fs = fine_sync_block(p, scr, bin, s, sh);
                }
            }
            if (tid == 0) {
                bool block_done = false;
                uint32_t cr = st->phdr[1] >> 5;
                if (do_demod) {
                    const bool reduced = is_first || p.reduced_rate;      // :495
                    uint32_t b = (uint32_t)bin;
                    if (reduced) b = reduce_bin(b, p.n_bins_hdr);  // :507-509
                    st->words[st->n_words++] = gray_encode(b);    // :512,:517
                    if (st->n_words == 4u + (is_first ? 4u : cr)) {       // :521
                        const uint32_t ppm = reduced ? p.sf - 2u : p.sf;
                        uint8_t cwb[16];
                        deinterleave_block(st->words, st->n_words, ppm, cwb);
                        for (uint32_t k = 0; k < ppm; k++)
                            if (st->n_demod < (uint32_t)LB_MAX_CW) st->demodulated[st->n_demod++] = cwb[k];
                        st->n_words = 0;
                        block_done = true;
                    }
                } else {
                    st->payload_symbols = 0;                      // :862-864
                    st->payload_length = st->n_demod / 2u;
                }
                if (is_first) {
                    if (block_done) {
                        if (p.implicit) {
                            st->payload_symbols = 1;              // :829
                        } else {
                            const uint32_t nb = decode_len_bytes(6u, cr);            // decode(true) :831
                            uint8_t hb[4] = {0, 0, 0, 0};
                            for (uint32_t k = 0; k < nb && k < 4u; k++) hb[k] = decode_byte(st->demodulated, st->n_demod, 1, cr, k);
                            st->n_hdr_print = (uint8_t)(nb < 4u ? nb : 4u);          // :832 prints d_decoded
                            for (int k = 0; k < 4; k++) st->hdr_print[k] = hb[k];
                            const uint32_t erase = st->n_demod < 5u ? st->n_demod : 5u;   // :632
                            for (uint32_t k = erase; k < st->n_demod; k++) st->demodulated[k - erase] = st->demodulated[k];
                            st->n_demod -= erase;
                            st->phdr[0] = hb[0]; st->phdr[1] = hb[1]; st->phdr[2] = hb[2];   // :833
                            if ((st->phdr[1] >> 5) > 4) st->phdr[1] = (uint8_t)((st->phdr[1] & 0x1f) | (4u << 5));   // :834-835
                            cr = st->phdr[1] >> 5;
                            st->payload_length = st->phdr[0] + 2u * ((st->phdr[1] >> 4) & 1u);   // :838
                            st->payload_symbols = payload_symbols(st->payload_length, cr, p.sf, p.reduced_rate);
                        }
                        sh.state = LORA_B200_DECODE_PAYLOAD;      // :853
                    }
                } else {
                    if (block_done && !p.implicit) st->payload_symbols -= (int32_t)(4u + cr);   // :866-867
                    if (st->payload_symbols <= 0) {               // :870
                        sh.flag = 1;
                        sh.frame_slot = atomicAdd(p.n_frames, 1u);
                    }
                }
                sh.bin = bin;
                sh.fine_sync = fs;
                sh.consumed = sps + fs;                           // :856,:883
            }
            __syncthreads();
            if (sh.flag) {                                        // decode(false) + msg_lora_frame happen in K8
                const uint32_t slot = sh.frame_slot;
                if (slot < p.frame_cap) {
                    RxFrameRec *fr = p.frames + slot;
                    const uint32_t n = st->n_demod;
                    for (uint32_t k = tid; k < n; k += RX_THREADS) fr->cw[k] = st->demodulated[k];
                    if (tid == 0) {
                        fr->stream = stream; fr->seq = st->frame_seq++; fr->n_cw = n; fr->cr = st->phdr[1] >> 5;
                        fr->payload_length = st->payload_length; fr->snr = st->snr;
                        fr->phdr[0] = st->phdr[0]; fr->phdr[1] = st->phdr[1]; fr->phdr[2] = st->phdr[2];
                        fr->n_hdr_print = p.implicit ? 0 : st->n_hdr_print;
                        for (int k = 0; k < 4; k++) fr->hdr_print[k] = st->hdr_print[k];
                    }
                }
                __syncthreads();
                if (tid == 0) {
                    sh.state = LORA_B200_DETECT;                  // :875-880
                    st->n_words = 0; st->n_demod = 0;
                    sh.frames_here++;
                }
            }
            break;
        }
        default: {                                                // STOP :888-891
            if (tid == 0) sh.consumed = sps;
            break;
        }
        }
        __syncthreads();
        if (tid == 0) {
            if (trace && sh.steps < p.trace_cap) {
                lora_b200_step t;
                t.state = state; t.consumed = sh.consumed; t.bin = sh.bin; t.fine_sync = sh.fine_sync; t.metric = sh.metric;
                trace[sh.steps] = t;
            }
            sh.steps++;
            sh.pos = pos + (unsigned long long)(sh.consumed > 0 ? sh.consumed : 0);
        }
        __syncthreads();
    }
    if (tid == 0) {
        st->state = sh.state;
        p.consumed[stream] = sh.pos;
        if (p.trace_n) p.trace_n[stream] = sh.steps;
    }
}

// K2 batch: max_frequency_gradient_idx on aligned windows (parity entry point for A5)
__global__ void __launch_bounds__(RX_THREADS)
k2_gradient_kernel(const float2 *__restrict__ iq, size_t n_symbols, uint32_t sps, uint32_t n_bins, uint32_t decim,
                   float *__restrict__ scratch /* gridDim.x * (sps + n_bins) */, uint32_t *__restrict__ bins) {
    __shared__ RxShared sh;
    float *scr = scratch + (size_t)blockIdx.x * (sps + n_bins);
    float *avg = scr + sps;
    for (size_t sym = blockIdx.x; sym < n_symbols; sym += gridDim.x) {
        ifreq_block(iq + sym * sps, scr, (int)sps);
        for (int i = threadIdx.x; i < (int)n_bins; i += RX_THREADS) {
            float acc = 0.0f;
            for (uint32_t k = 0; k < decim; k++) acc += scr[i * decim + k];
            avg[i] = acc / (float)decim;
        }
        __syncthreads();
        unsigned long long best = 0ull;
        for (int i = 1 + threadIdx.x; i < (int)n_bins; i += RX_THREADS) {
            const float g = avg[i - 1] - avg[i];
            if (g > 0.1f) { const unsigned long long k = pack_key(g, (uint32_t)i); best = k > best ? k : best; }
        }
        best = block_max_key(best, sh);
        if (threadIdx.x == 0) {
            const int max_index = best ? (int)key_idx(best) + 1 : 0;
            bins[sym] = (uint32_t)(((int)n_bins - max_index) % (int)n_bins);
        }
        __syncthreads();
    }
}

// K8: decode(false) + msg_lora_frame for every queued frame (B2-B4, B7)
__global__ void __launch_bounds__(128)
k8_frames_kernel(const RxFrameRec *__restrict__ frames, const uint32_t *__restrict__ n_frames, uint32_t cap,
                 RxFrameOut *__restrict__ out) {
    uint32_t n = *n_frames;
    if (n > cap) n = cap;
    for (uint32_t f = blockIdx.x; f < n; f += gridDim.x) {
        const RxFrameRec *fr = frames + f;
        RxFrameOut *o = out + f;
        const uint32_t cr = fr->cr, n_cw = fr->n_cw;
        const uint32_t n_dec = decode_len_bytes(decode_len_words(n_cw, 0), cr);
        uint32_t plen = fr->payload_length;
        if (plen > (uint32_t)LB_MAX_FRAME - 18u) plen = (uint32_t)LB_MAX_FRAME - 18u;
        for (uint32_t i = threadIdx.x; i < plen; i += blockDim.x)
            o->bytes[18 + i] = i < n_dec ? decode_byte(fr->cw, n_cw, 0, cr, i) : 0;   // missing bytes read 0 (oracle D5)
        if (threadIdx.x < 15) {
            uint8_t b = 0;
            if (threadIdx.x == 13) {                              // loratap rssi.snr, :597
                const double v = (double)(10.0f * log10f(fr->snr)) + 0.5;
                b = (uint8_t)(int32_t)v;
            }
            o->bytes[threadIdx.x] = b;
        }
        if (threadIdx.x < 3) o->bytes[15 + threadIdx.x] = fr->phdr[threadIdx.x];   // :600
        if (threadIdx.x == 0) {
            o->stream = fr->stream; o->seq = fr->seq; o->len = 18u + plen;
            o->n_hdr_print = fr->n_hdr_print;
            for (int k = 0; k < 4; k++) o->hdr_print[k] = fr->hdr_print[k];
        }
    }
}

// K8 generic entry: decode() on arbitrary code-word vectors (parity tests for B2-B4)
__global__ void __launch_bounds__(128)
k8_decode_vectors_kernel(const uint8_t *__restrict__ cw, const uint32_t *__restrict__ lengths, size_t stride,
                         const uint8_t *__restrict__ cr, const uint8_t *__restrict__ is_header, size_t n_vec,
                         uint8_t *__restrict__ out, size_t out_stride, uint32_t *__restrict__ out_len) {
    for (size_t v = blockIdx.x; v < n_vec; v += gridDim.x) {
        const uint32_t n = lengths[v], c = cr[v];
        const int hdr = is_header[v] != 0;
        uint32_t nb = decode_len_bytes(decode_len_words(n, hdr), c);
        if (nb > out_stride) nb = (uint32_t)out_stride;
        for (uint32_t i = threadIdx.x; i < nb; i += blockDim.x) out[v * out_stride + i] = decode_byte(cw + v * stride, n, hdr, c, i);
        if (threadIdx.x == 0) out_len[v] = nb;
    }
}

// B1 batch: Gray-coded words of whole interleaver blocks -> code words
__global__ void k8_deinterleave_kernel(const uint32_t *__restrict__ words, uint32_t n_words, uint32_t ppm,
                                       size_t n_blocks, uint8_t *__restrict__ cw) {
    const size_t b = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    uint32_t w[8];
    uint8_t o[16];
    for (uint32_t i = 0; i < n_words && i < 8u; i++) w[i] = words[b * n_words + i];
    deinterleave_block(w, n_words < 8u ? n_words : 8u, ppm, o);
    for (uint32_t x = 0; x < ppm; x++) cw[b * ppm + x] = o[x];
}

#endif  // __CUDACC__
}  // namespace lb
