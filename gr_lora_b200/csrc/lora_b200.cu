// lora_b200.cu -- C-ABI implementation of liblora_b200.so (see include/lora_b200.h).
// Host side: parameter derivation and table construction exactly as the reference's
// constructor does them (lib/decoder_impl.cc:49-122,141-175), device memory, streams,
// pinned staging and kernel launches.  There is no CPU compute path in this file.
#include "../../include/lora_b200.h"
#include "k1_fft.cuh"
#include "k1_warp.cuh"
#include "k1_group.cuh"
#include "k1_sf10.cuh"
#include "rx_stream.cuh"
#include "rx_warp.cuh"
#include "tx_channel.cuh"
#include "k1_rows.h"
#include "k1_packed.h"
#include "rx_internal.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <vector>

using namespace lb;

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) return fail(LORA_B200_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

struct Tables {          // offsets (bytes) inside the device blob, see lora_b200_tables_bytes
    size_t down, up, down_ifreq, up_ifreq, up_ifreq_v, tw, total;
};

// Scratch of one K1 launch in flight: the 64-bit argmax keys that the split kernels merge with atomicMax and the
// L2-resident exchange image + flags of the team kernels.  A launch zeroes it on its stream first, so two launches that
// share one K1Scratch must not overlap: slot 0 (lora_b200_demod_fft_dev) is ordered across user streams by `done`,
// and every slot of the host pipeline (lora_b200_demod_fft_host) owns its own.
struct K1Scratch {
    unsigned long long *packed = nullptr;
    size_t packed_cap = 0;
    void *xs = nullptr;
    size_t xs_cap = 0;
    cudaEvent_t done = nullptr;
    cudaStream_t last = nullptr;
    bool used = false;
};

}  // namespace

struct lora_b200_decoder {
    lora_b200_config cfg;
    // derived, decoder_impl.cc:69-91
    uint32_t samples_per_second, sps, n_bins, n_bins_hdr, decim, delay_after_sync;
    double dt, symbols_per_second, bits_per_second, bits_per_symbol;
    bool k1_ok;                           // fs/bw == 8 and SF7..12: FFT kernels usable
    int device, n_sms;
    Tables toff;
    uint8_t *d_tables = nullptr;
    std::vector<uint8_t> h_tables;
    float down_ifreq_avg = 0.f, down_ifreq_sd = 0.f;
    // K1
    K1Scratch k1s[3];                     // [0] device entry point, [1], [2] host pipeline slots
    float *d_k2_scratch = nullptr;
    int k2_grid = 0;
    // e2e host path
    cudaStream_t copy_streams[2] = {nullptr, nullptr};
    void *d_chunk[2] = {nullptr, nullptr};
    void *d_chunk16[2] = {nullptr, nullptr};
    void *h_chunk[2] = {nullptr, nullptr};
    uint32_t *d_chunk_bins[2] = {nullptr, nullptr};
    float *d_chunk_mags[2] = {nullptr, nullptr};
    size_t chunk_symbols = 0;
    // stream path
    cudaStream_t rx_stream = nullptr, rx_stream2 = nullptr;
    cudaEvent_t rx2_done = nullptr, rx_begin_ev = nullptr;
    RxStreamState *d_states = nullptr;
    uint8_t phdr1_init = 0;
    float *d_scratch = nullptr;
    unsigned long long *d_consumed = nullptr;
    RxFrameRec *d_frames = nullptr;
    RxFrameOut *d_frames_out = nullptr;
    uint32_t *d_n_frames = nullptr;
    uint32_t frame_cap = 0;
    lora_b200_step *d_trace = nullptr;
    uint32_t *d_trace_n = nullptr;
    float2 *d_stage = nullptr;            // [n_streams][max_items]
    short2 *d_stage16 = nullptr;          // same shape, int16 I/Q ingest (lora_b200_work_batch_sc16)
    std::vector<cudaEvent_t> stage_events;
    float2 *h_stage = nullptr;            // pinned, same shape
    size_t stage_cap = 0;                 // items
    std::vector<unsigned long long> h_consumed;
    RxFrameOut *h_frames = nullptr;           // pinned, frame_cap records
    std::vector<RxFrameOut> h_sorted;
    std::vector<std::string> stdout_last;
    uint64_t launches = 0;
    bool cfo_estimate = false;            // lora_b200_set_cfo_estimate
};

namespace {

// ---- table construction (host, float phase + sincosf exactly like gr_expj) ---------------
void ifreq_host(const float2 *in, float *out, uint32_t window) {     // decoder_impl.cc:224-244
    for (uint32_t i = 1u; i < window; i++) {
        const float p1 = atan2f(in[i - 1].y, in[i - 1].x);
        float p2 = atan2f(in[i].y, in[i].x);
        while ((p2 - p1) > M_PI) p2 = (float)(p2 - 2.0f * M_PI);
        while ((p2 - p1) < -M_PI) p2 = (float)(p2 + 2.0f * M_PI);
        out[i - 1] = p2 - p1;
    }
    out[window - 1] = out[window - 2];
}

void build_tables(lora_b200_decoder *d) {
    const uint32_t sps = d->sps;
    Tables &t = d->toff;
    size_t o = 0;
    t.down = o; o += sizeof(float2) * sps;
    t.up = o; o += sizeof(float2) * sps;
    t.down_ifreq = o; o += sizeof(float) * sps;
    t.up_ifreq = o; o += sizeof(float) * sps;
    t.up_ifreq_v = o; o += sizeof(float) * sps * 3;
    t.tw = o; o += sizeof(float2) * sps;
    t.total = (o + 255) & ~(size_t)255;
    d->h_tables.assign(t.total, 0);
    float2 *down = (float2 *)(d->h_tables.data() + t.down);
    float2 *up = (float2 *)(d->h_tables.data() + t.up);
    float *dif = (float *)(d->h_tables.data() + t.down_ifreq);
    float *uif = (float *)(d->h_tables.data() + t.up_ifreq);
    float *uifv = (float *)(d->h_tables.data() + t.up_ifreq_v);
    float2 *tw = (float2 *)(d->h_tables.data() + t.tw);

    const double T = -0.5 * d->cfg.bandwidth * d->symbols_per_second;    // :149
    const double f0 = d->cfg.bandwidth / 2.0;                            // :150
    const double pre_dir = 2.0 * M_PI;
    for (uint32_t i = 0; i < sps; i++) {
        const double tt = d->dt * i;                                     // :158
        const float ph_d = (float)(pre_dir * tt * (f0 + T * tt));        // gr_expj(float), :159
        const float ph_u = (float)(pre_dir * tt * (f0 + T * tt) * -1.0f);    // :160
        const float cd = cosf(ph_d), sd = sinf(ph_d), cu = cosf(ph_u), su = sinf(ph_u);
        down[i] = make_float2(cd - sd, sd + cd);                         // (1+1j) * e^{j phase}
        up[i] = make_float2(cu - su, su + cu);
    }
    ifreq_host(down, dif, sps);                                          // :164
    ifreq_host(up, uif, sps);                                            // :165
    std::vector<float2> tmp(3 * (size_t)sps);
    for (int k = 0; k < 3; k++) memcpy(tmp.data() + (size_t)k * sps, up, sizeof(float2) * sps);   // :171-173
    ifreq_host(tmp.data(), uifv, 3 * sps);                               // :174
    for (uint32_t j = 0; j < sps; j++) {                                 // forward DFT twiddles W_sps^j
        const double a = -2.0 * M_PI * (double)j / (double)sps;
        tw[j] = make_float2((float)cos(a), (float)sin(a));
    }
}

void table_stats(lora_b200_decoder *d) {     // chirp_avg and stddev of the ideal down-chirp, :287-289
    const float *dif = (const float *)(d->h_tables.data() + d->toff.down_ifreq);
    const uint32_t to_idx = d->sps - 1u;
    float acc = 0.0f;
    for (uint32_t i = 0; i < to_idx; i++) acc += dif[i];
    const float avg = acc / (float)to_idx;
    float var = 0.0f;
    for (uint32_t i = 0; i < to_idx; i++) { const float t = dif[i] - avg; var += t * t; }
    var /= (float)to_idx;
    d->down_ifreq_avg = avg;
    d->down_ifreq_sd = sqrtf(var);
}

template <typename T>
const T *tab(const lora_b200_decoder *d, size_t off) { return (const T *)(d->d_tables + off); }

// ---- K1 launch -----------------------------------------------------------------------------
template <int SF>
int launch_k1(lora_b200_decoder *d, K1Scratch &ks, const float2 *iq, size_t n_symbols, uint32_t *bins, float *mags, cudaStream_t st) {
    using C = K1Cfg<SF>;
    static bool attr_set[64] = {};
    const size_t smem = sizeof(float2) * C::SMEM_ELEMS;
    if (!attr_set[d->device & 63]) {
        CU(cudaFuncSetAttribute(k1_fft_kernel<SF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[d->device & 63] = true;
    }
    K1Args a{iq, tab<float2>(d, d->toff.down), tab<float2>(d, d->toff.tw), n_symbols};
    const size_t n_work = ((n_symbols + C::G - 1) / C::G) * C::S;
    const int grid = (int)std::min<size_t>(n_work, (size_t)d->n_sms * 2);
    if (C::S > 1) {
        if (ks.packed_cap < n_symbols) {
            if (ks.packed) cudaFree(ks.packed);
            ks.packed = nullptr; ks.packed_cap = 0;
            CU(cudaMalloc(&ks.packed, sizeof(unsigned long long) * n_symbols));
            ks.packed_cap = n_symbols;
        }
        CU(cudaMemsetAsync(ks.packed, 0, sizeof(unsigned long long) * n_symbols, st));
    }
    k1_fft_kernel<SF><<<grid, K1_THREADS, smem, st>>>(a, bins, mags, ks.packed);
    d->launches++;
    if (C::S > 1) {
        k1_finalize_kernel<<<(unsigned)((n_symbols + 255) / 256), 256, 0, st>>>(ks.packed, n_symbols, bins, mags);
        d->launches++;
    }
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

// SF8: a group of 2 warps per symbol (k1_group.cuh; the SF7 warp kernel and the SF9 group kernel are launched from k1_packed.cu)
template <int SF, int NGROUPS, int NSLOT>
int launch_k1_group(lora_b200_decoder *d, K1Scratch &ks, const float2 *iq, size_t n_symbols, uint32_t *bins, float *mags, cudaStream_t st) {
    static bool attr_set[64] = {};
    const size_t smem = sizeof(GSmem<SF, NGROUPS, NSLOT>);
    if (!attr_set[d->device & 63]) {
        CU(cudaFuncSetAttribute(k1_group_kernel<SF, NGROUPS, NSLOT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[d->device & 63] = true;
    }
    K1Args a{iq, tab<float2>(d, d->toff.down), tab<float2>(d, d->toff.tw), n_symbols};
    const int grid = (int)std::min<size_t>((n_symbols + NGROUPS - 1) / NGROUPS, (size_t)d->n_sms);
    k1_group_kernel<SF, NGROUPS, NSLOT><<<grid, NGROUPS * GCfg<SF>::T, smem, st>>>(a, bins, mags);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

// SF10: one 256-thread group per symbol, two radix-32 passes (k1_sf10.cuh)
int launch_k1_sf10(lora_b200_decoder *d, K1Scratch &ks, const float2 *iq, size_t n_symbols, uint32_t *bins, float *mags, cudaStream_t st) {
    static bool attr_set[64] = {};
    const size_t smem = sizeof(S10Smem<3>);
    if (!attr_set[d->device & 63]) {
        CU(cudaFuncSetAttribute(k1_sf10_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[d->device & 63] = true;
    }
    K1Args a{iq, tab<float2>(d, d->toff.down), tab<float2>(d, d->toff.tw), n_symbols};
    const int grid = (int)std::min<size_t>(n_symbols, (size_t)d->n_sms);
    k1_sf10_kernel<3><<<grid, S10_T, smem, st>>>(a, bins, mags);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

// SF11 / SF12: every sample stays inside one SM (k1_rows.cuh; SF12 = cluster of two CTAs per symbol); own translation unit
int launch_k1_rows(lora_b200_decoder *d, K1Scratch &ks, const float2 *iq, size_t n_symbols, uint32_t *bins, float *mags, cudaStream_t st) {
    const int sf = d->cfg.sf;
    if (sf == 12) {
        if (ks.packed_cap < n_symbols) {
            if (ks.packed) cudaFree(ks.packed);
            ks.packed = nullptr; ks.packed_cap = 0;
            CU(cudaMalloc(&ks.packed, sizeof(unsigned long long) * n_symbols));
            ks.packed_cap = n_symbols;
        }
        CU(cudaMemsetAsync(ks.packed, 0, sizeof(unsigned long long) * n_symbols, st));
    }
    char err[256] = {0};
    const int rc = k1_rows_launch(sf, d->device, d->n_sms, iq, tab<float2>(d, d->toff.down), tab<float2>(d, d->toff.tw),
                                  (const float2 *)(d->h_tables.data() + d->toff.tw), n_symbols, bins, mags, ks.packed, st, err, sizeof err);
    if (rc) return fail(LORA_B200_ECUDA, "k1_rows: %s", err);
    d->launches++;
    if (sf == 12) {
        k1_finalize_kernel<<<(unsigned)((n_symbols + 255) / 256), 256, 0, st>>>(ks.packed, n_symbols, bins, mags);
        d->launches++;
        CU(cudaGetLastError());
    }
    return LORA_B200_OK;
}

// SF7 / SF9: the warp / group kernels built with the packed complex product (k1_packed.cu)
int launch_k1_packed(lora_b200_decoder *d, const float2 *iq, size_t n_symbols, uint32_t *bins, float *mags, cudaStream_t st) {
    char err[256] = {0};
    const int rc = k1_packed_launch(d->cfg.sf, d->device, d->n_sms, iq, tab<float2>(d, d->toff.down), tab<float2>(d, d->toff.tw), n_symbols,
                                    bins, mags, st, err, sizeof err);
    if (rc) return fail(LORA_B200_ECUDA, "k1_packed: %s", err);
    d->launches++;
    return LORA_B200_OK;
}

// LORA_B200_K1=generic selects k1_fft_kernel (the CTA-wide kernel the stream state machine also uses) for every SF;
// LORA_B200_K1_ROWS=0 does the same for SF11 / SF12 only.  Both exist for A/B runs (tools/k1_ab.py); the defaults are the
// measured best per SF (DESIGN.md 5).
bool k1_generic() {
    static int v = -1;
    if (v < 0) { const char *e = getenv("LORA_B200_K1"); v = e && !strcmp(e, "generic") ? 1 : 0; }
    return v == 1;
}

int dispatch_k1_impl(lora_b200_decoder *d, K1Scratch &ks, const float2 *iq, size_t n, uint32_t *bins, float *mags, cudaStream_t st) {
    if (!d->k1_ok) return fail(LORA_B200_EUNSUPPORTED, "FFT demodulator needs samp_rate/bandwidth == 8 and SF7..SF12");
    if (n == 0) return LORA_B200_OK;
    if (!k1_generic()) {
        static const char *rows = getenv("LORA_B200_K1_ROWS");
        switch (d->cfg.sf) {
        case 7: return launch_k1_packed(d, iq, n, bins, mags, st);
        case 8: return launch_k1_group<8, 6, 2>(d, ks, iq, n, bins, mags, st);
        case 9: return launch_k1_packed(d, iq, n, bins, mags, st);
        case 10: return launch_k1_sf10(d, ks, iq, n, bins, mags, st);
        case 11: case 12:
            if (!(rows && rows[0] == '0')) return launch_k1_rows(d, ks, iq, n, bins, mags, st);
            break;
        }
    }
    switch (d->cfg.sf) {
    case 7: return launch_k1<7>(d, ks, iq, n, bins, mags, st);
    case 8: return launch_k1<8>(d, ks, iq, n, bins, mags, st);
    case 9: return launch_k1<9>(d, ks, iq, n, bins, mags, st);
    case 10: return launch_k1<10>(d, ks, iq, n, bins, mags, st);
    case 11: return launch_k1<11>(d, ks, iq, n, bins, mags, st);
    case 12: return launch_k1<12>(d, ks, iq, n, bins, mags, st);
    }
    return fail(LORA_B200_EUNSUPPORTED, "unsupported SF %u", d->cfg.sf);
}

// K1 on stream `st` with scratch `ks`: a launch that follows one on ANOTHER stream with the same scratch waits for it
// (the memset of the keys / flags at the head of a launch must not run under the previous kernel)
int dispatch_k1(lora_b200_decoder *d, K1Scratch &ks, const float2 *iq, size_t n, uint32_t *bins, float *mags, cudaStream_t st) {
    if (!ks.done) CU(cudaEventCreateWithFlags(&ks.done, cudaEventDisableTiming));
    if (ks.used && ks.last != st) CU(cudaStreamWaitEvent(st, ks.done, 0));
    const int rc = dispatch_k1_impl(d, ks, iq, n, bins, mags, st);
    if (rc) return rc;
    CU(cudaEventRecord(ks.done, st));
    ks.last = st; ks.used = true;
    return LORA_B200_OK;
}

// ---- stream-path launch -----------------------------------------------------------------------
template <int SF, bool FFT>
int launch_rx_t(lora_b200_decoder *d, const RxParams &p, int grid, cudaStream_t st) {
    size_t smem = 0;
    if (FFT) {
        smem = sizeof(float2) * K1Cfg<SF>::SMEM_ELEMS;
        static bool attr_set[64] = {};
        if (!attr_set[d->device & 63]) {
            CU(cudaFuncSetAttribute(rx_stream_kernel<SF, FFT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_set[d->device & 63] = true;
        }
    }
    rx_stream_kernel<SF, FFT><<<grid, RX_THREADS, smem, st>>>(p);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

// SF7 at fs / bw = 8: one warp per stream (rx_warp.cuh); LORA_B200_RX=cta keeps the CTA-per-stream kernel (A/B runs)
template <bool FFT>
int launch_rx_warp(lora_b200_decoder *d, const RxParams &p, int n_streams, cudaStream_t st) {
    static bool attr_set[64] = {};
    const size_t smem = sizeof(RWSmem);
    if (!attr_set[d->device & 63]) {
        CU(cudaFuncSetAttribute(rx_warp_kernel<FFT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[d->device & 63] = true;
    }
    rx_warp_kernel<FFT><<<(n_streams + RW_WARPS - 1) / RW_WARPS, RW_WARPS * 32, smem, st>>>(p);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

int launch_rx(lora_b200_decoder *d, const RxParams &p, int grid, cudaStream_t st) {
    const bool fft = d->cfg.demod == LORA_B200_DEMOD_FFT;
    static const char *rxk = getenv("LORA_B200_RX");
    if (d->cfg.sf == 7 && d->sps == (uint32_t)RW_SPS && d->n_bins == (uint32_t)RW_N && !(rxk && !strcmp(rxk, "cta")))
        return fft ? launch_rx_warp<true>(d, p, grid, st) : launch_rx_warp<false>(d, p, grid, st);
    if (!fft) return launch_rx_t<7, false>(d, p, grid, st);       // SF is a run-time value on the gradient path
    switch (d->cfg.sf) {
    case 7: return launch_rx_t<7, true>(d, p, grid, st);
    case 8: return launch_rx_t<8, true>(d, p, grid, st);
    case 9: return launch_rx_t<9, true>(d, p, grid, st);
    case 10: return launch_rx_t<10, true>(d, p, grid, st);
    case 11: return launch_rx_t<11, true>(d, p, grid, st);
    case 12: return launch_rx_t<12, true>(d, p, grid, st);
    }
    return fail(LORA_B200_EUNSUPPORTED, "unsupported SF %u", d->cfg.sf);
}

void append_hex(std::string &s, const uint8_t *v, size_t n, bool endline, bool ascii) {   // print_vector_hex, utilities.h:351-368
    static const char digits[] = "0123456789abcdef";
    // (one snprintf per byte was 20 ms per call at 16 384 frames: more than the state machine of the last staging group)
    const size_t at = s.size();
    s.resize(at + 3 * n);
    char *o = &s[at];
    for (size_t i = 0; i < n; i++) { *o++ = ' '; *o++ = digits[v[i] >> 4]; *o++ = digits[v[i] & 15]; }
    if (ascii) {
        s += " (";
        for (size_t i = 0; i < n; i++)
            if (v[i] >= ' ' && v[i] <= '~') s.push_back((char)v[i]);
        s += ")";
    }
    if (endline) s += "\n";
}

int rx_begin(lora_b200_decoder *d) {
    CU(cudaMemsetAsync(d->d_n_frames, 0, sizeof(uint32_t), d->rx_stream));
    return LORA_B200_OK;
}

// the state machine for streams [stream_base, stream_base + n_launch) over staged IQ (one CTA per stream), async on rx_stream
// (n_items_s: per-stream item counts on the device, indexed by stream; nullptr = n_items for all)
int rx_launch(lora_b200_decoder *d, const float2 *d_iq, size_t stride_items, size_t n_items, uint32_t stream_base, uint32_t n_launch,
              cudaStream_t st = nullptr, const uint32_t *n_items_s = nullptr) {
    RxParams p;
    memset(&p, 0, sizeof p);
    p.iq = d_iq; p.stride_items = stride_items; p.n_items = n_items; p.n_items_s = n_items_s;
    p.stream_base = stream_base; p.n_launch = n_launch;
    p.down = tab<float2>(d, d->toff.down);
    p.down_ifreq = tab<float>(d, d->toff.down_ifreq);
    p.up_ifreq = tab<float>(d, d->toff.up_ifreq);
    p.up_ifreq_v = tab<float>(d, d->toff.up_ifreq_v);
    p.tw = tab<float2>(d, d->toff.tw);
    p.down_ifreq_avg = d->down_ifreq_avg; p.down_ifreq_sd = d->down_ifreq_sd;
    p.sps = d->sps; p.n_bins = d->n_bins; p.n_bins_hdr = d->n_bins_hdr; p.decim = d->decim; p.sf = d->cfg.sf;
    p.implicit = d->cfg.implicit; p.reduced_rate = d->cfg.reduced_rate; p.enable_fine_sync = !d->cfg.disable_drift_correction;
    p.cfo_estimate = d->cfo_estimate ? 1 : 0; p.samples_per_second = (float)d->samples_per_second;
    p.states = d->d_states; p.scratch = d->d_scratch; p.consumed = d->d_consumed;
    p.frames = d->d_frames; p.n_frames = d->d_n_frames; p.frame_cap = d->frame_cap;
    p.max_frames_per_stream = d->cfg.max_frames_per_call;
    p.trace = d->d_trace; p.trace_cap = d->cfg.trace_capacity; p.trace_n = d->d_trace_n;
    return launch_rx(d, p, (int)n_launch, st ? st : d->rx_stream);
}

// K8 on the queued frames, results back to the host, frames delivered per stream in sequence order
int rx_finish(lora_b200_decoder *d, uint32_t stream_base, uint32_t n_launch, size_t *consumed, lora_b200_frame_cb cb, void *user) {
    cudaStream_t st = d->rx_stream;
    const int k8_grid = (int)std::min<uint32_t>(d->frame_cap, (uint32_t)d->n_sms * 4u);
    k8_frames_kernel<<<k8_grid, 128, 0, st>>>(d->d_frames, d->d_n_frames, d->frame_cap, d->d_frames_out);
    d->launches++;
    CU(cudaGetLastError());
    uint32_t n_frames = 0;
    CU(cudaMemcpyAsync(&n_frames, d->d_n_frames, sizeof n_frames, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(d->h_consumed.data() + stream_base, d->d_consumed + stream_base,
                       sizeof(unsigned long long) * n_launch, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (n_frames > d->frame_cap) n_frames = d->frame_cap;
    if (n_frames) {
        if (!d->h_frames) CU(cudaMallocHost(&d->h_frames, sizeof(RxFrameOut) * d->frame_cap));      // pinned: the D2H runs at link speed
        CU(cudaMemcpyAsync(d->h_frames, d->d_frames_out, sizeof(RxFrameOut) * n_frames, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    for (uint32_t s = 0; s < n_launch; s++) {
        consumed[s] = (size_t)d->h_consumed[stream_base + s];
        d->stdout_last[stream_base + s].clear();
    }
    // queue order is arrival order across streams; deliver per stream in sequence order
    std::vector<uint32_t> order(n_frames);
    for (uint32_t i = 0; i < n_frames; i++) order[i] = i;
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
        const RxFrameOut &x = d->h_frames[a], &y = d->h_frames[b];
        return x.stream != y.stream ? x.stream < y.stream : x.seq < y.seq;
    });
    d->h_sorted.resize(n_frames);
    for (uint32_t k = 0; k < n_frames; k++) {
        const RxFrameOut &f = d->h_frames[order[k]];
        d->h_sorted[k] = f;
        std::string &so = d->stdout_last[f.stream];
        if (f.n_hdr_print) append_hex(so, f.hdr_print, f.n_hdr_print, false, false);    // :832
        append_hex(so, f.bytes + 18, f.len - 18, true, true);                           // :872
        if (cb) cb(user, f.stream, f.bytes, f.len);
    }
    return LORA_B200_OK;
}

int run_rx(lora_b200_decoder *d, const float2 *d_iq, size_t stride_items, size_t n_items, uint32_t stream_base,
           uint32_t n_launch, size_t *consumed, lora_b200_frame_cb cb, void *user) {
    int rc = rx_begin(d);
    if (!rc) rc = rx_launch(d, d_iq, stride_items, n_items, stream_base, n_launch);
    if (!rc) rc = rx_finish(d, stream_base, n_launch, consumed, cb, user);
    return rc;
}

// A3 on a batch of windows: one warp per window, the stream kernel's rw_ifreq on global memory
__global__ void k3_ifreq_kernel(const float2 *__restrict__ iq, size_t n_windows, uint32_t window, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const size_t warps = (size_t)gridDim.x * (blockDim.x >> 5);
    for (size_t w = (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); w < n_windows; w += warps)
        rw_ifreq<false>(iq + w * window, out + w * window, (int)window, lane);
}

// SDR-native ingest: interleaved int16 I/Q -> gr_complex scaled by `scale` (what a host-side sc16 -> fc32 converter does)
__global__ void sc16_to_cf32_kernel(const short2 *__restrict__ in, float2 *__restrict__ out, size_t n, float scale) {
    const size_t stride = (size_t)gridDim.x * blockDim.x * 4;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
        if (i + 4 <= n && (((uintptr_t)(in + i)) & 15u) == 0 && (((uintptr_t)(out + i)) & 15u) == 0) {
            const int4 v = __ldcs(reinterpret_cast<const int4 *>(in + i));
            const short2 s0 = *reinterpret_cast<const short2 *>(&v.x), s1 = *reinterpret_cast<const short2 *>(&v.y);
            const short2 s2 = *reinterpret_cast<const short2 *>(&v.z), s3 = *reinterpret_cast<const short2 *>(&v.w);
            float4 *o = reinterpret_cast<float4 *>(out + i);
            o[0] = make_float4(s0.x * scale, s0.y * scale, s1.x * scale, s1.y * scale);
            o[1] = make_float4(s2.x * scale, s2.y * scale, s3.x * scale, s3.y * scale);
        } else {
            for (size_t k = i; k < n && k < i + 4; k++) out[k] = make_float2(in[k].x * scale, in[k].y * scale);
        }
    }
}

// ... and interleaved int8 I/Q (GNU Radio's interleaved_char_to_complex; 2 bytes per sample over PCIe)
__global__ void sc8_to_cf32_kernel(const char2 *__restrict__ in, float2 *__restrict__ out, size_t n, float scale) {
    const size_t stride = (size_t)gridDim.x * blockDim.x * 8;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += stride) {
        if (i + 8 <= n && (((uintptr_t)(in + i)) & 15u) == 0 && (((uintptr_t)(out + i)) & 15u) == 0) {
            const int4 v = __ldcs(reinterpret_cast<const int4 *>(in + i));
            const int w[4] = {v.x, v.y, v.z, v.w};
            float4 *o = reinterpret_cast<float4 *>(out + i);
#pragma unroll
            for (int k = 0; k < 4; k++)
                o[k] = make_float4((float)(signed char)(w[k] & 0xff) * scale, (float)(signed char)((w[k] >> 8) & 0xff) * scale,
                                   (float)(signed char)((w[k] >> 16) & 0xff) * scale, (float)(signed char)((w[k] >> 24) & 0xff) * scale);
        } else {
            for (size_t k = i; k < n && k < i + 8; k++) out[k] = make_float2((float)in[k].x * scale, (float)in[k].y * scale);
        }
    }
}

}  // namespace

// ---- internal entry points for gateway.cu (rx_internal.h) ---------------------------------------
int lb_fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    return fail(code, "%s", buf);
}

int lb_rx_launch_streams(lora_b200_decoder *d, const float2 *iq, size_t stride_items, const uint32_t *n_items_s, cudaEvent_t ready,
                         cudaEvent_t done) {
    CU(cudaSetDevice(d->device));
    CU(cudaStreamWaitEvent(d->rx_stream, ready, 0));
    int rc = rx_begin(d);
    if (!rc) rc = rx_launch(d, iq, stride_items, stride_items, 0, d->cfg.n_streams, d->rx_stream, n_items_s);
    if (!rc) CU(cudaEventRecord(done, d->rx_stream));
    return rc;
}

int lb_rx_finish_streams(lora_b200_decoder *d, size_t *consumed) {
    CU(cudaSetDevice(d->device));
    return rx_finish(d, 0, d->cfg.n_streams, consumed, nullptr, nullptr);
}

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char *lora_b200_last_error(void) { return g_err.c_str(); }
int lora_b200_abi_version(void) { return LORA_B200_ABI_VERSION; }

// decoder_impl's members as the constructor leaves them (:55-66), for every stream
static cudaError_t init_states(lora_b200_decoder *d) {
    const uint32_t ns = d->cfg.n_streams;
    std::vector<RxStreamState> init(ns);
    memset(init.data(), 0, sizeof(RxStreamState) * ns);
    for (auto &s : init) {
        s.state = LORA_B200_DETECT;                                      // :55
        s.snr = 1.0f;                                                    // reference leaves d_snr uninitialised (oracle D4)
        s.phdr[1] = d->phdr1_init;
    }
    return cudaMemcpy(d->d_states, init.data(), sizeof(RxStreamState) * ns, cudaMemcpyHostToDevice);
}

lora_b200_decoder *lora_b200_create(const lora_b200_config *cfg) {
    if (!cfg) { fail(LORA_B200_EINVAL, "null config"); return nullptr; }
    if (cfg->sf < 6 || cfg->sf > 13) {            // decoder_impl.cc:57-61 (the reference prints this and exit(1)s)
        fail(LORA_B200_EINVAL, "[LoRa Decoder] ERROR : Spreading factor should be between 6 and 12 (inclusive)!\n"
                               "                       Other values are currently not supported.");
        return nullptr;
    }
    if (cfg->n_streams == 0) { fail(LORA_B200_EINVAL, "n_streams must be >= 1"); return nullptr; }
    if (cfg->cr > 4) {     // the reference would abort in deinterleave ("More than 8 bits per word", decoder_impl.cc:541-545)
        fail(LORA_B200_EINVAL, "coding rate must be 0..4 (4/4 .. 4/8), got %u", cfg->cr);
        return nullptr;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        fail(LORA_B200_ECUDA, "no CUDA device: liblora_b200 has no CPU fallback");
        return nullptr;
    }
    lora_b200_decoder *d = new lora_b200_decoder();
    d->cfg = *cfg;
    if (d->cfg.max_items_per_call == 0) d->cfg.max_items_per_call = 1u << 20;
    if (d->cfg.max_frames_per_call == 0) d->cfg.max_frames_per_call = 8;
    int dev = cfg->device;
    if (dev < 0) cudaGetDevice(&dev);
    d->device = dev;
    auto bail = [&](const char *what, cudaError_t e) {
        fail(LORA_B200_ECUDA, "%s: %s", what, cudaGetErrorString(e));
        lora_b200_destroy(d);
        return (lora_b200_decoder *)nullptr;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(dev)) != cudaSuccess) return bail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, dev)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
    d->n_sms = prop.multiProcessorCount;

    // A1: derived parameters, decoder_impl.cc:69-91 (same types, same order)
    d->samples_per_second = (uint32_t)cfg->samp_rate;                    // :74 (uint32_t member)
    d->dt = 1.0f / d->samples_per_second;                                // :77 float divide kept in a double
    const uint8_t cr3 = cfg->cr & 7u;                                    // 3-bit field
    d->bits_per_second = (double)cfg->sf * (double)(4.0 / (4.0 + cr3)) / (1u << cfg->sf) * cfg->bandwidth;   // :79
    d->symbols_per_second = (double)cfg->bandwidth / (1u << cfg->sf);    // :80
    d->bits_per_symbol = (double)(d->bits_per_second / d->symbols_per_second);   // :82
    d->sps = (uint32_t)(d->samples_per_second / d->symbols_per_second);  // :83
    d->delay_after_sync = d->sps / 4u;                                   // :84
    d->n_bins = 1u << cfg->sf;                                           // :85
    d->n_bins_hdr = 1u << (cfg->sf - 2);                                 // :86
    d->decim = d->sps / d->n_bins;                                       // :87
    if (d->sps < 2 * d->n_bins / 2 || d->decim == 0) {
        fail(LORA_B200_EINVAL, "samp_rate %.1f too low for bandwidth %u", cfg->samp_rate, cfg->bandwidth);
        delete d;
        return nullptr;
    }
    d->k1_ok = (d->sps == 8u * d->n_bins) && cfg->sf >= 7 && cfg->sf <= 12;
    if (cfg->demod == LORA_B200_DEMOD_FFT && !d->k1_ok) {
        fail(LORA_B200_EUNSUPPORTED, "FFT demodulator needs samp_rate/bandwidth == 8 and SF7..SF12");
        delete d;
        return nullptr;
    }

    build_tables(d);
    table_stats(d);
    if ((e = cudaMalloc(&d->d_tables, d->toff.total)) != cudaSuccess) return bail("cudaMalloc tables", e);
    if ((e = cudaMemcpy(d->d_tables, d->h_tables.data(), d->toff.total, cudaMemcpyHostToDevice)) != cudaSuccess) return bail("upload tables", e);

    const uint32_t ns = d->cfg.n_streams;
    if ((e = cudaStreamCreateWithFlags(&d->rx_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    if ((e = cudaMalloc(&d->d_states, sizeof(RxStreamState) * ns)) != cudaSuccess) return bail("cudaMalloc states", e);
    d->phdr1_init = (uint8_t)((cr3 << 5) | ((cfg->crc ? 1u : 0u) << 4));       // :72-73
    if ((e = init_states(d)) != cudaSuccess) return bail("init states", e);
    const size_t scr_per = 2 * (size_t)d->sps + d->n_bins;
    if ((e = cudaMalloc(&d->d_scratch, sizeof(float) * scr_per * ns)) != cudaSuccess) return bail("cudaMalloc scratch", e);
    if ((e = cudaMalloc(&d->d_consumed, sizeof(unsigned long long) * ns)) != cudaSuccess) return bail("cudaMalloc consumed", e);
    if ((e = cudaMemset(d->d_consumed, 0, sizeof(unsigned long long) * ns)) != cudaSuccess) return bail("memset", e);
    d->frame_cap = ns * d->cfg.max_frames_per_call;
    if ((e = cudaMalloc(&d->d_frames, sizeof(RxFrameRec) * d->frame_cap)) != cudaSuccess) return bail("cudaMalloc frames", e);
    if ((e = cudaMalloc(&d->d_frames_out, sizeof(RxFrameOut) * d->frame_cap)) != cudaSuccess) return bail("cudaMalloc frames_out", e);
    if ((e = cudaMalloc(&d->d_n_frames, sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc n_frames", e);
    if (d->cfg.trace_capacity) {
        if ((e = cudaMalloc(&d->d_trace, sizeof(lora_b200_step) * (size_t)d->cfg.trace_capacity * ns)) != cudaSuccess) return bail("cudaMalloc trace", e);
        if ((e = cudaMalloc(&d->d_trace_n, sizeof(uint32_t) * ns)) != cudaSuccess) return bail("cudaMalloc trace_n", e);
        cudaMemset(d->d_trace_n, 0, sizeof(uint32_t) * ns);
    }
    d->h_consumed.assign(ns, 0);
    d->stdout_last.assign(ns, std::string());
    d->k2_grid = d->n_sms * 4;
    return d;
}

void lora_b200_destroy(lora_b200_decoder *d) {
    if (!d) return;
    cudaSetDevice(d->device);
    cudaDeviceSynchronize();
    cudaFree(d->d_tables); cudaFree(d->d_k2_scratch);
    for (auto &ks : d->k1s) {
        cudaFree(ks.packed); cudaFree(ks.xs);
        if (ks.done) cudaEventDestroy(ks.done);
    }
    for (int i = 0; i < 2; i++) {
        if (d->copy_streams[i]) cudaStreamDestroy(d->copy_streams[i]);
        cudaFree(d->d_chunk[i]); cudaFree(d->d_chunk16[i]); cudaFree(d->d_chunk_bins[i]); cudaFree(d->d_chunk_mags[i]);
        if (d->h_chunk[i]) cudaFreeHost(d->h_chunk[i]);
    }
    if (d->rx_stream) cudaStreamDestroy(d->rx_stream);
    if (d->rx_stream2) cudaStreamDestroy(d->rx_stream2);
    if (d->rx2_done) cudaEventDestroy(d->rx2_done);
    if (d->rx_begin_ev) cudaEventDestroy(d->rx_begin_ev);
    cudaFree(d->d_states); cudaFree(d->d_scratch); cudaFree(d->d_consumed); cudaFree(d->d_frames);
    cudaFree(d->d_frames_out); cudaFree(d->d_n_frames); cudaFree(d->d_trace); cudaFree(d->d_trace_n);
    cudaFree(d->d_stage); cudaFree(d->d_stage16);
    for (cudaEvent_t e : d->stage_events) if (e) cudaEventDestroy(e);
    if (d->h_stage) cudaFreeHost(d->h_stage);
    if (d->h_frames) cudaFreeHost(d->h_frames);
    delete d;
}

uint32_t lora_b200_samples_per_symbol(const lora_b200_decoder *d) { return d ? d->sps : 0; }
uint32_t lora_b200_bins(const lora_b200_decoder *d) { return d ? d->n_bins : 0; }
uint32_t lora_b200_decimation(const lora_b200_decoder *d) { return d ? d->decim : 0; }
uint64_t lora_b200_launch_count(const lora_b200_decoder *d) { return d ? d->launches : 0; }

int lora_b200_banner(const lora_b200_decoder *d, char *buf, size_t cap) {    // decoder_impl.cc:93-103
    if (!d || !buf) return fail(LORA_B200_EINVAL, "null argument");
    int n = snprintf(buf, cap, "Bits (nominal) per symbol: \t%g\nBins per symbol: \t%u\nSamples per symbol: \t%u\nDecimation: \t\t%u\n",
                     d->bits_per_symbol, d->n_bins, d->sps, d->decim);
    if (d->cfg.disable_drift_correction && n >= 0 && (size_t)n < cap)
        n += snprintf(buf + n, cap - n, "Warning: clock drift correction disabled\n");
    if (d->cfg.implicit && n >= 0 && (size_t)n < cap)
        n += snprintf(buf + n, cap - n, "CR: \t\t%d\nCRC: \t\t%d\n", (int)(d->cfg.cr & 7), (int)(d->cfg.crc ? 1 : 0));
    return n;
}

int lora_b200_set_sf(lora_b200_decoder *d, uint8_t) {                         // :905-909
    return fail(LORA_B200_EUNSUPPORTED, "[LoRa Decoder] WARNING : Setting the spreading factor during execution is currently not supported.\n"
                                        "Nothing set, kept SF of %u.", d ? d->cfg.sf : 0);
}
int lora_b200_set_samp_rate(lora_b200_decoder *d, float) {                    // :911-915
    return fail(LORA_B200_EUNSUPPORTED, "[LoRa Decoder] WARNING : Setting the sample rate during execution is currently not supported.\n"
                                        "Nothing set, kept SR of %u.", d ? d->samples_per_second : 0);
}

size_t lora_b200_tables_build_host(const lora_b200_config *cfg, void *dst, size_t cap) {
    if (!cfg || cfg->sf < 6 || cfg->sf > 13) { fail(LORA_B200_EINVAL, "bad config"); return 0; }
    lora_b200_decoder tmp;
    tmp.cfg = *cfg;
    tmp.samples_per_second = (uint32_t)cfg->samp_rate;
    tmp.dt = 1.0f / tmp.samples_per_second;
    tmp.symbols_per_second = (double)cfg->bandwidth / (1u << cfg->sf);
    tmp.sps = (uint32_t)(tmp.samples_per_second / tmp.symbols_per_second);
    tmp.n_bins = 1u << cfg->sf;
    if (tmp.sps < tmp.n_bins) { fail(LORA_B200_EINVAL, "samp_rate too low"); return 0; }
    build_tables(&tmp);
    if (dst) {
        if (cap < tmp.toff.total) { fail(LORA_B200_EINVAL, "buffer too small"); return 0; }
        memcpy(dst, tmp.h_tables.data(), tmp.toff.total);
    }
    return tmp.toff.total;
}

size_t lora_b200_tables_bytes(const lora_b200_decoder *d) { return d ? d->toff.total : 0; }
void *lora_b200_tables_device_ptr(lora_b200_decoder *d) { return d ? d->d_tables : nullptr; }
int lora_b200_tables_export(const lora_b200_decoder *d, void *dst, size_t cap) {
    if (!d || !dst || cap < d->toff.total) return fail(LORA_B200_EINVAL, "tables_export: buffer too small");
    CU(cudaSetDevice(d->device));
    CU(cudaMemcpy(dst, d->d_tables, d->toff.total, cudaMemcpyDeviceToHost));
    return LORA_B200_OK;
}
int lora_b200_tables_import(lora_b200_decoder *d, const void *src, size_t bytes) {
    if (!d || !src || bytes != d->toff.total) return fail(LORA_B200_EINVAL, "tables_import: size mismatch");
    CU(cudaSetDevice(d->device));
    memcpy(d->h_tables.data(), src, bytes);
    table_stats(d);
    CU(cudaMemcpy(d->d_tables, src, bytes, cudaMemcpyHostToDevice));
    return LORA_B200_OK;
}

int lora_b200_tables_commit(lora_b200_decoder *d) {
    if (!d) return fail(LORA_B200_EINVAL, "null argument");
    CU(cudaSetDevice(d->device));
    CU(cudaMemcpy(d->h_tables.data(), d->d_tables, d->toff.total, cudaMemcpyDeviceToHost));
    table_stats(d);
    return LORA_B200_OK;
}

int lora_b200_demod_fft_dev(lora_b200_decoder *d, const void *iq, size_t n_symbols, uint32_t *bins, float *mags, void *stream) {
    if (!d || (!iq && n_symbols) || (!bins && n_symbols)) return fail(LORA_B200_EINVAL, "null argument");
    if (((uintptr_t)iq & 15u) != 0) return fail(LORA_B200_EINVAL, "iq must be 16-byte aligned");
    CU(cudaSetDevice(d->device));
    return dispatch_k1(d, d->k1s[0], (const float2 *)iq, n_symbols, bins, mags, (cudaStream_t)stream);
}

// K1 from host memory: double-buffered 64 MiB chunks, H2D + kernel + D2H overlapped on two streams (each slot owns its
// own keys / exchange scratch).  elem = 8: gr_complex; elem = 4: int16 I/Q, converted on the device right after the copy.
static int demod_fft_host_any(lora_b200_decoder *d, const void *iq, size_t elem, float scale, size_t n_symbols, uint32_t *bins, float *mags) {
    if (!d || (!iq && n_symbols) || (!bins && n_symbols)) return fail(LORA_B200_EINVAL, "null argument");
    if (!d->k1_ok) return fail(LORA_B200_EUNSUPPORTED, "FFT demodulator needs samp_rate/bandwidth == 8 and SF7..SF12");
    CU(cudaSetDevice(d->device));
    const size_t sym_bytes = sizeof(float2) * (size_t)d->sps, sym_in = elem * (size_t)d->sps;
    const bool sc16 = elem == 4;
    if (!d->chunk_symbols) {                          // lazily create the double-buffered pipeline (64 MiB chunks)
        d->chunk_symbols = std::max<size_t>(1, ((size_t)64 << 20) / sym_bytes);
        for (int i = 0; i < 2; i++) {
            if (!d->copy_streams[i]) CU(cudaStreamCreateWithFlags(&d->copy_streams[i], cudaStreamNonBlocking));
            CU(cudaMalloc(&d->d_chunk[i], d->chunk_symbols * sym_bytes));
            CU(cudaMalloc(&d->d_chunk_bins[i], d->chunk_symbols * sizeof(uint32_t)));
            CU(cudaMalloc(&d->d_chunk_mags[i], d->chunk_symbols * sizeof(float)));
        }
    }
    if (sc16 && !d->d_chunk16[0])
        for (int i = 0; i < 2; i++) CU(cudaMalloc(&d->d_chunk16[i], d->chunk_symbols * sym_in));
    cudaPointerAttributes attr;
    bool pinned = cudaPointerGetAttributes(&attr, iq) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (!pinned && !d->h_chunk[0])
        for (int i = 0; i < 2; i++) CU(cudaMallocHost(&d->h_chunk[i], d->chunk_symbols * sym_bytes));
    const uint8_t *src = (const uint8_t *)iq;
    size_t done = 0;
    int k = 0;
    while (done < n_symbols) {
        const size_t n = std::min(d->chunk_symbols, n_symbols - done);
        const int b = k & 1;
        cudaStream_t st = d->copy_streams[b];
        CU(cudaStreamSynchronize(st));                // buffer b is free again (its D2H finished)
        const void *h = src + done * sym_in;
        if (!pinned) { memcpy(d->h_chunk[b], h, n * sym_in); h = d->h_chunk[b]; }
        if (sc16) {
            CU(cudaMemcpyAsync(d->d_chunk16[b], h, n * sym_in, cudaMemcpyHostToDevice, st));
            const size_t ns = n * (size_t)d->sps;
            const int grid = (int)std::min<size_t>((ns / 4 + 255) / 256, (size_t)d->n_sms * 8);
            sc16_to_cf32_kernel<<<grid, 256, 0, st>>>((const short2 *)d->d_chunk16[b], (float2 *)d->d_chunk[b], ns, scale);
            d->launches++;
            CU(cudaGetLastError());
        } else {
            CU(cudaMemcpyAsync(d->d_chunk[b], h, n * sym_bytes, cudaMemcpyHostToDevice, st));
        }
        int rc = dispatch_k1(d, d->k1s[1 + b], (const float2 *)d->d_chunk[b], n, d->d_chunk_bins[b], d->d_chunk_mags[b], st);
        if (rc) return rc;
        CU(cudaMemcpyAsync(bins + done, d->d_chunk_bins[b], n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if (mags) CU(cudaMemcpyAsync(mags + done, d->d_chunk_mags[b], n * sizeof(float), cudaMemcpyDeviceToHost, st));
        done += n;
        k++;
    }
    CU(cudaStreamSynchronize(d->copy_streams[0]));
    CU(cudaStreamSynchronize(d->copy_streams[1]));
    return LORA_B200_OK;
}

int lora_b200_demod_fft_host(lora_b200_decoder *d, const void *iq, size_t n_symbols, uint32_t *bins, float *mags) {
    return demod_fft_host_any(d, iq, sizeof(float2), 1.0f, n_symbols, bins, mags);
}

int lora_b200_demod_fft_host_sc16(lora_b200_decoder *d, const void *iq_sc16, float scale, size_t n_symbols, uint32_t *bins, float *mags) {
    return demod_fft_host_any(d, iq_sc16, sizeof(short2), scale, n_symbols, bins, mags);
}

int lora_b200_demod_gradient_dev(lora_b200_decoder *d, const void *iq, size_t n_symbols, uint32_t *bins, void *stream) {
    if (!d || (!iq && n_symbols) || (!bins && n_symbols)) return fail(LORA_B200_EINVAL, "null argument");
    CU(cudaSetDevice(d->device));
    if (!d->d_k2_scratch) CU(cudaMalloc(&d->d_k2_scratch, sizeof(float) * (size_t)d->k2_grid * (d->sps + d->n_bins)));
    if (n_symbols == 0) return LORA_B200_OK;
    const int grid = (int)std::min<size_t>(n_symbols, (size_t)d->k2_grid);
    k2_gradient_kernel<<<grid, RX_THREADS, 0, (cudaStream_t)stream>>>((const float2 *)iq, n_symbols, d->sps, d->n_bins, d->decim,
                                                                     d->d_k2_scratch, bins);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

int lora_b200_ifreq_dev(lora_b200_decoder *d, const void *iq, size_t n_windows, uint32_t window, float *out, void *stream) {
    if (!d || (!iq && n_windows) || (!out && n_windows)) return fail(LORA_B200_EINVAL, "null argument");
    if (window == 0 || window % 128u) return fail(LORA_B200_EINVAL, "window must be a positive multiple of 128");
    CU(cudaSetDevice(d->device));
    if (n_windows == 0) return LORA_B200_OK;
    const int grid = (int)std::min<size_t>((n_windows + 7) / 8, (size_t)d->n_sms * 8);
    k3_ifreq_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float2 *)iq, n_windows, window, out);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

int lora_b200_decode_codewords_dev(lora_b200_decoder *d, const uint8_t *codewords, const uint32_t *lengths, size_t stride,
                                   const uint8_t *cr, const uint8_t *is_header, size_t n_vec, uint8_t *out,
                                   size_t out_stride, uint32_t *out_len, void *stream) {
    if (!d || !codewords || !lengths || !cr || !is_header || !out || !out_len) return fail(LORA_B200_EINVAL, "null argument");
    CU(cudaSetDevice(d->device));
    if (n_vec == 0) return LORA_B200_OK;
    const int grid = (int)std::min<size_t>(n_vec, (size_t)d->n_sms * 8);
    k8_decode_vectors_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(codewords, lengths, stride, cr, is_header, n_vec, out, out_stride, out_len);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

int lora_b200_deinterleave_dev(lora_b200_decoder *d, const uint32_t *words, uint32_t n_words, uint32_t ppm, size_t n_blocks,
                               uint8_t *codewords, void *stream) {
    if (!d || !words || !codewords) return fail(LORA_B200_EINVAL, "null argument");
    if (n_words == 0 || n_words > 8 || ppm == 0 || ppm > 16) return fail(LORA_B200_EINVAL, "n_words must be 1..8, ppm 1..16");
    CU(cudaSetDevice(d->device));
    if (n_blocks == 0) return LORA_B200_OK;
    k8_deinterleave_kernel<<<(unsigned)((n_blocks + 127) / 128), 128, 0, (cudaStream_t)stream>>>(words, n_words, ppm, n_blocks, codewords);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

// device staging for the host-pointer entry points (grows on demand); the pinned host mirror is only needed by the
// single-stream work() call, whose caller's buffer is pageable GNU Radio memory
static int ensure_stage(lora_b200_decoder *d, size_t items, bool want_host, bool want_sc16) {
    if (items > d->stage_cap) {
        if (d->d_stage) cudaFree(d->d_stage);
        if (d->h_stage) cudaFreeHost(d->h_stage);
        if (d->d_stage16) cudaFree(d->d_stage16);
        d->d_stage = nullptr; d->h_stage = nullptr; d->d_stage16 = nullptr; d->stage_cap = 0;
        CU(cudaMalloc(&d->d_stage, sizeof(float2) * items));
        d->stage_cap = items;
    }
    if (want_host && !d->h_stage) CU(cudaMallocHost(&d->h_stage, sizeof(float2) * d->stage_cap));
    if (want_sc16 && !d->d_stage16) CU(cudaMalloc(&d->d_stage16, sizeof(short2) * d->stage_cap));
    return LORA_B200_OK;
}

int lora_b200_work(lora_b200_decoder *d, uint32_t stream, const void *iq_host, size_t n_items, size_t *consumed,
                   lora_b200_frame_cb cb, void *user) {
    if (!d || !consumed || (!iq_host && n_items)) return fail(LORA_B200_EINVAL, "null argument");
    if (stream >= d->cfg.n_streams) return fail(LORA_B200_EINVAL, "stream %u out of range", stream);
    CU(cudaSetDevice(d->device));
    if (n_items > d->cfg.max_items_per_call) n_items = d->cfg.max_items_per_call;     // never read past what was staged
    *consumed = 0;
    if (n_items < 2 * (size_t)d->sps) return LORA_B200_OK;                             // output_multiple, :91
    int rc = ensure_stage(d, n_items, true, false);
    if (rc) return rc;
    memcpy(d->h_stage, iq_host, sizeof(float2) * n_items);
    CU(cudaMemcpyAsync(d->d_stage, d->h_stage, sizeof(float2) * n_items, cudaMemcpyHostToDevice, d->rx_stream));
    return run_rx(d, d->d_stage, n_items, n_items, stream, 1, consumed, cb, user);
}

// all streams at once.  Host input is staged in groups of streams: the copy of group g + 1 (copy stream) runs under the
// state machine of group g (rx stream), so the call costs max(PCIe, kernel) instead of their sum.  elem = 8: gr_complex,
// elem = 4: interleaved int16 I/Q converted on the device (x * scale) before the state machine reads it.
static int work_batch_any(lora_b200_decoder *d, const void *iq, size_t elem, float scale, size_t n_items, size_t stride_items,
                          int host_ptr, size_t *consumed, lora_b200_frame_cb cb, void *user) {
    if (!d || !consumed || (!iq && n_items)) return fail(LORA_B200_EINVAL, "null argument");
    CU(cudaSetDevice(d->device));
    const uint32_t ns = d->cfg.n_streams;
    for (uint32_t s = 0; s < ns; s++) consumed[s] = 0;
    if (n_items < 2 * (size_t)d->sps) return LORA_B200_OK;
    const bool sc16 = elem != sizeof(float2);             // an integer format (int16 or int8 I/Q) staged raw, converted on the device
    if (!host_ptr && !sc16) return run_rx(d, (const float2 *)iq, stride_items, n_items, 0, ns, consumed, cb, user);
    if (n_items > d->cfg.max_items_per_call) n_items = d->cfg.max_items_per_call;
    int rc = ensure_stage(d, n_items * ns, false, sc16);
    if (rc) return rc;
    if (!d->copy_streams[0]) CU(cudaStreamCreateWithFlags(&d->copy_streams[0], cudaStreamNonBlocking));
    // groups: one launch each; a group should fill the machine about once (rx_warp_kernel: RW_WARPS streams per CTA, one CTA per
    // SM; rx_stream_kernel: one stream per CTA, two CTAs per SM), small batches stay whole.  Consecutive groups run on two
    // alternating compute streams so that the tail of one launch overlaps the head of the next.
    const bool warp_kernel = d->cfg.sf == 7 && d->sps == (uint32_t)RW_SPS;
    const uint32_t per_wave = (uint32_t)d->n_sms * (warp_kernel ? (uint32_t)RW_WARPS : 2u);
    // (a group of per_wave + 1 streams would take two waves: round the number of groups UP, so that the last group -- the
    // only one whose state machine is not hidden under a copy -- is a single wave)
    const uint32_t n_groups = std::max<uint32_t>(1u, std::min<uint32_t>(8u, (ns + per_wave - 1) / per_wave));
    const uint32_t gs = (ns + n_groups - 1) / n_groups;
    if (!d->rx_stream2) {
        CU(cudaStreamCreateWithFlags(&d->rx_stream2, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&d->rx2_done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&d->rx_begin_ev, cudaEventDisableTiming));
    }
    if (d->stage_events.size() < n_groups) {
        const size_t have = d->stage_events.size();
        d->stage_events.resize(n_groups, nullptr);
        for (size_t i = have; i < n_groups; i++) CU(cudaEventCreateWithFlags(&d->stage_events[i], cudaEventDisableTiming));
    }
    cudaStream_t cs = d->copy_streams[0];
    if ((rc = rx_begin(d))) return rc;
    CU(cudaEventRecord(d->rx_begin_ev, d->rx_stream));            // the frame counter is reset before any group runs
    CU(cudaStreamWaitEvent(d->rx_stream2, d->rx_begin_ev, 0));
    for (uint32_t g = 0; g * gs < ns; g++) {
        const uint32_t s0 = g * gs, cnt = std::min<uint32_t>(gs, ns - s0);
        cudaStream_t xs = (g & 1) ? d->rx_stream2 : d->rx_stream;
        const uint8_t *src = (const uint8_t *)iq + (size_t)s0 * stride_items * elem;
        void *dst = sc16 ? (void *)((uint8_t *)d->d_stage16 + (size_t)s0 * n_items * elem) : (void *)(d->d_stage + (size_t)s0 * n_items);
        if (stride_items == n_items)                                  // dense rows: one linear copy (the 2-D form is for strided captures)
            CU(cudaMemcpyAsync(dst, src, elem * n_items * cnt, host_ptr ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, cs));
        else
            CU(cudaMemcpy2DAsync(dst, elem * n_items, src, elem * stride_items, elem * n_items, cnt,
                                 host_ptr ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, cs));
        CU(cudaEventRecord(d->stage_events[g], cs));
        CU(cudaStreamWaitEvent(xs, d->stage_events[g], 0));
        if (sc16) {
            const size_t n = (size_t)cnt * n_items;
            const int grid = (int)std::min<size_t>((n / 4 + 255) / 256, (size_t)d->n_sms * 8);
            if (elem == 4) sc16_to_cf32_kernel<<<grid, 256, 0, xs>>>(d->d_stage16 + (size_t)s0 * n_items, d->d_stage + (size_t)s0 * n_items, n, scale);
            else sc8_to_cf32_kernel<<<grid, 256, 0, xs>>>((const char2 *)d->d_stage16 + (size_t)s0 * n_items, d->d_stage + (size_t)s0 * n_items, n, scale);
            d->launches++;
            CU(cudaGetLastError());
        }
        if ((rc = rx_launch(d, d->d_stage + (size_t)s0 * n_items, n_items, n_items, s0, cnt, xs))) return rc;
    }
    CU(cudaEventRecord(d->rx2_done, d->rx_stream2));
    CU(cudaStreamWaitEvent(d->rx_stream, d->rx2_done, 0));
    return rx_finish(d, 0, ns, consumed, cb, user);
}

int lora_b200_work_batch(lora_b200_decoder *d, const void *iq, size_t n_items, size_t stride_items, int host_ptr,
                         size_t *consumed, lora_b200_frame_cb cb, void *user) {
    return work_batch_any(d, iq, sizeof(float2), 1.0f, n_items, stride_items, host_ptr, consumed, cb, user);
}

int lora_b200_work_batch_sc16(lora_b200_decoder *d, const void *iq_sc16, float scale, size_t n_items, size_t stride_items,
                              int host_ptr, size_t *consumed, lora_b200_frame_cb cb, void *user) {
    return work_batch_any(d, iq_sc16, sizeof(short2), scale, n_items, stride_items, host_ptr, consumed, cb, user);
}

int lora_b200_reset(lora_b200_decoder *d) {
    if (!d) return fail(LORA_B200_EINVAL, "null argument");
    CU(cudaSetDevice(d->device));
    CU(cudaStreamSynchronize(d->rx_stream));
    if (d->rx_stream2) CU(cudaStreamSynchronize(d->rx_stream2));
    CU(init_states(d));
    CU(cudaMemset(d->d_consumed, 0, sizeof(unsigned long long) * d->cfg.n_streams));
    if (d->d_trace_n) CU(cudaMemset(d->d_trace_n, 0, sizeof(uint32_t) * d->cfg.n_streams));
    d->h_sorted.clear();
    for (auto &so : d->stdout_last) so.clear();
    return LORA_B200_OK;
}

int lora_b200_tx_symbols_dev(lora_b200_decoder *d, const void *up_table, const uint32_t *values, const float *cfo_hz, float noise_sigma,
                             uint64_t seed, size_t n_symbols, void *out, void *stream) {
    if (!d || (!values && n_symbols) || (!out && n_symbols)) return fail(LORA_B200_EINVAL, "null argument");
    if (d->sps & 1u) return fail(LORA_B200_EUNSUPPORTED, "odd samples per symbol");
    CU(cudaSetDevice(d->device));
    if (n_symbols == 0) return LORA_B200_OK;
    const float2 *up = up_table ? (const float2 *)up_table : tab<float2>(d, d->toff.up);
    const size_t threads = n_symbols * (d->sps / 2);
    const int grid = (int)std::min<size_t>((threads + 255) / 256, (size_t)d->n_sms * 16);
    tx_symbols_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(up, d->sps, d->decim, values, cfo_hz, 1.0 / (double)d->cfg.samp_rate, noise_sigma,
                                                              (unsigned long long)seed, n_symbols, (float2 *)out);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

int lora_b200_tx_expand_dev(lora_b200_decoder *d, const void *base, uint32_t k, size_t n_items, float noise_sigma, uint64_t seed,
                            size_t n_streams, void *out, void *stream) {
    if (!d || !base || !out || k == 0) return fail(LORA_B200_EINVAL, "null argument");
    if (n_items & 1u) return fail(LORA_B200_EINVAL, "n_items must be even");
    CU(cudaSetDevice(d->device));
    if (n_streams == 0 || n_items == 0) return LORA_B200_OK;
    const size_t threads = n_streams * (n_items / 2);
    const int grid = (int)std::min<size_t>((threads + 255) / 256, (size_t)d->n_sms * 16);
    tx_expand_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float2 *)base, k, n_items, noise_sigma, (unsigned long long)seed, n_streams,
                                                             (float2 *)out);
    d->launches++;
    CU(cudaGetLastError());
    return LORA_B200_OK;
}

int lora_b200_work_batch_sc8(lora_b200_decoder *d, const void *iq_sc8, float scale, size_t n_items, size_t stride_items,
                             int host_ptr, size_t *consumed, lora_b200_frame_cb cb, void *user) {
    return work_batch_any(d, iq_sc8, sizeof(char2), scale, n_items, stride_items, host_ptr, consumed, cb, user);
}

int lora_b200_stream_state(lora_b200_decoder *d, uint32_t stream) {
    if (!d || stream >= d->cfg.n_streams) return fail(LORA_B200_EINVAL, "bad stream");
    CU(cudaSetDevice(d->device));
    int32_t st = 0;
    CU(cudaMemcpy(&st, &d->d_states[stream].state, sizeof st, cudaMemcpyDeviceToHost));
    return st;
}

static_assert(sizeof(lora_b200_frame) == sizeof(RxFrameOut) && LORA_B200_MAX_FRAME_BYTES == LB_MAX_FRAME + 2, "public frame record == K8 output record");

size_t lora_b200_frames_last(lora_b200_decoder *d, const lora_b200_frame **frames) {
    if (!d || !frames) { fail(LORA_B200_EINVAL, "null argument"); return 0; }
    *frames = reinterpret_cast<const lora_b200_frame *>(d->h_sorted.data());
    return d->h_sorted.size();
}

int lora_b200_set_cfo_estimate(lora_b200_decoder *d, int enable) {
    if (!d) return fail(LORA_B200_EINVAL, "null argument");
    d->cfo_estimate = enable != 0;
    return LORA_B200_OK;
}

int lora_b200_last_cfo(lora_b200_decoder *d, uint32_t stream, float *cfo_hz, uint32_t *count) {
    if (!d || stream >= d->cfg.n_streams || !cfo_hz) return fail(LORA_B200_EINVAL, "bad argument");
    CU(cudaSetDevice(d->device));
    struct { float cfo; uint32_t n; } v;
    CU(cudaMemcpy(&v, &d->d_states[stream].cfo_est, sizeof v, cudaMemcpyDeviceToHost));
    *cfo_hz = v.cfo;
    if (count) *count = v.n;
    return LORA_B200_OK;
}

int lora_b200_stdout_last(lora_b200_decoder *d, uint32_t stream, char *buf, size_t cap) {
    if (!d || !buf || stream >= d->cfg.n_streams) return fail(LORA_B200_EINVAL, "bad argument");
    return snprintf(buf, cap, "%s", d->stdout_last[stream].c_str());
}

int lora_b200_trace_read(lora_b200_decoder *d, uint32_t stream, lora_b200_step *steps, size_t cap, size_t *n) {
    if (!d || !steps || !n || stream >= d->cfg.n_streams) return fail(LORA_B200_EINVAL, "bad argument");
    if (!d->d_trace) return fail(LORA_B200_EINVAL, "trace_capacity was 0 at creation");
    CU(cudaSetDevice(d->device));
    uint32_t cnt = 0;
    CU(cudaMemcpy(&cnt, d->d_trace_n + stream, sizeof cnt, cudaMemcpyDeviceToHost));
    size_t m = std::min<size_t>(std::min<size_t>(cnt, d->cfg.trace_capacity), cap);
    if (m) CU(cudaMemcpy(steps, d->d_trace + (size_t)stream * d->cfg.trace_capacity, sizeof(lora_b200_step) * m, cudaMemcpyDeviceToHost));
    *n = cnt;
    return cnt > d->cfg.trace_capacity ? LORA_B200_EOVERFLOW : LORA_B200_OK;
}

}  // extern "C"
