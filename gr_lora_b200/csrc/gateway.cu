// gateway.cu -- N4: every channel and every spreading factor of a wideband capture (lora_b200_gateway_*, include/lora_b200.h).
//
// One call: wideband chunk -> lora_b200_channelizer_work_dev into O[n_ch][M] -> gw_gather_kernel appends O to what every
// (channel, SF) stream left unconsumed (gateway_gather.cuh) -> one decoder per SF runs its state machine over all channels
// with per-stream item counts (rx_internal.h), the SFs on their own CUDA streams concurrently -> frames collected.
// The decoders and the channelizer are the library's own objects; nothing here restates their DSP.
#include "../../include/lora_b200.h"
#include "gateway_gather.cuh"
#include "rx_internal.h"

#include <cuda_runtime.h>
#include <algorithm>
#include <cstring>
#include <vector>

using namespace lb;

namespace {

#define GCU(call)                                                                                    \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) return lb_fail(LORA_B200_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

constexpr uint32_t SF_MIN = 7, SF_MAX = 12, SF_BITS = ((1u << (SF_MAX + 1)) - 1u) & ~((1u << SF_MIN) - 1u);

struct GwSf {                            // one spreading factor: a decoder over all channels and its two buffers
    uint32_t sf = 0;
    lora_b200_decoder *dec = nullptr;
    float2 *buf[2] = {nullptr, nullptr}; // [n_ch][cap]
    int cur = 0;                         // buf[cur] holds what the last call presented
    std::vector<uint32_t> off, pending;  // per channel: start and length of the unconsumed tail in buf[cur]
    std::vector<uint64_t> total;         // per channel: items consumed since create / reset
};

}  // namespace

struct lora_b200_gateway {
    lora_b200_gateway_config cfg;
    std::vector<float> channel_list;
    int device = 0;
    uint32_t m_max = 0;                  // channel items per call at most
    uint32_t cap = 0;                    // row stride of every decoder buffer: m_max + the longest tail of any SF (even)
    lora_b200_channelizer *chan = nullptr;
    std::vector<GwSf> sfs;               // ascending SF
    cudaStream_t st = nullptr;
    float2 *d_in = nullptr;              // [max_in_per_call] staging of host input
    float2 *d_out = nullptr;             // [n_ch][m_max] channelizer output
    uint32_t *d_meta = nullptr, *h_meta = nullptr;   // per SF: off[n_ch] | pending[n_ch] | len[n_ch] (h_meta pinned)
    cudaEvent_t ev[5] = {};              // start | H2D done | channelizer done | gather done | state machines done
    std::vector<cudaEvent_t> ev_sf;      // per SF: its state machine done
    std::vector<size_t> consumed;
    lora_b200_gateway_frame *h_frames = nullptr;     // pinned, frame_cap records
    size_t frame_cap = 0, n_frames = 0;
    bool ran = false;
};

namespace {

int make_channelizer(lora_b200_gateway *g) {
    const lora_b200_gateway_config &c = g->cfg;
    g->chan = lora_b200_channelizer_create(c.samp_rate, c.center_freq, g->channel_list.data(), c.n_channels, c.bandwidth,
                                           c.decimation, g->device);
    if (!g->chan) return lb_fail(LORA_B200_ECUDA, "gateway: %s", lora_b200_channelizer_last_error());
    if (c.conj) lora_b200_channelizer_set_conjugate(g->chan, 1);
    return LORA_B200_OK;
}

bool reduced_rate(const lora_b200_gateway_config &c, uint32_t sf) {
    const uint32_t mask = c.reduced_rate_mask ? c.reduced_rate_mask : (1u << 11) | (1u << 12);
    return (mask >> sf) & 1u;
}

int gw_init(lora_b200_gateway *g) {
    const lora_b200_gateway_config &c = g->cfg;
    const uint32_t n_ch = c.n_channels;
    GCU(cudaSetDevice(g->device));
    GCU(cudaStreamCreateWithFlags(&g->st, cudaStreamNonBlocking));
    for (auto &e : g->ev) GCU(cudaEventCreate(&e));
    int rc = make_channelizer(g);
    if (rc) return rc;
    g->m_max = c.max_in_per_call / c.decimation;
    const float fs = c.samp_rate / (float)c.decimation;
    // the tail a stream leaves is shorter than one step's 2 sps look-ahead (unless it stopped at max_frames_per_call);
    // sps as the decoder derives it (lora_b200_create), the largest over the SFs
    unsigned long long sps_max = 0;
    for (uint32_t sf = SF_MIN; sf <= SF_MAX; sf++)
        if ((c.sf_mask >> sf) & 1u) sps_max = std::max(sps_max, (unsigned long long)((uint32_t)fs / ((double)c.bandwidth / (1u << sf))));
    const unsigned long long cap = ((unsigned long long)g->m_max + 2ull * sps_max + 256ull + 1ull) & ~1ull;   // even: float4 rows
    if (cap > 0xffffffffull) return lb_fail(LORA_B200_EINVAL, "gateway: max_in_per_call too large");
    g->cap = (uint32_t)cap;
    for (uint32_t sf = SF_MIN; sf <= SF_MAX; sf++) {
        if (!((c.sf_mask >> sf) & 1u)) continue;
        g->sfs.emplace_back();
        GwSf &s = g->sfs.back();
        s.sf = sf;
        lora_b200_config dc;
        memset(&dc, 0, sizeof dc);
        dc.samp_rate = fs;
        dc.bandwidth = c.bandwidth; dc.sf = (uint8_t)sf; dc.implicit = c.implicit; dc.cr = c.cr; dc.crc = c.crc;
        dc.reduced_rate = reduced_rate(c, sf) ? 1 : 0; dc.disable_drift_correction = c.disable_drift_correction; dc.demod = c.demod;
        dc.n_streams = n_ch; dc.device = g->device; dc.max_frames_per_call = c.max_frames_per_call;
        dc.max_items_per_call = g->cap;
        s.dec = lora_b200_create(&dc);   // all rate / SF checks are the decoder's own (its message stays in last_error)
        if (!s.dec) return LORA_B200_EINVAL;
        for (auto &b : s.buf) GCU(cudaMalloc(&b, sizeof(float2) * (size_t)n_ch * g->cap));
        s.off.assign(n_ch, 0); s.pending.assign(n_ch, 0); s.total.assign(n_ch, 0);
        cudaEvent_t e;
        GCU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        g->ev_sf.push_back(e);
    }
    const size_t n_sf = g->sfs.size();
    GCU(cudaMalloc(&g->d_in, sizeof(float2) * (size_t)c.max_in_per_call));
    GCU(cudaMalloc(&g->d_out, sizeof(float2) * (size_t)n_ch * (g->m_max ? g->m_max : 1)));
    GCU(cudaMalloc(&g->d_meta, sizeof(uint32_t) * 3 * n_ch * n_sf));
    GCU(cudaMallocHost(&g->h_meta, sizeof(uint32_t) * 3 * n_ch * n_sf));
    g->frame_cap = n_sf * n_ch * (size_t)(c.max_frames_per_call);
    GCU(cudaMallocHost(&g->h_frames, sizeof(lora_b200_gateway_frame) * g->frame_cap));
    g->consumed.assign(n_ch, 0);
    return LORA_B200_OK;
}

}  // namespace

extern "C" {

lora_b200_gateway *lora_b200_gateway_create(const lora_b200_gateway_config *cfg) {
    if (!cfg) { lb_fail(LORA_B200_EINVAL, "gateway: null config"); return nullptr; }
    if (!cfg->channel_list || cfg->n_channels == 0) { lb_fail(LORA_B200_EINVAL, "gateway: empty channel list"); return nullptr; }
    if (cfg->decimation == 0) { lb_fail(LORA_B200_EINVAL, "gateway: decimation must be >= 1"); return nullptr; }
    if (!(cfg->samp_rate > 0.0f)) { lb_fail(LORA_B200_EINVAL, "gateway: samp_rate must be > 0"); return nullptr; }
    if (cfg->sf_mask == 0 || (cfg->sf_mask & ~SF_BITS)) {
        lb_fail(LORA_B200_EINVAL, "gateway: sf_mask 0x%x must select SFs within 7..12", cfg->sf_mask);
        return nullptr;
    }
    if (cfg->reduced_rate_mask & ~SF_BITS) {
        lb_fail(LORA_B200_EINVAL, "gateway: reduced_rate_mask 0x%x has bits outside 7..12", cfg->reduced_rate_mask);
        return nullptr;
    }
    if (cfg->cr > 4) { lb_fail(LORA_B200_EINVAL, "gateway: coding rate must be 0..4 (4/4 .. 4/8), got %u", cfg->cr); return nullptr; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        lb_fail(LORA_B200_ECUDA, "no CUDA device: liblora_b200 has no CPU fallback");
        return nullptr;
    }
    lora_b200_gateway *g = new lora_b200_gateway();
    g->cfg = *cfg;
    if (g->cfg.max_in_per_call == 0) g->cfg.max_in_per_call = 1u << 22;
    if (g->cfg.max_frames_per_call == 0) g->cfg.max_frames_per_call = 8;
    g->channel_list.assign(cfg->channel_list, cfg->channel_list + cfg->n_channels);
    g->cfg.channel_list = g->channel_list.data();
    int dev = cfg->device;
    if (dev < 0) cudaGetDevice(&dev);
    g->device = dev;
    if (gw_init(g)) {                        // the reason stays in lora_b200_last_error
        lora_b200_gateway_destroy(g);
        return nullptr;
    }
    return g;
}

void lora_b200_gateway_destroy(lora_b200_gateway *g) {
    if (!g) return;
    cudaSetDevice(g->device);
    if (g->st) cudaStreamSynchronize(g->st);
    for (GwSf &s : g->sfs) {
        lora_b200_destroy(s.dec);
        cudaFree(s.buf[0]); cudaFree(s.buf[1]);
    }
    lora_b200_channelizer_destroy(g->chan);
    for (cudaEvent_t e : g->ev) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : g->ev_sf) cudaEventDestroy(e);
    cudaFree(g->d_in); cudaFree(g->d_out); cudaFree(g->d_meta);
    if (g->h_meta) cudaFreeHost(g->h_meta);
    if (g->h_frames) cudaFreeHost(g->h_frames);
    if (g->st) cudaStreamDestroy(g->st);
    delete g;
}

int lora_b200_gateway_reset(lora_b200_gateway *g) {
    if (!g) return lb_fail(LORA_B200_EINVAL, "gateway: null argument");
    GCU(cudaSetDevice(g->device));
    GCU(cudaStreamSynchronize(g->st));
    for (GwSf &s : g->sfs) {
        const int rc = lora_b200_reset(s.dec);
        if (rc) return rc;
        s.cur = 0;
        std::fill(s.off.begin(), s.off.end(), 0u);
        std::fill(s.pending.begin(), s.pending.end(), 0u);
        std::fill(s.total.begin(), s.total.end(), 0ull);
    }
    lora_b200_channelizer_destroy(g->chan);   // a new one: zero history, rotators at phase 0
    g->chan = nullptr;
    const int rc = make_channelizer(g);
    if (rc) return rc;
    g->n_frames = 0;
    g->ran = false;
    return LORA_B200_OK;
}

int lora_b200_gateway_work(lora_b200_gateway *g, const void *iq, size_t n_in, int host_ptr, size_t *n_frames) {
    if (!g || !n_frames || (!iq && n_in)) return lb_fail(LORA_B200_EINVAL, "gateway_work: null argument");
    const lora_b200_gateway_config &c = g->cfg;
    if (n_in % c.decimation) return lb_fail(LORA_B200_EINVAL, "gateway_work: n_in %zu is not a multiple of the decimation %u", n_in, c.decimation);
    if (n_in > c.max_in_per_call) return lb_fail(LORA_B200_EINVAL, "gateway_work: n_in %zu > max_in_per_call %u", n_in, c.max_in_per_call);
    *n_frames = 0;
    const uint32_t n_ch = c.n_channels, m = (uint32_t)(n_in / c.decimation);
    const size_t n_sf = g->sfs.size();
    // capacity first: on overflow nothing has been consumed or changed
    for (size_t k = 0; k < n_sf; k++) {
        const GwSf &s = g->sfs[k];
        uint32_t *meta = g->h_meta + 3 * n_ch * k;
        for (uint32_t ch = 0; ch < n_ch; ch++) {
            int ovf = 0;
            const uint32_t len = gw_next_len(s.pending[ch], m, g->cap, &ovf);
            if (ovf)
                return lb_fail(LORA_B200_EOVERFLOW, "gateway_work: channel %u SF%u holds %u unconsumed items; with %u new ones they exceed its "
                               "buffer of %u (it stopped at max_frames_per_call): call again with a smaller chunk", ch, s.sf, s.pending[ch], m, g->cap);
            meta[ch] = s.off[ch]; meta[n_ch + ch] = s.pending[ch]; meta[2 * n_ch + ch] = len;
        }
    }
    GCU(cudaSetDevice(g->device));
    cudaStream_t st = g->st;
    GCU(cudaEventRecord(g->ev[0], st));
    const float2 *in = (const float2 *)iq;
    if (host_ptr && n_in) {
        GCU(cudaMemcpyAsync(g->d_in, iq, sizeof(float2) * n_in, cudaMemcpyHostToDevice, st));
        in = g->d_in;
    }
    GCU(cudaEventRecord(g->ev[1], st));
    size_t n_out = 0;
    if (const int rc = lora_b200_channelizer_work_dev(g->chan, in, n_in, g->d_out, g->m_max, &n_out, st))
        return lb_fail(rc, "gateway_work: %s", lora_b200_channelizer_last_error());
    GCU(cudaEventRecord(g->ev[2], st));
    GCU(cudaMemcpyAsync(g->d_meta, g->h_meta, sizeof(uint32_t) * 3 * n_ch * n_sf, cudaMemcpyHostToDevice, st));
    GwGatherArgs a;
    memset(&a, 0, sizeof a);
    a.out = g->d_out; a.o_stride = g->m_max; a.m = m; a.cap = g->cap;
    uint32_t max_len = 1;
    for (size_t k = 0; k < n_sf; k++) {
        const GwSf &s = g->sfs[k];
        a.prev[k] = s.buf[s.cur]; a.next[k] = s.buf[s.cur ^ 1];
        a.consumed[k] = g->d_meta + 3 * n_ch * k; a.pending[k] = a.consumed[k] + n_ch;
        for (uint32_t ch = 0; ch < n_ch; ch++) max_len = std::max(max_len, g->h_meta[3 * n_ch * k + 2 * n_ch + ch]);
    }
    const unsigned gx = std::min<uint32_t>((max_len / 2 + 256) / 256, 4096u);
    gw_gather_kernel<<<dim3(gx, n_ch, (unsigned)n_sf), 256, 0, st>>>(a);
    GCU(cudaGetLastError());
    GCU(cudaEventRecord(g->ev[3], st));
    for (size_t k = 0; k < n_sf; k++) {
        GwSf &s = g->sfs[k];
        const int rc = lb_rx_launch_streams(s.dec, s.buf[s.cur ^ 1], g->cap, g->d_meta + 3 * n_ch * k + 2 * n_ch, g->ev[3], g->ev_sf[k]);
        if (rc) return rc;
    }
    for (size_t k = 0; k < n_sf; k++) GCU(cudaStreamWaitEvent(st, g->ev_sf[k], 0));
    GCU(cudaEventRecord(g->ev[4], st));
    // finish every SF (K8, consumed, frames) in turn; ascending SF, then (channel, seq) as the decoder sorts them
    size_t nf = 0;
    for (size_t k = 0; k < n_sf; k++) {
        GwSf &s = g->sfs[k];
        const int rc = lb_rx_finish_streams(s.dec, g->consumed.data());
        if (rc) return rc;
        const uint32_t *len = g->h_meta + 3 * n_ch * k + 2 * n_ch;
        for (uint32_t ch = 0; ch < n_ch; ch++) {
            const uint32_t used = (uint32_t)g->consumed[ch];
            s.off[ch] = used;
            s.pending[ch] = gw_pending(len[ch], used);
            s.total[ch] += used;
        }
        s.cur ^= 1;
        const lora_b200_frame *fr = nullptr;
        const size_t n = lora_b200_frames_last(s.dec, &fr);
        for (size_t i = 0; i < n && nf < g->frame_cap; i++, nf++) {
            g->h_frames[nf].channel = fr[i].stream;
            g->h_frames[nf].sf = s.sf;
            g->h_frames[nf].frame = fr[i];
        }
    }
    GCU(cudaStreamSynchronize(st));
    g->n_frames = nf;
    g->ran = true;
    *n_frames = nf;
    return LORA_B200_OK;
}

size_t lora_b200_gateway_frames_last(lora_b200_gateway *g, const lora_b200_gateway_frame **frames) {
    if (!g || !frames) { lb_fail(LORA_B200_EINVAL, "gateway_frames_last: null argument"); return 0; }
    *frames = g->h_frames;
    return g->n_frames;
}

int lora_b200_gateway_position(lora_b200_gateway *g, uint32_t channel, uint32_t sf, uint64_t *consumed, uint32_t *pending) {
    if (!g || !consumed || !pending) return lb_fail(LORA_B200_EINVAL, "gateway_position: null argument");
    if (channel >= g->cfg.n_channels) return lb_fail(LORA_B200_EINVAL, "gateway_position: channel %u out of range", channel);
    for (const GwSf &s : g->sfs)
        if (s.sf == sf) {
            *consumed = s.total[channel];
            *pending = s.pending[channel];
            return LORA_B200_OK;
        }
    return lb_fail(LORA_B200_EINVAL, "gateway_position: SF%u is not decoded by this gateway", sf);
}

int lora_b200_gateway_timing(const lora_b200_gateway *g, float *ms, size_t n) {
    if (!g || (!ms && n)) return lb_fail(LORA_B200_EINVAL, "gateway_timing: null argument");
    if (!g->ran) return lb_fail(LORA_B200_EINVAL, "gateway_timing: no work call yet");
    GCU(cudaSetDevice(g->device));
    for (size_t i = 0; i < n && i < 4; i++) GCU(cudaEventElapsedTime(ms + i, g->ev[i], g->ev[i + 1]));
    return LORA_B200_OK;
}

}  // extern "C"
