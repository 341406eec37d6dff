// rx_warp.cuh -- the receive state machine for SF7 at fs / bw = 8 (sps = 1024), ONE WARP PER STREAM.
//
// rx_stream_kernel (rx_stream.cuh) spends a 256-thread CTA on one stream: ~2 100 instructions per thread and symbol window,
// 16 CTA barriers and several dependent global round trips per step (ncu, profiles/r2_rx_sf7_cta.txt: issue slots 42 %
// active, stalls wait / barrier / long scoreboard 19 % each; 8.1e6 windows/s on 4096 streams).  At SF7 a window is 1024
// samples = 32 per lane, which is exactly the shape of the SF7 K1 warp kernel (k1_warp.cuh).  Here a warp owns a stream:
//   * the window (<= 2 sps samples, 16 KiB), its instantaneous frequency (8 KiB) and the decoder_impl members
//     (RxStreamState) live in the warp's own shared memory; the four tables (down-chirp, up / down ifreq, 3 x up ifreq)
//     are shared by the CTA's 10 warps; nothing but the IQ itself is read from global memory inside the loop;
//   * every step of work() (lib/decoder_impl.cc:740-903) is warp wide with __syncwarp() only: detect_preamble_autocorr,
//     sliding_norm_cross_correlate_upchirp, detect_downchirp, fine_sync, max_frequency_gradient_idx, determine_energy;
//     the FFT demodulator is the k1_warp.cuh pipeline on the window in place;
//   * the sliding correlation of the SYNC step (:399-413), sps lags x (sps - 1) products, keeps 32 consecutive lags per lane
//     in registers together with the sliding window of the instantaneous frequency they need (one new float per step), and
//     adds the products of every lag IN INDEX ORDER with separate multiply and add -- the order of the reference's scalar
//     dot product -- so the chosen index is the oracle's bit for bit (the CTA kernel's tree sum may pick the neighbouring
//     sample on ties, DESIGN.md 3).  The 63-lag fine_sync of the preamble uses the same register-resident window per
//     lane over a block of 32 products; the three-lag fine_sync of a payload symbol keeps the CTA kernel's lane-strided
//     order.  arg() is lb_atan2f (lora_common.cuh), four groups of 32 samples at a time.
//   * what bounds it: two or three warps per scheduler, every one a chain of dependent steps (ncu,
//     profiles/r2_rx_warp_final.txt: issue slots 42 % active, stalls wait 24 %, long scoreboard 18 %); 4 700 warp
//     instructions per window, a third of them the per-sample arg() and unwrap.  The kernel alone runs 4096 streams x 256
//     windows in 12 ms (8.7e7 windows/s); history in profiles/r2_rx_path.md.
// Same observable behaviour as rx_stream_kernel: frames, consume amounts, per-step trace.  Other SFs and sample rates use
// rx_stream_kernel.
#pragma once
#include "rx_stream.cuh"
#include "k1_warp.cuh"

namespace lb {

#ifndef LB_RW_WARPS
#define LB_RW_WARPS 10
#endif
// 10 warps: three per scheduler on two of the four (168 registers each), 198 KiB of shared memory; 4096 streams are then
// 2.8 waves of 1480 (with 9 warps they were 3.08 waves: a fourth, almost empty wave cost 25 %, sm__cycles_elapsed vs active)
constexpr int RW_SPS = 1024, RW_N = 128, RW_WARPS = LB_RW_WARPS;

#ifdef __CUDACC__
struct RWWarp {
    float4 win[RW_SPS / 2];           // sps samples (float2): the window of the SFD / decode steps (DETECT and SYNC stream from global)
    float ifq[2 * RW_SPS];            // instantaneous frequency of the window; [sps, sps + N) doubles as the bin averages
    RxStreamState st;
};
struct RWSmem {
    float4 chirp[RW_SPS / 2];         // down-chirp, natural order
    float up_ifreq[RW_SPS];
    float down_ifreq[RW_SPS];
    float up_ifreq_v[3 * RW_SPS + 3 * RW_SPS / 32];   // padded: float n at n + (n >> 5)
    RWWarp w[RW_WARPS];
};

// window samples [0, n) of the stream into the warp's buffer (8-byte accesses: the window starts at any sample); the lines
// of the following window are requested into L2 meanwhile -- where the next step starts is only known at the end of this
// one (consumed = sps +- fine sync), but it is within a few samples of g + n, and a step's first act is this load
// (11 % of the stall samples sat on it, profiles/r2b_rx_warp.txt)
LB_D void rw_load(const float2 *__restrict__ g, float2 *win, int n, int lane, const float2 *g_end) {
    {
        const char *nx = reinterpret_cast<const char *>(g + n) + 128 * lane;
#pragma unroll
        for (int j = 0; j < RW_SPS * 8 / (128 * 32); j++, nx += 128 * 32)
            if (nx < reinterpret_cast<const char *>(g_end)) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx));
    }
#pragma unroll 8
    for (int k = lane; k < n; k += 32) win[k] = __ldcs(g + k);
}

// A3 instantaneous_frequency (:224-244) of win[0, w) (shared or global memory) into out[0, w); one arg() per sample.
// PAD: out is written with one unused float after every 32 (index j + (j >> 5)), the layout rw_sync_xcorr reads.
template <bool PAD = false>
LB_D void rw_ifreq(const float2 *win, float *out, int w, int lane) {
    // Four groups of 32 samples per iteration: their arg() chains (~26 dependent instructions each) are independent, and
    // with two warps per scheduler the kernel lives on instruction-level parallelism (w is a multiple of 128).
    // The wrap is two selects, not the reference's two while loops: both arguments are in [-pi, pi], so either loop runs at
    // most once (a NaN fails both comparisons here as it fails both loop conditions there); the second test sees the
    // result of the first correction, like the second loop.
    float a[5];
    { const float2 s = win[lane]; a[0] = lb_atan2f(s.y, s.x); }
    for (int base = 0; base < w; base += 128) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int nb = base + 32 * (u + 1) + lane;
            a[u + 1] = 0.0f;
            if (nb < w) { const float2 s = win[nb]; a[u + 1] = lb_atan2f(s.y, s.x); }
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const float n1 = __shfl_sync(0xffffffffu, a[u], (lane + 1) & 31);
            const float n2 = __shfl_sync(0xffffffffu, a[u + 1], 0);
            const int j = base + 32 * u + lane;             // out[j] = wrap(arg x[j+1] - arg x[j])
            const float p1 = a[u];
            const float p2 = lane == 31 ? n2 : n1;
            // :236-237, float difference against the double M_PI (LB_PI_BELOW, lora_common.cuh), correction in double
            float q2 = p2 - p1 > LB_PI_BELOW ? (float)((double)p2 - 6.283185307179586) : p2;
            q2 = q2 - p1 < -LB_PI_BELOW ? (float)((double)q2 + 6.283185307179586) : q2;
            if (j < w - 1) out[PAD ? j + (j >> 5) : j] = q2 - p1;
        }
        a[0] = a[4];
    }
    __syncwarp();
    if (lane == 0) out[PAD ? w - 1 + ((w - 1) >> 5) : w - 1] = out[PAD ? w - 2 + ((w - 2) >> 5) : w - 2];
    __syncwarp();
}

// A9 sliding_norm_cross_correlate_upchirp (:392-413): c[lag] = sum_k f[lag + k] up[k], lag = 0 .. sps - 1, k = 0 .. sps - 2,
// every sum in k order with separate multiply and add like the reference's scalar dot product (cross_correlate_ifreq_fast ->
// volk_32f_x2_dot_prod_32f, :259-263), so the first maximum is the reference's sample index.
//
// Lane l owns the 32 consecutive lags 32 l + j.  At step k it needs f[32 l + k + j], j = 0..31: a window that slides by one
// float per step, so it lives in registers (V: 8 steps are unrolled so that every register index is a compile-time
// number, then the window moves down by 8) and ONE new float is loaded per step; the first version fetched all 32 from shared
// memory, 97 instructions per step and 22 % of the kernel's instructions.  Per step: 32 FMUL, 16 FADD2 (add.rn.f32x2 on
// accumulator pairs), one LDS = 49 instructions.  The products stay scalar on purpose: ptxas contracts mul.rn.f32x2 +
// add.rn.f32x2 into FFMA2 despite the explicit rounding (checked on the SASS, also with -fmad=false), which would round
// once where the reference rounds twice; a scalar FMUL feeding a packed add is left alone.
// f is read from the padded layout (33 floats per 32): the lanes are 33 floats apart, conflict-free.
constexpr int RW_XC_B = 8;                                            // steps per unrolled block
// one block of RW_XC_B steps; V[0 .. 31 + B) is the window on entry, moved down by B on exit.  The loop body is ~430
// instructions: the fully unrolled form (32 steps, 27 KiB of code, no reuse) left 24 % of the stall samples in
// "no instruction" -- nine warps streaming through different straight-line code defeat the instruction caches.
LB_D void rw_xc_block(float (&V)[32 + RW_XC_B], lb_u64 (&c2)[16], const float *next, const float *u, int steps) {
#ifdef __CUDA_ARCH__                                                  // (the packed helpers exist in the device pass only)
    float nv[RW_XC_B];
#pragma unroll
    for (int n = 0; n < RW_XC_B; n++) nv[n] = next[n];                // the floats the next block adds to the window
    const float4 u0 = *reinterpret_cast<const float4 *>(u), u1 = *reinterpret_cast<const float4 *>(u + 4);
    const float us[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
    for (int t = 0; t < RW_XC_B; t++) {
        if (t < steps) {
#pragma unroll
            for (int i = 0; i < 16; i++)
                c2[i] = add2(c2[i], pk2(__fmul_rn(V[2 * i + t], us[t]), __fmul_rn(V[2 * i + 1 + t], us[t])));
        }
    }
#pragma unroll
    for (int n = 0; n < 32; n++) V[n] = V[n + RW_XC_B];
#pragma unroll
    for (int n = 0; n < RW_XC_B; n++) V[32 + n] = nv[n];
#endif
}
// f: padded instantaneous frequency of two windows; up: up_ifreq (16-byte aligned).  Returns the warp's best key (0: no c > 0).
LB_D unsigned long long rw_sync_xcorr(const float *f, const float *up, int lane) {
    unsigned long long best = 0ull;
#ifdef __CUDA_ARCH__
    float V[32 + RW_XC_B];
    lb_u64 c2[16];
#pragma unroll
    for (int i = 0; i < 16; i++) c2[i] = pk2(0.0f, 0.0f);
    const float *rows = f + 33 * lane;                                // float n of this lane's sequence: rows[n + (n >> 5)]
#pragma unroll
    for (int n = 0; n < 32 + RW_XC_B; n++) V[n] = rows[n + (n >> 5)];
#pragma unroll 1
    for (int b = 0; b < RW_SPS / RW_XC_B; b++) {
        const int n0 = RW_XC_B * b + 32 + RW_XC_B;                    // first float of the next block's addition (8-aligned: one padded run)
        rw_xc_block(V, c2, rows + n0 + (n0 >> 5), up + RW_XC_B * b, b == RW_SPS / RW_XC_B - 1 ? RW_XC_B - 1 : RW_XC_B);   // k stops at sps - 2
    }
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const float2 c = up2(c2[i]);
        const unsigned long long k0 = corr_key(c.x, (uint32_t)(32 * lane + 2 * i)), k1 = corr_key(c.y, (uint32_t)(32 * lane + 2 * i + 1));
        best = k0 > best ? k0 : best;
        best = k1 > best ? k1 : best;
    }
    best = warp_max_key(best);
#endif
    return best;
}

// A6 fine_sync (:300-338) on ifq[0, sps), the three-lag search of a payload symbol: lane-strided products + butterfly sum per
// lag, as fine_sync_block does.  up_v is the padded table.
LB_D int rw_fine_sync(const float *ifq, const float *up_v, int bin_idx, int search, int lane) {
    const int shift_ref = (bin_idx + 1) * 8;                      // :301, decim = 8
    const int last = 3 * RW_SPS - 1;
    unsigned long long best = 0ull;
    for (int li = 0; li < 2 * search - 1; li++) {
        const int start = shift_ref + (li - (search - 1)) + RW_SPS;   // :310
        float c = 0.0f;
#pragma unroll 8
        for (int k = lane; k < RW_SPS; k += 32) {
            int idx = start + k;
            idx = idx < 0 ? 0 : (idx > last ? last : idx);        // defined over-read (oracle D1)
            c = fmaf(ifq[k], up_v[idx + (idx >> 5)], c);
        }
        c = warp_sum(c);
        const unsigned long long key = corr_key(c, (uint32_t)li);
        best = key > best ? key : best;
    }
    const int lag = best ? (int)key_idx(best) - (search - 1) : 0;
    return -lag;                                                  // :321
}

// A6 fine_sync (:300-338) for the preamble call fine_sync(ifreq, -1, decim * 4) (:803): 63 lags, shift = li - 31, of
//     c[li] = sum_k ifq[k] up_v[sps - 31 + li + k],  k = 0 .. sps - 1        (no index leaves the table: no clamping).
// One lag at a time that is 2 loads per product (the first version: 12 000 instructions per call, 14 % of the kernel's
// instructions).  Here lane l owns the products of k = 32 l .. 32 l + 31 for ALL lags: the table window it needs slides
// by one float per k, so it lives in registers (one new float per step) next to the 63 accumulators -- 65 instructions per
// step.  The 32 partial sums of every lag are then added in lane order through a 32 x 63 scratch array.
// ifq_p and up_vp are padded (float n at n + (n >> 5)): the lanes' rows are 33 floats apart, conflict-free.
constexpr int RW_FS_B = 4;                                            // products per unrolled block (see rw_xc_block on code size)
LB_D int rw_fine_sync63(const float *ifq_p, const float *up_vp, float *scratch, int lane) {
    constexpr int first = RW_SPS - 31;                                // table index of (li = 0, k = 0); first % 32 == 1
    const float *a = ifq_p + 33 * lane;
    const float *w = up_vp + (first + (first >> 5)) + 33 * lane;      // W[n] = table[first + 32 lane + n] = w[n + ((n + 1) >> 5)]
    float c[63], W[63 + RW_FS_B];
#pragma unroll
    for (int li = 0; li < 63; li++) c[li] = 0.0f;
#pragma unroll
    for (int n = 0; n < 63 + RW_FS_B; n++) W[n] = w[n + ((n + 1) >> 5)];
#pragma unroll 1
    for (int b = 0; b < 32 / RW_FS_B; b++) {
        float ak[RW_FS_B], nw[RW_FS_B];
        const int n0 = RW_FS_B * (b + 1) + 63;                        // next block's additions: n0 .. n0 + B - 1 (n0 + 1 is 8-aligned)
#pragma unroll
        for (int i = 0; i < RW_FS_B; i++) {
            ak[i] = a[RW_FS_B * b + i];
            const int n = n0 + i;
            nw[i] = w[n + ((n + 1) >> 5)];                            // (read past the last needed float in the last block: inside the table)
        }
#pragma unroll
        for (int i = 0; i < RW_FS_B; i++)
#pragma unroll
            for (int li = 0; li < 63; li++) c[li] = fmaf(ak[i], W[i + li], c[li]);
#pragma unroll
        for (int n = 0; n < 63; n++) W[n] = W[n + RW_FS_B];
#pragma unroll
        for (int i = 0; i < RW_FS_B; i++) W[63 + i] = nw[i];
    }
    __syncwarp();
#pragma unroll
    for (int li = 0; li < 63; li++) scratch[63 * lane + li] = c[li];
    __syncwarp();
    float s0 = 0.0f, s1 = 0.0f;                                       // lags lane and lane + 32
#pragma unroll
    for (int l = 0; l < 32; l++) {
        s0 += scratch[63 * l + lane];
        if (lane < 31) s1 += scratch[63 * l + lane + 32];
    }
    __syncwarp();
    const unsigned long long k0 = corr_key(s0, (uint32_t)lane), k1 = lane < 31 ? corr_key(s1, (uint32_t)(lane + 32)) : 0ull;
    const unsigned long long best = warp_max_key(k0 > k1 ? k0 : k1);
    const int lag = best ? (int)key_idx(best) - 31 : 0;
    return -lag;                                                      // :321
}

template <bool FFT>
__global__ void __launch_bounds__(RW_WARPS * 32, 1)
rx_warp_kernel(RxParams p) {
    extern __shared__ __align__(128) unsigned char rw_raw[];
    RWSmem &sm = *reinterpret_cast<RWSmem *>(rw_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int sps = RW_SPS, N = RW_N;

    for (int i = threadIdx.x; i < RW_SPS / 2; i += RW_WARPS * 32) sm.chirp[i] = k1_ld_table4(p.down + 2 * i);
    for (int i = threadIdx.x; i < RW_SPS; i += RW_WARPS * 32) { sm.up_ifreq[i] = __ldg(p.up_ifreq + i); sm.down_ifreq[i] = __ldg(p.down_ifreq + i); }
    for (int i = threadIdx.x; i < 3 * RW_SPS; i += RW_WARPS * 32) sm.up_ifreq_v[i + (i >> 5)] = __ldg(p.up_ifreq_v + i);
    __syncthreads();

    const uint32_t local = blockIdx.x * RW_WARPS + warp;          // stream of this launch
    if (local >= p.n_launch) return;                              // (no CTA barrier below)
    const uint32_t stream = p.stream_base + local;
    const float2 *xs = p.iq + (size_t)local * p.stride_items;
    RWWarp &ws = sm.w[warp];
    RxStreamState *gst = p.states + stream;
    RxStreamState *st = &ws.st;
    {   // decoder_impl members: global -> shared for the whole call
        const uint32_t *src = reinterpret_cast<const uint32_t *>(gst);
        uint32_t *dst = reinterpret_cast<uint32_t *>(st);
        for (int i = lane; i < (int)(sizeof(RxStreamState) / 4); i += 32) dst[i] = src[i];
    }
    __syncwarp();
    float2 *win = reinterpret_cast<float2 *>(ws.win);
    float *ifq = ws.ifq;
    lora_b200_step *trace = p.trace ? p.trace + (size_t)stream * p.trace_cap : nullptr;
    W7Consts kc;
    if (FFT) w7_consts(lane, p.tw, kc);

    int state = st->state;
    unsigned long long pos = 0;
    unsigned int frames_here = 0, steps = 0;

    while (true) {
        if (pos + 2ull * (unsigned long long)sps > LB_RX_N_ITEMS(p, stream)) break;
        if (frames_here >= p.max_frames_per_stream) break;
        const float2 *x = xs + pos;
        int consumed = 0, fine = 0, bin = -1, next_state = state;     // :749
        float metric = 0.0f;

        switch (state) {
        case LORA_B200_DETECT: {                                  // :752-768, A8 :340-366
            float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
#pragma unroll 8
            for (int i = lane; i < sps; i += 32) {
                const float2 a = __ldcs(x + i), b = __ldcs(x + i + sps);
                v0 += a.x * b.x + a.y * b.y;                      // a * conj(b)
                v1 += a.y * b.x - a.x * b.y;
                v2 += a.x * a.x + a.y * a.y;
                v3 += b.x * b.x + b.y * b.y;
            }
            v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2); v3 = warp_sum(v3);
            const float s = sqrtf(v2 * v3);
            const float corr = hypotf(v0 / s, v1 / s);            // :363
            metric = corr;
            if (lane == 0) {
                st->energy_threshold = v3 / 2.0f;                 // :357
                const float pw = v2 / (float)sps;                 // :360 push_back on the 4-deep ring
                if (st->pwr_n < 4) { st->pwr_queue[(st->pwr_head + st->pwr_n) & 3] = pw; st->pwr_n++; }
                else { st->pwr_queue[st->pwr_head] = pw; st->pwr_head = (st->pwr_head + 1) & 3; }
                if (corr >= 0.90f) {                              // :755
                    if (st->pwr_n >= 2)                           // determine_snr :377-383
                        st->snr = st->pwr_queue[(st->pwr_head + st->pwr_n - 1) & 3] / st->pwr_queue[st->pwr_head];
                    st->corr_fails = 0u;
                }
            }
            if (corr >= 0.90f) next_state = LORA_B200_SYNC; else consumed = sps;
            break;
        }
        case LORA_B200_SYNC: {                                    // :770-783, A9 :392-413
            // straight from global memory (every sample is touched once) into the padded layout, over win and the head of ifq
            float *fpad = reinterpret_cast<float *>(ws.win);
            rw_ifreq<true>(x, fpad, 2 * sps, lane);
            const unsigned long long best = rw_sync_xcorr(fpad, sm.up_ifreq, lane);
            metric = best ? key_mag2(best) : 0.0f;
            consumed = best ? (int)key_idx(best) : 0;             // :780 consume_each(i)
            next_state = LORA_B200_FIND_SFD;
            if (p.cfo_estimate && lane == 0) {                    // experimental_determine_cfo(&input[i], sps), :730-738,774
                const float2 m0 = cmul(x[consumed + 256], __ldg(p.down + 256)), m1 = cmul(x[consumed + 257], __ldg(p.down + 257));
                const float p1 = atan2f(m0.y, m0.x);
                float p2 = atan2f(m1.y, m1.x);
                while (p2 - p1 > LB_PI_BELOW) p2 = (float)((double)p2 - 6.283185307179586);
                while (p2 - p1 < -LB_PI_BELOW) p2 = (float)((double)p2 + 6.283185307179586);
                st->cfo_est = (float)((double)(p2 - p1) / (2.0 * 3.14159265358979323846) * (double)p.samples_per_second);
                st->cfo_count++;
            }
            break;
        }
        case LORA_B200_FIND_SFD: {                                // :785-818, A10
            rw_load(x, win, sps, lane, xs + LB_RX_N_ITEMS(p, stream));
            __syncwarp();
            rw_ifreq<true>(win, ifq, sps, lane);                  // padded: float i at i + (i >> 5) = lane + 33 j for i = lane + 32 j
            const int to_idx = sps - 1;
            float s1 = 0.f;
#pragma unroll 8
            for (int i = lane, ip = lane; i < to_idx; i += 32, ip += 33) s1 += ifq[ip];
            s1 = warp_sum(s1);
            const float average = s1 / (float)to_idx;             // :286
            float q0 = 0.f, q1 = 0.f;
#pragma unroll 8
            for (int i = lane, ip = lane; i < to_idx; i += 32, ip += 33) {
                const float t = ifq[ip] - average;
                q0 = fmaf(t, t, q0);                              // stddev :415-425
                q1 = fmaf(t, sm.down_ifreq[i] - p.down_ifreq_avg, q1);
            }
            q0 = warp_sum(q0); q1 = warp_sum(q1);
            const float sd = sqrtf(q0 / (float)to_idx) * p.down_ifreq_sd;   // :288-289
            const float cc = q1 / sd / (float)to_idx;             // :291-295
            const bool up_again = !(cc > 0.96f) && (cc < -0.97f);
            if (up_again) fine = rw_fine_sync63(ifq, sm.up_ifreq_v, reinterpret_cast<float *>(ws.win), lane);   // :803, fine_sync(ifreq, -1, decim * 4)
            metric = cc;
            if (cc > 0.96f) {
                next_state = LORA_B200_PAUSE;                     // :799
            } else {
                unsigned int fails = st->corr_fails;
                if (!up_again) fails++;                           // :805
                __syncwarp();
                if (lane == 0) st->corr_fails = fails;
                if (fails > 4u) next_state = LORA_B200_DETECT;    // :808-813
            }
            consumed = sps + fine;                                // :816
            break;
        }
        case LORA_B200_PAUSE: {                                   // :820-824
            next_state = LORA_B200_DECODE_HEADER;
            consumed = sps + sps / 4;
            break;
        }
        case LORA_B200_DECODE_HEADER:
        case LORA_B200_DECODE_PAYLOAD: {                          // :826-886
            const bool is_first = state == LORA_B200_DECODE_HEADER;
            rw_load(x, win, sps, lane, xs + LB_RX_N_ITEMS(p, stream));
            __syncwarp();
            bool do_demod = true;
            if (!is_first && p.implicit) {                        // :861 determine_energy
                float e = 0.f;
#pragma unroll 8
                for (int i = lane; i < sps; i += 32) { const float2 a = win[i]; e += a.x * a.x + a.y * a.y; }
                e = warp_sum(e);
                if (e < st->energy_threshold) do_demod = false;
            }
            if (do_demod) {                                       // demodulate(), :493-529
                if (!FFT || p.enable_fine_sync) rw_ifreq(win, ifq, sps, lane);
                if (FFT) {                                        // get_shift_fft (:430-464) as in k1_sf7_warp_kernel, window in place
                    float2 v0[16], v1[16];
                    w7_pass0(lane, ws.win, sm.chirp, v0, v1);
                    __syncwarp();
                    w7_store(lane, ws.win, v0, v1);
                    __syncwarp();
                    float2 P[8], Pq;
                    w7_pass1(lane, ws.win, kc, P, Pq);
                    const int h = lane & 1;
                    float2 own[4], other[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const float2 send = h ? P[j] : P[4 + j];
                        own[j] = h ? P[4 + j] : P[j];
                        other[j].x = __shfl_xor_sync(0xffffffffu, send.x, 1);
                        other[j].y = __shfl_xor_sync(0xffffffffu, send.y, 1);
                    }
                    float2 other_q;
                    other_q.x = __shfl_xor_sync(0xffffffffu, Pq.x, 1);
                    other_q.y = __shfl_xor_sync(0xffffffffu, Pq.y, 1);
                    unsigned long long best = w7_final(lane, kc, own, other, Pq, other_q);
                    best = warp_max_key(best);
                    bin = ((int)key_idx(best) + N - 1) % N;       // gradient-index convention (SURVEY A7)
                } else {                                          // A5 :466-491
                    float *avg = ifq + sps;
#pragma unroll
                    for (int m = 0; m < N / 32; m++) {
                        const int i = lane + 32 * m;
                        float acc = 0.0f;
#pragma unroll
                        for (int k = 0; k < 8; k++) acc += ifq[i * 8 + k];   // :475
                        avg[i] = acc / 8.0f;                      // :476
                    }
                    __syncwarp();
                    unsigned long long best = 0ull;
#pragma unroll
                    for (int m = 0; m < N / 32; m++) {
                        const int i = lane + 32 * m;
                        if (i >= 1) {
                            const float g = avg[i - 1] - avg[i];  // :483
                            if (g > 0.1f) { const unsigned long long k = pack_key(g, (uint32_t)i); best = k > best ? k : best; }
                        }
                    }
                    best = warp_max_key(best);
                    const int max_index = best ? (int)key_idx(best) + 1 : 0;   // :486
                    bin = (N - max_index) % N;                    // :490
                }
                if (p.enable_fine_sync) fine = rw_fine_sync(ifq, sm.up_ifreq_v, bin, 2, lane);   // :501-502, max(decim / 4, 2)
            }
            int flag = 0;
            unsigned int frame_slot = 0;
            if (lane == 0) {
                bool block_done = false;
                uint32_t cr = st->phdr[1] >> 5;
                if (do_demod) {
                    const bool reduced = is_first || p.reduced_rate;      // :495
                    uint32_t b = (uint32_t)bin;
                    if (reduced) b = reduce_bin(b, p.n_bins_hdr);  // :507-509
                    if (st->n_words < 8u) st->words[st->n_words] = gray_encode(b);    // :512,:517
                    st->n_words++;
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
                        flag = 2;                                 // -> DECODE_PAYLOAD, :853
                    }
                } else {
                    if (block_done && !p.implicit) st->payload_symbols -= (int32_t)(4u + cr);   // :866-867
                    if (st->payload_symbols <= 0) {               // :870
                        flag = 1;
                        frame_slot = atomicAdd(p.n_frames, 1u);
                    }
                }
            }
            __syncwarp();                                         // lane 0's stores to the decoder state above -> every lane's reads below
            flag = __shfl_sync(0xffffffffu, flag, 0);
            frame_slot = __shfl_sync(0xffffffffu, frame_slot, 0);
            if (flag == 2) next_state = LORA_B200_DECODE_PAYLOAD;
            consumed = sps + fine;                                // :856,:883
            if (flag == 1) {                                      // decode(false) + msg_lora_frame happen in K8
                if (frame_slot < p.frame_cap) {
                    RxFrameRec *fr = p.frames + frame_slot;
                    const uint32_t n = st->n_demod;
                    for (uint32_t k = lane; k < n; k += 32) fr->cw[k] = st->demodulated[k];
                    if (lane == 0) {
                        fr->stream = stream; fr->seq = st->frame_seq++; fr->n_cw = n; fr->cr = st->phdr[1] >> 5;
                        fr->payload_length = st->payload_length; fr->snr = st->snr;
                        fr->phdr[0] = st->phdr[0]; fr->phdr[1] = st->phdr[1]; fr->phdr[2] = st->phdr[2];
                        fr->n_hdr_print = p.implicit ? 0 : st->n_hdr_print;
                        for (int k = 0; k < 4; k++) fr->hdr_print[k] = st->hdr_print[k];
                    }
                }
                __syncwarp();
                if (lane == 0) { st->n_words = 0; st->n_demod = 0; }     // :875-880
                next_state = LORA_B200_DETECT;
                frames_here++;
            }
            break;
        }
        default: {                                                // STOP :888-891
            consumed = sps;
            break;
        }
        }
        if (lane == 0 && trace && steps < p.trace_cap) {
            lora_b200_step t;
            t.state = state; t.consumed = consumed; t.bin = bin; t.fine_sync = fine; t.metric = metric;
            trace[steps] = t;
        }
        steps++;
        pos += (unsigned long long)(consumed > 0 ? consumed : 0);
        state = next_state;
        __syncwarp();                                             // the window and the state are rewritten by the next step
    }
    if (lane == 0) st->state = state;
    __syncwarp();
    {
        uint32_t *dst = reinterpret_cast<uint32_t *>(gst);
        const uint32_t *src = reinterpret_cast<const uint32_t *>(st);
        for (int i = lane; i < (int)(sizeof(RxStreamState) / 4); i += 32) dst[i] = src[i];
    }
    if (lane == 0) {
        p.consumed[stream] = pos;
        if (p.trace_n) p.trace_n[stream] = steps;
    }
}
#endif  // __CUDACC__

}  // namespace lb
