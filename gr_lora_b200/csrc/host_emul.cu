// host_emul.cu -- CPU entry points for the __host__ __device__ phase functions (tests only).
// Lets the non-GPU test-suite run the kernels' index arithmetic, twiddles and integer chain
// on the host and compare them with the oracle.  Not part of liblora_b200.so.
#include "k1_fft.cuh"
#include "k1_warp.cuh"
#include "k1_group.cuh"
#include "k1_sf10.cuh"
#include "k1_rows.cuh"
#include "int_chain.cuh"
#include "tx_channel.cuh"
#include "gateway_gather.cuh"

extern "C" {

int lb_k1_emulate(int sf, const float2 *x, size_t n_symbols, const float2 *chirp, const float2 *tw,
                  uint32_t *bins, float *mags) {
    lb::K1Args a{x, chirp, tw, n_symbols};
    switch (sf) {
    case 7: lb::k1_emulate<7>(a, bins, mags); break;
    case 8: lb::k1_emulate<8>(a, bins, mags); break;
    case 9: lb::k1_emulate<9>(a, bins, mags); break;
    case 10: lb::k1_emulate<10>(a, bins, mags); break;
    case 11: lb::k1_emulate<11>(a, bins, mags); break;
    case 12: lb::k1_emulate<12>(a, bins, mags); break;
    default: return -1;
    }
    return 0;
}

int lb_k1_emulate_warp_sf7(const float2 *x, size_t n_symbols, const float2 *chirp, const float2 *tw, uint32_t *bins, float *mags) {
    lb::K1Args a{x, chirp, tw, n_symbols};
    lb::w7_emulate(a, bins, mags);
    return 0;
}

int lb_k1_emulate_group(int sf, const float2 *x, size_t n_symbols, const float2 *chirp, const float2 *tw, uint32_t *bins, float *mags) {
    lb::K1Args a{x, chirp, tw, n_symbols};
    switch (sf) {
    case 7: lb::g_emulate<7>(a, bins, mags); break;
    case 8: lb::g_emulate<8>(a, bins, mags); break;
    case 9: lb::g_emulate<9>(a, bins, mags); break;
    case 10: lb::s10_emulate(a, bins, mags); break;
    default: return -1;
    }
    return 0;
}

int lb_k1_emulate_rows(int sf, const float2 *x, size_t n_symbols, const float2 *chirp, const float2 *tw, uint32_t *bins, float *mags) {
    lb::K1Args a{x, chirp, tw, n_symbols};
    if (sf == 11) lb::r_emulate<11>(a, bins, mags);
    else if (sf == 12) lb::r_emulate<12>(a, bins, mags);
    else return -1;
    return 0;
}


// the counter-based generator of the transmitter / channel kernels (tx_channel.cuh), on the host
void lb_emul_philox4x32_10(const uint32_t *ctr, const uint32_t *key, uint32_t *out) {
    uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
    lb::philox4x32_10(c, key[0], key[1]);
    for (int i = 0; i < 4; i++) out[i] = c[i];
}

// the stream kernels' arg() (lora_common.cuh), on the host
void lb_emul_atan2f(const float *y, const float *x, float *out, size_t n) {
    for (size_t i = 0; i < n; i++) out[i] = lb::lb_atan2f(y[i], x[i]);
}

uint32_t lb_emul_decode(const uint8_t *cw, uint32_t n_cw, int is_header, uint32_t cr, uint8_t *out, uint32_t cap) {
    uint32_t n = lb::decode_len_bytes(lb::decode_len_words(n_cw, is_header), cr);
    if (n > cap) n = cap;
    for (uint32_t i = 0; i < n; i++) out[i] = lb::decode_byte(cw, n_cw, is_header, cr, i);
    return n;
}
void lb_emul_deinterleave(const uint32_t *words, uint32_t n_words, uint32_t ppm, uint8_t *out) { lb::deinterleave_block(words, n_words, ppm, out); }
uint32_t lb_emul_reduce_bin(uint32_t bin, uint32_t n_hdr) { return lb::reduce_bin(bin, n_hdr); }
uint32_t lb_emul_gray(uint32_t bin) { return lb::gray_encode(bin); }
uint8_t lb_emul_hamming84_decode(uint8_t cw) { return lb::hamming84_decode(cw); }
uint8_t lb_emul_hamming84_encode(uint8_t v) { return lb::hamming84_encode(v); }
uint8_t lb_emul_deshuffle(uint8_t v) { return lb::deshuffle_byte(v); }
int32_t lb_emul_payload_symbols(uint32_t len, uint32_t cr, uint32_t sf, int rr) { return lb::payload_symbols(len, cr, sf, rr); }

// the gateway's gather (gateway_gather.cuh) on the host: next[0, pending + m) from prev's tail and o, element by element
// through the kernel's index map; returns the new length, or -1 (next untouched) when it would exceed cap
int64_t lb_emul_gw_gather(const float2 *prev, uint32_t consumed, uint32_t pending, const float2 *o, uint32_t m, uint32_t cap,
                          float2 *next) {
    int ovf = 0;
    const uint32_t n = lb::gw_next_len(pending, m, cap, &ovf);
    if (ovf) return -1;
    for (uint32_t i = 0; i < n; i++) {
        int fp;
        const uint32_t s = lb::gw_src(i, consumed, pending, &fp);
        next[i] = fp ? prev[s] : o[s];
    }
    return n;
}
uint32_t lb_emul_gw_pending(uint32_t len, uint32_t consumed) { return lb::gw_pending(len, consumed); }

}
