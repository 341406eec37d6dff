/*
 * lora_b200.h -- C ABI of liblora_b200.so, the B200 (sm_100a) replacement for the hot path of
 * rpp0/gr-lora: gr::lora::decoder_impl::work() and the DSP helpers it calls
 * (lib/decoder_impl.cc:141-903 of the reference).
 *
 * Drop-in boundary (SURVEY.md 8b): the GNU Radio scheduler, PMT message ports and the
 * hier-block wiring stay on the host.  A thin gr::lora::decoder_impl shim (see
 * INTEGRATION.md) forwards its constructor arguments to lora_b200_create() and its
 * work() buffer to lora_b200_work(); everything numerical happens behind this header.
 * Plain C types only: no torch, no C++ in the signatures.
 *
 * All functions return 0 on success or a negative LORA_B200_E* code; the message of the
 * last failure on the calling thread is available from lora_b200_last_error().
 * There is NO CPU fallback: without a CUDA device lora_b200_create() fails.
 */
#ifndef LORA_B200_H
#define LORA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LORA_B200_ABI_VERSION 1

enum {
    LORA_B200_OK = 0,
    LORA_B200_EINVAL = -1,     /* bad argument (the reference exit(1)s for sf outside [6,13], decoder_impl.cc:57-61) */
    LORA_B200_ECUDA = -2,      /* CUDA runtime failure / no device */
    LORA_B200_ENOMEM = -3,
    LORA_B200_EUNSUPPORTED = -4,
    LORA_B200_EOVERFLOW = -5   /* per-call frame or trace capacity exhausted */
};

/* demodulator selection for demodulate() (decoder_impl.cc:499-500) */
enum {
    LORA_B200_DEMOD_GRADIENT = 0,  /* max_frequency_gradient_idx: what the reference runs today (:499)      */
    LORA_B200_DEMOD_FFT = 1        /* dechirp + FFT + argmax (get_shift_fft :430-464), mapped (bin-1) mod N */
};

/* decoder states, lib/decoder_impl.h:40-48 */
enum { LORA_B200_DETECT = 0, LORA_B200_SYNC, LORA_B200_FIND_SFD, LORA_B200_PAUSE,
       LORA_B200_DECODE_HEADER, LORA_B200_DECODE_PAYLOAD, LORA_B200_STOP };

/* Replaces the argument list of lora::decoder::make (include/lora/decoder.h:705,
 * lib/decoder_impl.cc:41-44,49): the first eight fields are exactly those arguments. */
typedef struct lora_b200_config {
    float    samp_rate;
    uint32_t bandwidth;
    uint8_t  sf;
    uint8_t  implicit;
    uint8_t  cr;
    uint8_t  crc;
    uint8_t  reduced_rate;
    uint8_t  disable_drift_correction;
    uint8_t  demod;              /* LORA_B200_DEMOD_*                                         */
    uint8_t  reserved0;
    uint32_t n_streams;          /* independent (channel, SF) streams sharing this config; >=1 */
    int32_t  device;             /* CUDA device ordinal; -1 = current device                   */
    uint32_t max_items_per_call; /* capacity of the per-stream staging buffer (0 = 1<<20)      */
    uint32_t max_frames_per_call;/* per stream (0 = 8)                                         */
    uint32_t trace_capacity;     /* per-stream lora_b200_step records kept per call (0 = none) */
} lora_b200_config;

typedef struct lora_b200_decoder lora_b200_decoder;

/* one state-machine step, for parity tests against the oracle's work() trace */
typedef struct lora_b200_step {
    int32_t state;       /* state at entry of the step                        */
    int32_t consumed;    /* what the reference would pass to consume_each      */
    int32_t bin;         /* raw demodulated bin, -1 when the step has none     */
    int32_t fine_sync;   /* d_fine_sync after the step                         */
    float   metric;      /* autocorr (DETECT), max corr (SYNC), pearson (FIND_SFD) */
} lora_b200_step;

/* Frame callback: replaces message_port_pub("frames", blob) (decoder_impl.cc:607-608).
 * `frame` = 15-byte loratap header | 3-byte loraphy header | payload (decoder_impl.cc:588-601);
 * valid only during the callback. */
typedef void (*lora_b200_frame_cb)(void *user, uint32_t stream, const uint8_t *frame, size_t len);

/* ---- lifecycle: decoder::make / ~decoder_impl (decoder_impl.cc:41-139) ---- */
lora_b200_decoder *lora_b200_create(const lora_b200_config *cfg);
void lora_b200_destroy(lora_b200_decoder *d);
/* Every stream back to the state of a freshly made block (DETECT, empty power queue, no partial frame, counters 0): what
 * stopping and restarting the flowgraph does to decoder_impl's members (:55-66).  Device buffers and tables are kept. */
int lora_b200_reset(lora_b200_decoder *d);
const char *lora_b200_last_error(void);
int lora_b200_abi_version(void);

/* derived parameters (decoder_impl.cc:69-91) and the constructor's stdout banner (:93-103) */
uint32_t lora_b200_samples_per_symbol(const lora_b200_decoder *d);
uint32_t lora_b200_bins(const lora_b200_decoder *d);
uint32_t lora_b200_decimation(const lora_b200_decoder *d);
int lora_b200_banner(const lora_b200_decoder *d, char *buf, size_t cap);
/* set_sf / set_samp_rate are unsupported at run time in the reference too (:905-915): they
 * return LORA_B200_EUNSUPPORTED and leave the decoder untouched. */
int lora_b200_set_sf(lora_b200_decoder *d, uint8_t sf);
int lora_b200_set_samp_rate(lora_b200_decoder *d, float samp_rate);

/* ---- chirp / twiddle tables (build_ideal_chirps, decoder_impl.cc:141-175) ----
 * One contiguous device blob: downchirp cf32[sps] | upchirp cf32[sps] | down_ifreq f32[sps] |
 * up_ifreq f32[sps] | up_ifreq_v f32[3*sps] | FFT twiddles cf32[sps].  Rank 0 builds it, the
 * other ranks receive it by ONE ncclBroadcast at init (SURVEY.md 8e) and call _commit. */
size_t lora_b200_tables_bytes(const lora_b200_decoder *d);
/* host-only: build the blob for `cfg` into dst (no device needed); returns its size in bytes
 * (dst == NULL: size query), 0 on error.  Layout: the six arrays above, back to back,
 * total rounded up to 256 bytes. */
size_t lora_b200_tables_build_host(const lora_b200_config *cfg, void *dst, size_t cap);
void *lora_b200_tables_device_ptr(lora_b200_decoder *d);
int lora_b200_tables_export(const lora_b200_decoder *d, void *host_dst, size_t cap);
int lora_b200_tables_import(lora_b200_decoder *d, const void *host_src, size_t bytes);
/* after writing the device blob in place (e.g. ncclBroadcast into lora_b200_tables_device_ptr):
 * refresh the host copy and the constants derived from it */
int lora_b200_tables_commit(lora_b200_decoder *d);

/* ---- K1: dechirp + FFT + argmax on aligned symbol windows (get_shift_fft, :430-464) ----
 * iq: n_symbols * sps interleaved cf32.  bins[i] in [0, N), mags[i] = |tmp[bin]| (may be NULL).
 * _dev: all pointers are device pointers, the launch is asynchronous on `cuda_stream`
 * (a cudaStream_t passed as void*, NULL = default stream).
 * _host: host pointers; copies (pinned, chunked, overlapped with compute) are inside. */
int lora_b200_demod_fft_dev(lora_b200_decoder *d, const void *iq, size_t n_symbols,
                            uint32_t *bins, float *mags, void *cuda_stream);
int lora_b200_demod_fft_host(lora_b200_decoder *d, const void *iq, size_t n_symbols,
                             uint32_t *bins, float *mags);
/* SDR-native ingest: iq_sc16 = interleaved little-endian int16 I/Q (what a USRP / file source delivers before the
 * host-side conversion to gr_complex); the device converts x * scale right after the copy, so PCIe moves 4 instead of
 * 8 bytes per sample.  Results equal lora_b200_demod_fft_host on the host-converted buffer bit for bit. */
int lora_b200_demod_fft_host_sc16(lora_b200_decoder *d, const void *iq_sc16, float scale, size_t n_symbols,
                                  uint32_t *bins, float *mags);
/* K2: max_frequency_gradient_idx on aligned windows (:466-491), same layout */
int lora_b200_demod_gradient_dev(lora_b200_decoder *d, const void *iq, size_t n_symbols,
                                 uint32_t *bins, void *cuda_stream);
/* A3: instantaneous_frequency (:224-244) of n_windows windows of `window` gr_complex each (window a multiple of 128),
 * out[n_windows][window] floats; the last value of a window repeats the one before it (:243).  The arg() per sample is
 * the stream kernels' own (1.8 ulp; the values agree with libm-based ones to 1e-6 rad); device pointers, async on cuda_stream. */
int lora_b200_ifreq_dev(lora_b200_decoder *d, const void *iq, size_t n_windows, uint32_t window, float *out, void *cuda_stream);

/* ---- synthetic transmitter / channel on the device (SURVEY 8(f) N3; the reference is a receiver only) ----
 * tx_symbols: n_symbols aligned data symbols, out[s][n] = up[(n + decim * values[s]) mod sps] * e^{j 2 pi cfo_hz[s] n / fs}
 *   + noise_sigma * (N(0,1) + j N(0,1)).  up_table = device cf32[sps] or NULL for the decoder's own ideal up-chirp
 *   (lib/decoder_impl.cc:149-160: (1 + 1j) e^{j phase}, i.e. amplitude sqrt 2); cfo_hz = device float[n_symbols] or NULL; noise_sigma = 0: no noise.  The noise is a
 *   counter-based generator (Philox4x32-10) keyed by `seed`: the same call gives the same samples on any launch geometry.
 * tx_expand: n_streams concurrent channels from k base captures, out[s] = base[s mod k] + the stream's own noise
 *   (base device cf32[k][n_items], n_items even).  Device pointers, async on cuda_stream. */
int lora_b200_tx_symbols_dev(lora_b200_decoder *d, const void *up_table, const uint32_t *values, const float *cfo_hz,
                             float noise_sigma, uint64_t seed, size_t n_symbols, void *out, void *cuda_stream);
int lora_b200_tx_expand_dev(lora_b200_decoder *d, const void *base, uint32_t k, size_t n_items, float noise_sigma, uint64_t seed,
                            size_t n_streams, void *out, void *cuda_stream);

/* ---- K8: integer decode of whole code-word vectors (decode(), :567-586, B2-B4) ----
 * For each of n_vec vectors: codewords[i*stride .. +lengths[i]) -> deshuffle, dewhiten,
 * Hamming decode.  out[i*out_stride ..]; out_len[i] = bytes produced.  cr[i] = d_phdr.cr,
 * is_header[i] as in decode(is_header).  Device pointers, async on cuda_stream. */
int lora_b200_decode_codewords_dev(lora_b200_decoder *d, const uint8_t *codewords, const uint32_t *lengths,
                                   size_t stride, const uint8_t *cr, const uint8_t *is_header, size_t n_vec,
                                   uint8_t *out, size_t out_stride, uint32_t *out_len, void *cuda_stream);
/* B1 + Gray: words (u32, one per symbol) of one interleaver block -> ppm code words; batch of blocks */
int lora_b200_deinterleave_dev(lora_b200_decoder *d, const uint32_t *words, uint32_t n_words, uint32_t ppm,
                               size_t n_blocks, uint8_t *codewords, void *cuda_stream);

/* ---- the drop-in: decoder_impl::work (decoder_impl.cc:740-903) ----
 * Feeds `n_items` cf32 items of stream `stream` (HOST pointer, as GNU Radio hands them to
 * work(); not retained after return).  Runs the whole state machine on the GPU for as many
 * steps as fit (each step needs 2*sps items of look-ahead, the block's output_multiple :91),
 * sets *consumed to the number of items the caller must drop (the sum of the reference's
 * consume_each() calls) and invokes cb once per completed frame, in order.
 * The caller re-presents the unconsumed tail at the start of the next call. */
int lora_b200_work(lora_b200_decoder *d, uint32_t stream, const void *iq_host, size_t n_items,
                   size_t *consumed, lora_b200_frame_cb cb, void *user);
/* Same for all streams at once: iq is [n_streams][n_items] (row stride `stride_items`).
 * host_ptr != 0: iq is host memory (copied inside); 0: iq is device memory. */
int lora_b200_work_batch(lora_b200_decoder *d, const void *iq, size_t n_items, size_t stride_items,
                         int host_ptr, size_t *consumed /* [n_streams] */, lora_b200_frame_cb cb, void *user);
/* the same with int16 I/Q input (see lora_b200_demod_fft_host_sc16); frames, consume amounts and stdout equal those of
 * lora_b200_work_batch on the host-converted buffer. */
int lora_b200_work_batch_sc16(lora_b200_decoder *d, const void *iq_sc16, float scale, size_t n_items, size_t stride_items,
                              int host_ptr, size_t *consumed /* [n_streams] */, lora_b200_frame_cb cb, void *user);
/* ... and with int8 I/Q (interleaved signed bytes, GNU Radio's interleaved_char_to_complex followed by a multiply):
 * a quarter of the gr_complex bytes over PCIe, the only lever left once the copy is the bound. */
int lora_b200_work_batch_sc8(lora_b200_decoder *d, const void *iq_sc8, float scale, size_t n_items, size_t stride_items,
                             int host_ptr, size_t *consumed /* [n_streams] */, lora_b200_frame_cb cb, void *user);
/* Bulk access to what the last work / work_batch call published, for hosts that drain thousands of streams per call and do
 * not want one callback per frame (cb may be NULL then): records in delivery order (by stream, then by sequence), valid
 * until the next work call on this decoder.  `bytes` = loratap | loraphy | payload, `len` of them valid
 * (decoder_impl.cc:588-601); hdr_print = the header bytes the reference prints first (:832). */
#define LORA_B200_MAX_FRAME_BYTES 564
typedef struct lora_b200_frame {
    uint32_t stream, seq, len;
    uint8_t  n_hdr_print;
    uint8_t  hdr_print[4];
    uint8_t  pad[3];
    uint8_t  bytes[LORA_B200_MAX_FRAME_BYTES];
} lora_b200_frame;
size_t lora_b200_frames_last(lora_b200_decoder *d, const lora_b200_frame **frames);
/* current state of a stream (LORA_B200_DETECT ...) */
int lora_b200_stream_state(lora_b200_decoder *d, uint32_t stream);
/* N4 (SURVEY.md 8f): the CFO estimate the reference computes in experimental_determine_cfo (lib/decoder_impl.cc:730-738:
 * instantaneous frequency of samples x downchirp at index 256 of the synchronised preamble symbol, in Hz) and would
 * publish as ("cfo" . x) on its "control" port for the channelizer (:774-776, commented out there; consumer
 * lib/controller_impl.cc:52-57 -> channelizer_impl::apply_cfo).  Off by default: nothing observable changes.  With it
 * enabled every SYNC step stores the estimate; _last_cfo returns the latest one and how many there have been, for the
 * host to forward to lora_b200_channelizer_apply_cfo. */
int lora_b200_set_cfo_estimate(lora_b200_decoder *d, int enable);
int lora_b200_last_cfo(lora_b200_decoder *d, uint32_t stream, float *cfo_hz, uint32_t *count);
/* the reference's std::cout hex lines for the frames delivered by the last work call of this
 * stream (" 04 90 40" + " de ad ... (ascii)\n", decoder_impl.cc:832,872) */
int lora_b200_stdout_last(lora_b200_decoder *d, uint32_t stream, char *buf, size_t cap);
/* per-step trace of the last work call (needs trace_capacity > 0) */
int lora_b200_trace_read(lora_b200_decoder *d, uint32_t stream, lora_b200_step *steps, size_t cap, size_t *n);

/* ---- N1 (SURVEY.md 8f): the channelizer in front of the decoder -------------------------------------
 * Replaces lora::channelizer::make(samp_rate, center_freq, channel_list, bandwidth, decimation)
 * (include/lora/channelizer.h:49, lib/channelizer_impl.cc:40-60): GNU Radio's
 * freq_xlating_fir_filter_ccf with firdes::low_pass(1, fs, bw/2 + 15000, 10000, Hamming) taps.  The
 * reference wires only channel_list[0]; here every listed channel is produced by one FIR-bank launch:
 * out[ch][n] for n < n_in / decimation (device pointers, async on cuda_stream).  Filter history and
 * rotator phase carry over between calls like a GNU Radio block's. */
typedef struct lora_b200_channelizer lora_b200_channelizer;
lora_b200_channelizer *lora_b200_channelizer_create(float samp_rate, float center_freq, const float *channel_list,
                                                    uint32_t n_channels, uint32_t bandwidth, uint32_t decimation,
                                                    int32_t device);
void lora_b200_channelizer_destroy(lora_b200_channelizer *c);
const char *lora_b200_channelizer_last_error(void);
uint32_t lora_b200_channelizer_ntaps(const lora_b200_channelizer *c);
int lora_b200_channelizer_taps(const lora_b200_channelizer *c, float *out, size_t cap);
/* channelizer_impl::apply_cfo (lib/channelizer_impl.cc:68-71), driven by the "cfo" control message
 * (lib/controller_impl.cc:52-57) */
int lora_b200_channelizer_apply_cfo(lora_b200_channelizer *c, uint32_t channel, float cfo);
/* conj != 0: every output sample is conjugated on its way out -- the blocks.conjugate_cc that lora_receiver(conj=True)
 * wires between the channelizer and the decoder (python/lora_receiver.py:50,70-75), without a host round trip */
int lora_b200_channelizer_set_conjugate(lora_b200_channelizer *c, int conj);
int lora_b200_channelizer_work_dev(lora_b200_channelizer *c, const void *in_dev, size_t n_in, void *out_dev,
                                   size_t out_stride, size_t *n_out, void *cuda_stream);
/* host entry: uploads `in_host`, filters into an internal device buffer; _output() returns the DEVICE
 * pointer of one channel's n_out items (valid until the next call) so the decoder can consume it
 * without a host round trip (lora_b200_work_batch(..., host_ptr = 0)). */
int lora_b200_channelizer_work_host(lora_b200_channelizer *c, const void *in_host, size_t n_in, size_t *n_out);
const void *lora_b200_channelizer_output(const lora_b200_channelizer *c, uint32_t channel, size_t *stride_items);
/* host copy of one channel's output of the last _work_host call (what a GNU Radio block's work() hands downstream) */
int lora_b200_channelizer_read_output(const lora_b200_channelizer *c, uint32_t channel, void *host_dst, size_t n_items);
uint64_t lora_b200_channelizer_launch_count(const lora_b200_channelizer *c);

/* ---- N4 (SURVEY.md 8f): the gateway receiver -- every channel AND every spreading factor of a wideband capture --------
 * Wideband IQ in, chunk by chunk; the frames of every (channel, SF) out, one call per chunk, the IQ staying in device
 * memory.  A call runs the channelizer above over the chunk (the same entry point, so every channel's samples are those a
 * standalone lora_b200_channelizer fed the same chunks produces), appends each channel's new samples to the items every
 * SF's decoder left unconsumed in the previous call, and runs one decoder per SF (lora_b200_create with
 * n_streams = n_channels, samp_rate / decimation) on all channels, the SFs concurrently.  Each (channel, SF) stream decodes
 * exactly what lora_b200_work on that channel's samples decodes. */
typedef struct lora_b200_gateway lora_b200_gateway;
typedef struct lora_b200_gateway_config {
    float        samp_rate;          /* wideband rate                                                               */
    float        center_freq;
    const float *channel_list;       /* n_channels absolute frequencies, as lora_b200_channelizer_create              */
    uint32_t     n_channels;
    uint32_t     bandwidth;
    uint32_t     decimation;         /* decoders run at samp_rate / decimation                                        */
    uint32_t     sf_mask;            /* bit s set: decode SF s (7..12) on every channel                               */
    uint32_t     reduced_rate_mask;  /* bit s set: reduced_rate for SF s; 0 = LoRa's default at 125 kHz (SF11, SF12) */
    uint8_t      implicit, cr, crc, demod;   /* as lora_b200_config, shared by all SFs                               */
    uint8_t      conj;               /* conjugate on the way out of the FIR bank (lora_receiver conj=True)            */
    uint8_t      disable_drift_correction;
    uint8_t      reserved[2];
    int32_t      device;
    uint32_t     max_in_per_call;    /* wideband items per call (0 = 1<<22)                                          */
    uint32_t     max_frames_per_call;/* per (channel, SF) stream (0 = 8)                                              */
} lora_b200_gateway_config;

typedef struct lora_b200_gateway_frame {
    uint32_t channel;                /* index into channel_list */
    uint32_t sf;
    lora_b200_frame frame;           /* frame.stream == channel */
} lora_b200_gateway_frame;

/* The arguments are checked before a device is looked for (EINVAL via lora_b200_last_error). */
lora_b200_gateway *lora_b200_gateway_create(const lora_b200_gateway_config *cfg);
void lora_b200_gateway_destroy(lora_b200_gateway *g);
/* decoders AND channelizer history / rotator back to the state of a fresh gateway */
int lora_b200_gateway_reset(lora_b200_gateway *g);
/* n_in: a multiple of decimation, <= max_in_per_call; host_ptr as lora_b200_work_batch.  *n_frames = frames decoded.
 * LORA_B200_EOVERFLOW (nothing consumed, nothing changed): a stream's unconsumed items plus this chunk would not fit its
 * buffer -- only possible when a stream stopped at max_frames_per_call; a smaller chunk fits. */
int lora_b200_gateway_work(lora_b200_gateway *g, const void *iq, size_t n_in, int host_ptr, size_t *n_frames);
/* the frames of the last work call, ordered by (sf ascending, channel, seq); valid until the next call */
size_t lora_b200_gateway_frames_last(lora_b200_gateway *g, const lora_b200_gateway_frame **frames);
/* progress of one stream: items consumed since create/reset, and items held over for the next call */
int lora_b200_gateway_position(lora_b200_gateway *g, uint32_t channel, uint32_t sf, uint64_t *consumed, uint32_t *pending);
/* where the last work call spent its device time, from CUDA events, in ms: [0] host-to-device copy, [1] channelizer,
 * [2] gather, [3] the decoders' state machines (all SFs, concurrently) */
int lora_b200_gateway_timing(const lora_b200_gateway *g, float *ms, size_t n);

/* how many kernels this library has launched since creation (bench.py's gpu_launches) */
uint64_t lora_b200_launch_count(const lora_b200_decoder *d);

#ifdef __cplusplus
}
#endif
#endif /* LORA_B200_H */
