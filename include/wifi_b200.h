/*
 * wifi_b200.h -- C ABI of libwifi_b200.so, the B200 (sm_100a) 802.11a/g OFDM
 * baseband that stands in for the `wifi_phy_hier` hierarchical block of
 * OedonLestrange42/GNURadio-WiFI-ImageTransfer.
 *
 * Reference interface replaced (all paths under /root/reference):
 *   gnu_radio/wifi_phy_hier.grc:641-660   stream in  `samp_in`   -> wifi_b200_rx_push / _rx_batch[_dev]
 *   gnu_radio/wifi_phy_hier.grc:623-640   msg out    `mac_out`   -> wifi_b200_rx_pop  / _rx_frames + _rx_psdus
 *   gnu_radio/wifi_phy_hier.grc:605-622   msg out    `carrier`   -> wifi_b200_rx_rows (equalised points)
 *   gnu_radio/wifi_phy_hier.grc:661-680   msg in     `mac_in`    -> wifi_b200_tx[_dev]
 *   gnu_radio/wifi_phy_hier.grc:587-604   stream out `samp_out`  -> iq_out of wifi_b200_tx[_dev]
 *   gnu_radio/wifi_phy_hier.grc:83-99,299-315,442-458,501-517,681-697
 *                                         params bandwidth, chan_est, encoding, frequency, sensitivity
 *                                                                -> wifi_b200_cfg / wifi_b200_set_param
 *   gnu_radio/IRS_tranceiver.py:178-184   constructor call       -> wifi_b200_create
 *   gnu_radio/IRS_tranceiver.py:386,427,442  set_bandwidth/_frequency/_encoding -> wifi_b200_set_param
 *   gnu_radio/IRS_tranceiver.py:271       ieee802_11.mac framing -> wifi_b200_mac_frame
 *   gnu_radio/IRS_tranceiver.py:282-288   channels.channel_model (loopback test channel)
 *                                                                -> wifi_b200_channel_dev (Philox)
 *
 * Conventions: plain C, no callbacks, no C++/torch types.  "iq" buffers are
 * interleaved float32 I,Q (GNU Radio gr_complex).  `_dev` entry points take
 * device pointers (same GPU as the handle) and never touch PCIe.  The caller
 * owns every buffer it passes; the library owns its device workspace and one
 * CUDA stream per handle.  A handle is single-owner (calls are serialised by an
 * internal mutex).  There is no CPU fallback: create() fails with
 * WIFI_E_NODEVICE when no sm_100 device is present.
 * Every call returns >= 0 on success or a negative wifi_b200_err code.
 */
#ifndef WIFI_B200_H
#define WIFI_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define WIFI_B200_ABI_VERSION 1

typedef enum wifi_b200_err {
    WIFI_OK = 0,
    WIFI_E_ARG = -1,        /* bad argument / enum out of range                                 */
    WIFI_E_TOO_LARGE = -2,  /* PSDU > 1528 B or > 511 symbols (upstream mapper throws)           */
    WIFI_E_CUDA = -3,       /* CUDA runtime error, see wifi_b200_last_error                       */
    WIFI_E_NOMEM = -4,
    WIFI_E_OVERFLOW = -5,   /* more samples / frames than the handle's capacity, or caller buffer too small */
    WIFI_E_NODEVICE = -6    /* no sm_100 GPU                                                     */
} wifi_b200_err;

/* ieee802_11.Encoding (IRS_tranceiver.py:129-131) and ieee802_11.Equalizer (:154-156) */
enum { WIFI_BPSK_1_2 = 0, WIFI_BPSK_3_4, WIFI_QPSK_1_2, WIFI_QPSK_3_4, WIFI_QAM16_1_2, WIFI_QAM16_3_4, WIFI_QAM64_2_3, WIFI_QAM64_3_4 };
enum { WIFI_EQ_LS = 0, WIFI_EQ_LMS = 1, WIFI_EQ_COMB = 2, WIFI_EQ_STA = 3 };
/* ids for wifi_b200_set_param: the hier block's parameters */
enum { WIFI_P_BANDWIDTH = 0, WIFI_P_FREQUENCY = 1, WIFI_P_SENSITIVITY = 2, WIFI_P_CHAN_EST = 3, WIFI_P_ENCODING = 4,
       WIFI_P_MIN_PLATEAU = 5, WIFI_P_WANT_CARRIER = 6, WIFI_P_SOFT_DECISION = 7,
       /* streaming only: wifi_b200_rx_push buffers until this many new samples wait (0 = run on every push).  A run
        * costs 1-3 ms whatever its size, so a live 20 Msps stream wants 65536 or more; results are unchanged.
        * An empty push (n = 0, flush = 0) runs the pipeline on whatever is buffered without ending the stream. */
       WIFI_P_STREAM_BATCH = 8,
       /* host-input batch calls (rx_batch, rx_batch_sc16) process the links in groups so that the copy of one group overlaps
        * the decoding of the previous one; a group is closed when it holds this many samples (0 = about 128 MB of host
        * bytes, the default).  Results do not depend on it. */
       WIFI_P_HOST_GROUP_SAMPLES = 9,
       /* which form of the hard-decision Viterbi kernel decodes a call's frames: 0 = by frame count (default), 1 = one
        * trellis per warp (a handful of frames), 2 = per four lanes (a few thousand), 3 = per thread (tens of thousands).
        * The three are the same decoder and give identical bytes; the id exists for tests and measurements. */
       WIFI_P_VITERBI_FORM = 10 };

typedef struct wifi_b200_cfg {
    double bandwidth;      /* Hz, hier default 10e6 (wifi_phy_hier.grc:92)                        */
    double frequency;      /* Hz, hier default 5.89e9 (:510)                                     */
    double sensitivity;    /* sync_short threshold, 0.56 (:690)                                  */
    int32_t chan_est;      /* WIFI_EQ_* (:308)                                                   */
    int32_t encoding;      /* WIFI_* MCS used by tx when enc == NULL (:451)                      */
    int32_t min_plateau;   /* 2 (:725)                                                           */
    int32_t device;        /* CUDA device ordinal                                                */
    int32_t want_carrier;  /* keep the equalised constellation points (`carrier` port)            */
    int32_t soft_decision; /* 0: hard decisions as the reference; 1: max-log LLR demapper + soft Viterbi (DESIGN.md 9) */
    int64_t max_samples;   /* capacity of one rx call, complex samples summed over links          */
    int64_t max_frames;    /* capacity of one rx/tx call, frames (sync_short triggers)            */
} wifi_b200_cfg;

/* one record per sync_short trigger; field meaning identical to the oracle's orc_frame */
typedef struct wifi_b200_frame {
    int64_t trigger;       /* sample index (within its link's stream) of the wifi_start tag       */
    int32_t link;
    int32_t burst_len;     /* samples sync_short copied for the tag (<= 43200)                    */
    float   freq_short;    /* coarse CFO, rad/sample                                             */
    float   freq_long;     /* sync_long fine CFO in force, rad/sample                            */
    int32_t found;         /* 0 or the LTS peak distance 63/64/65                                 */
    int32_t frame_start;
    int32_t n_syms;        /* 64-sample symbols handed to the equalizer                           */
    int32_t sig_ok;
    int32_t encoding;
    int32_t length;        /* PSDU bytes from SIGNAL                                             */
    int32_t frame_symbols;
    int32_t n_rows;        /* data symbols the equalizer emitted                                  */
    int32_t accepted;      /* decode_mac accepted the tag                                        */
    int32_t decoded;       /* decode_mac collected all symbols and decoded                        */
    int32_t crc_ok;        /* FCS residue == 0x2144DF1C: a PDU is published on mac_out            */
    double  snr;           /* dB, equalizer estimate                                             */
    int64_t row_off;       /* first row of this frame in the rows / carrier arrays                */
    int64_t psdu_off;      /* byte offset of the decoded PSDU (incl. FCS) in the psdu store, -1 if none */
} wifi_b200_frame;

typedef struct wifi_b200_stats {
    int64_t samples, frames_detected, signal_ok, decoded, crc_ok, pdu_bytes;
    int64_t per_mcs_crc_ok[8];
} wifi_b200_stats;

/* synthetic test channel, one descriptor per output segment (see DESIGN.md "channel") */
typedef struct wifi_b200_chan_seg {
    int64_t in_off, in_len;   /* input segment (complex samples); reads outside are 0             */
    int64_t out_off, n;       /* output segment                                                   */
    int64_t n0;               /* Philox counter of output sample 0                                */
    float gain, cfo, phase0, noise_sigma;
    int32_t n_taps;
    int32_t delay[8];
    float tap_re[8], tap_im[8];
    uint64_t seed, stream;
} wifi_b200_chan_seg;

/* Time-varying multipath fading for one segment of wifi_b200_channel_fading_dev (DESIGN.md "fading channel"):
 *     y(i) = gain * sum_t h_t(t0 + i) * x(i - delay[t]),  then the segment's CFO rotation and AWGN as in wifi_b200_channel_dev.
 * Every tap is a sum of n_sin sinusoids with complex Gaussian weights and Clarke-spread frequencies (|f| <= doppler); tap 0
 * adds a line-of-sight term of Rician factor k_factor.  doppler = 0 gives block fading, one CN(0, power[t]) value per tap.
 * The realisation depends only on (seed, stream); t0 places the segment in time, so segments that share (seed, stream)
 * and set t0 to their position form one continuous channel.  Phases are 32-bit NCOs: the process repeats every 2^32
 * samples.  112 bytes, no implicit padding. */
typedef struct wifi_b200_fading {
    int32_t n_taps;           /* 1..8                                                              */
    int32_t n_sin;            /* sinusoids per tap, 1..16                                           */
    int32_t delay[8];         /* samples, >= 0                                                     */
    float power[8];           /* E|h_t|^2, linear, >= 0                                            */
    float k_factor;           /* Rician K of tap 0, linear, >= 0 (0: Rayleigh)                     */
    float doppler;            /* maximum Doppler f_d / f_s, cycles/sample, 0 .. 0.25               */
    float los_doppler;        /* Doppler of the line-of-sight term, cycles/sample, -0.25 .. 0.25    */
    int32_t reserved;         /* 0                                                                 */
    int64_t t0;               /* time index of output sample 0                                     */
    uint64_t seed, stream;    /* Philox key and counter words of the realisation                    */
} wifi_b200_fading;

typedef struct wifi_b200 wifi_b200_t;

int  wifi_b200_abi_version(void);
int  wifi_b200_device_count(void);   /* number of visible sm_100 devices */
int  wifi_b200_create(const wifi_b200_cfg *cfg, wifi_b200_t **out);
void wifi_b200_destroy(wifi_b200_t *h);
int  wifi_b200_set_param(wifi_b200_t *h, int id, double value);
double wifi_b200_get_param(wifi_b200_t *h, int id);
const char *wifi_b200_last_error(wifi_b200_t *h);
const char *wifi_b200_strerror(int code);
/* CUDA stream of the handle (cudaStream_t as void*), for callers that enqueue their own work */
void *wifi_b200_stream(wifi_b200_t *h);
int  wifi_b200_sync(wifi_b200_t *h);

/* ---- MAC framing helper: [UPSTREAM] mac.cc generate_mac_data_frame ---- */
int  wifi_b200_mac_frame(const uint8_t *payload, int n, int seq, const uint8_t src[6], const uint8_t dst[6],
                         const uint8_t bss[6], uint8_t *psdu_out /* n + 28 bytes */);
int  wifi_b200_n_sym(int encoding, int psdu_len);
int  wifi_b200_frame_samples(int encoding, int psdu_len);   /* 80*(5+N_SYM)+1 */

/* ---- TX: mac_in -> samp_out.  PSDUs (with FCS) are psdu_blob[off[i] .. off[i]+len[i]).
 * enc/seed may be NULL: the handle's encoding and its running scrambler seed (1..127, mapper.cc)
 * are used.  Burst i occupies iq_out[burst_off[i] .. burst_off[i+1]) complex samples;
 * burst_off has n+1 entries.  Returns total samples. */
int64_t wifi_b200_tx(wifi_b200_t *h, const uint8_t *psdu_blob, const uint32_t *off, const uint32_t *len,
                     const uint8_t *enc, const uint8_t *seed, int n, float *iq_out, size_t cap_samples,
                     uint64_t *burst_off);
int64_t wifi_b200_tx_dev(wifi_b200_t *h, const uint8_t *psdu_blob, const uint32_t *off, const uint32_t *len,
                         const uint8_t *enc, const uint8_t *seed, int n, float *iq_out_dev, size_t cap_samples,
                         uint64_t *burst_off);
/* data-carrier indices the mapper produced for the last tx call: n_sym*48 bytes per frame, frames back to back */
int64_t wifi_b200_tx_symbols(wifi_b200_t *h, uint8_t *out, size_t cap);

/* ---- synthetic channel on device buffers ---- */
int  wifi_b200_channel_dev(wifi_b200_t *h, const float *in_dev, float *out_dev, const wifi_b200_chan_seg *segs, int n_segs);
/* same with host buffers (in: in_len complex samples, out: out_len, zero where no segment writes) */
int  wifi_b200_channel(wifi_b200_t *h, const float *in_host, int64_t in_len, float *out_host, int64_t out_len,
                       const wifi_b200_chan_seg *segs, int n_segs);
/* the same with fading taps: segment i takes its taps from fades[i] (segs[i].n_taps must be 0); everything else in segs[i]
 * keeps its meaning.  Out-of-range fields give WIFI_E_ARG before anything is written. */
int  wifi_b200_channel_fading_dev(wifi_b200_t *h, const float *in_dev, float *out_dev, const wifi_b200_chan_seg *segs,
                                  const wifi_b200_fading *fades, int n_segs);
int  wifi_b200_channel_fading(wifi_b200_t *h, const float *in_host, int64_t in_len, float *out_host, int64_t out_len,
                              const wifi_b200_chan_seg *segs, const wifi_b200_fading *fades, int n_segs);

/* ---- RX, batch form: n_links independent streams; link l is iq[link_off[l] .. link_off[l+1]) complex
 * samples.  final != 0: the streams end here (flush).  Results stay in the handle until the next rx call. */
int  wifi_b200_rx_batch(wifi_b200_t *h, const float *iq_host, const uint64_t *link_off, int n_links, int final);
int  wifi_b200_rx_batch_dev(wifi_b200_t *h, const float *iq_dev, const uint64_t *link_off, int n_links, int final);
/* The same for streams that are RESUMED in the middle (one long capture cut into segments that different GPUs decode,
 * SURVEY 8e): per link the state sync_short / sync_long carry across the cut.  With the state of the sequential
 * receiver at the cut, a segment's frames equal the sequential receiver's from there on. */
typedef struct wifi_b200_link_state {
    int64_t min_pos;   /* first sample index (relative to link_off[l]) sync_short may trigger on: previous trigger + 481; 0: none */
    float   fo_carry;  /* sync_long's d_freq_offset entering the segment (freq_long of the last burst before it), 0 at a stream start */
    int32_t hist;      /* valid samples stored in front of link_off[l] in the buffer (front-end history, up to 256) */
} wifi_b200_link_state;
int  wifi_b200_rx_batch_dev_state(wifi_b200_t *h, const float *iq_dev, const uint64_t *link_off, int n_links, int final,
                                  const wifi_b200_link_state *state /* n_links entries */);
/* Same from the radio's wire format: interleaved int16 I/Q (what uhd.usrp_source / the HackRF deliver before
 * the host driver converts to fc32; gnu_radio/IRS_AP.py:163-177 asks UHD for cpu_format "fc32").  The GPU forms
 * x = (float)i16 * scale, one rounding per component -- exactly UHD's sc16 -> fc32 host converter -- so the
 * result equals wifi_b200_rx_batch on the host-converted samples while the capture crosses PCIe at 4 B/sample. */
int  wifi_b200_rx_batch_sc16(wifi_b200_t *h, const int16_t *iq_host, float scale, const uint64_t *link_off, int n_links, int final);
int  wifi_b200_rx_counts(wifi_b200_t *h, int64_t *n_frames, int64_t *n_rows, int64_t *n_pdus, int64_t *psdu_store_bytes);
int  wifi_b200_rx_frames(wifi_b200_t *h, wifi_b200_frame *out, int64_t cap);
int  wifi_b200_rx_rows(wifi_b200_t *h, uint8_t *rows /* n_rows*48 or NULL */, float *carrier /* n_rows*96 or NULL */, int64_t cap_rows);
int  wifi_b200_rx_psdus(wifi_b200_t *h, uint8_t *store, size_t cap);
/* soft mode: int8 soft value per coded bit, 288 per row (first N_CBPS used, order carrier*N_BPSC+bit) */
int  wifi_b200_rx_soft(wifi_b200_t *h, int8_t *soft, int64_t cap_rows);
/* autocorrelation front-end decisions for one link: bit n of flags = (c[n] > sensitivity) */
int  wifi_b200_rx_flags(wifi_b200_t *h, int link, uint32_t *flags, int64_t cap_words);

/* ---- RX, streaming form (one continuous stream per handle): samp_in -> mac_out ---- */
int  wifi_b200_rx_push(wifi_b200_t *h, const float *iq_host, size_t n, int flush);
/* pops CRC-ok frames in stream order; psdu_buf receives PSDUs without FCS back to back,
 * meta[i].psdu_off is the offset into psdu_buf, meta[i].length-4 the size; trigger is absolute */
int  wifi_b200_rx_pop(wifi_b200_t *h, wifi_b200_frame *meta, int cap, uint8_t *psdu_buf, size_t psdu_cap, int *n_frames);
/* The same frames without a copy: *meta points at *n_frames records and *psdu_bytes at the (page-locked) buffer the copy
 * engine delivered their PSDUs into; record i's PSDU is (*psdu_bytes)[meta[i].psdu_off .. + meta[i].length - 4) (the
 * offsets are NOT back to back), *n_bytes is the extent of that buffer.  One call returns the results of one pipeline
 * run (the oldest not yet popped; call until *n_frames == 0).  The pointers stay valid until the next call on this
 * handle, which is also when the frames leave the queue. */
int  wifi_b200_rx_pop_view(wifi_b200_t *h, const wifi_b200_frame **meta, const uint8_t **psdu_bytes, size_t *n_bytes, int *n_frames);
int  wifi_b200_rx_reset(wifi_b200_t *h);
/* The same for n_links continuous streams at once (many live channels on one GPU share one pipeline run): link l
 * receives iq_host[link_off[l] .. link_off[l+1]) new complex samples (possibly none).  The number of links is fixed by
 * the first push after create / rx_reset; popped frames carry their link in wifi_b200_frame.link and come out ordered
 * by (run, link, trigger).  flush ends every stream.  Every link owns max_samples / n_links samples of a device
 * arena: size max_samples >= n_links * (largest push or stream batch + 2 * 43200 + 512) so that a held burst, a
 * deferred one in front of it and the next push fit (WIFI_E_OVERFLOW otherwise; nothing is dropped silently). */
int  wifi_b200_rx_push_links(wifi_b200_t *h, const float *iq_host, const uint64_t *link_off, int n_links, int flush);

/* Asynchronous form for callers that fill page-locked buffers in turn (an SDR driver's ring): _async queues the
 * host -> device copy of this push on the handle's copy stream and returns at once; the buffer must stay untouched until
 * the wifi_b200_rx_push_wait that completes this push.  _wait takes the OLDEST pending push, waits for its copy, appends
 * it to the streams and runs the pipeline as wifi_b200_rx_push_links would (results through wifi_b200_rx_pop); it returns
 * 1 if it completed a push, 0 if none was pending.  At most three pushes may be pending: with
 *     async(k + 1); wait()  (completes k);  pop ...
 * the copy of push k + 1 overlaps the decoding of push k.  Results are identical to the synchronous calls. */
int  wifi_b200_rx_push_links_async(wifi_b200_t *h, const float *iq_host, const uint64_t *link_off, int n_links, int flush);
int  wifi_b200_rx_push_wait(wifi_b200_t *h);
/* The same push in the radios' wire format (int16 I/Q pairs, as wifi_b200_rx_batch_sc16: x = (float)i16 * scale, the
 * conversion UHD's sc16 -> fc32 host converter performs before uhd_usrp_source hands samples to `samp_in`): half the bytes
 * over PCIe, converted on the GPU while the samples are appended to the streams.  Completed by wifi_b200_rx_push_wait like
 * the fc32 form; the two forms may be mixed on one handle.  link_off counts complex samples. */
int  wifi_b200_rx_push_links_sc16_async(wifi_b200_t *h, const int16_t *iq_host, float scale, const uint64_t *link_off, int n_links, int flush);

int  wifi_b200_get_stats(wifi_b200_t *h, wifi_b200_stats *out);
/* device time (ms) of each pipeline stage in the last rx_batch call; names via wifi_b200_stage_name */
int  wifi_b200_stage_times(wifi_b200_t *h, float *ms, int cap);
const char *wifi_b200_stage_name(int i);

/* ---- page-locked host memory for the host-buffer entry points (rx_batch, rx_push*, tx) ----
 * cudaHostAlloc'd, so copies are plain DMA, and zero-filled from the host cores on the GPU's side of the machine
 * (/sys/bus/pci/devices/<gpu>/local_cpulist): on a multi-socket box the pages land on the NUMA node of the GPU's PCIe root. */
int  wifi_b200_host_alloc(wifi_b200_t *h, size_t bytes, void **out);
int  wifi_b200_host_free(wifi_b200_t *h, void *p);

/* ---- diagnostics (no reference counterpart) ----
 * Element-wise evaluation of the numerical contract (include/wifi_detmath.h, wdm_selftest(fn, ...)) on the GPU with host
 * buffers: tests/test_detmath.py asks for bit equality with the same call on the host.  o0 / o1 are in-out. */
int  wifi_b200_selftest_detmath(wifi_b200_t *h, int fn, const float *a, const float *b, const float *c, const float *d,
                                float *o0, float *o1, int64_t n);
/* Measured issue rate of the integer ALU pipe (independent LOP3 / IADD3 chains on every SM, `iters` x 64 instructions
 * per thread): warp-instructions per second.  bench.py quotes the Viterbi kernel's roofline against it (SURVEY 8d). */
int  wifi_b200_alu_peak(wifi_b200_t *h, int iters, double *warp_inst_per_s, double *ms);

#ifdef __cplusplus
}
#endif
#endif
