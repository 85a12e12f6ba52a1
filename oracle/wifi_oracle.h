/*
 * wifi_oracle.h -- C interface of the CPU oracle (TEST INFRASTRUCTURE ONLY).
 *
 * The oracle is a scalar, single-threaded-per-link restatement of the 802.11a/g
 * PHY that gnu_radio/wifi_phy_hier.grc wires together (gr-ieee802-11 maint-3.10
 * + GNU Radio 3.10 blocks; neither is vendored under /root/reference, see
 * SURVEY.md 8c).  It exists to CHECK libwifi_b200.so; nothing in the product
 * path may link or call it.  Only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py use it.
 *
 * PARITY UNPINNED: the reference repository holds no test, golden vector or
 * fixture for this path and its PHY cannot be built or imported here, so the
 * oracle is pinned only by the IEEE 802.11 Annex-G/I known answers, by the
 * constants written in wifi_phy_hier.grc (tests/golden/hier_constants.json) and
 * by an independent float64 numpy model (tests/ref_model.py).
 */
#ifndef WIFI_ORACLE_H
#define WIFI_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* one record per sync_short trigger (same field meaning as wifi_b200_frame) */
typedef struct orc_frame {
    int64_t trigger;      /* sample index (in the link's stream) of the sync_short tag   */
    int32_t link;
    int32_t burst_len;    /* samples sync_short copied for this tag                      */
    float   freq_short;   /* arg(a[trigger])/16                                          */
    float   freq_long;    /* sync_long d_freq_offset in force for this burst             */
    int32_t found;        /* 0: no LTS pair (frame_start=320), else the index gap 63/64/65 */
    int32_t frame_start;
    int32_t n_syms;       /* 64-sample symbols handed to the equalizer (LTS1,LTS2,SIGNAL,..) */
    int32_t sig_ok;       /* SIGNAL parity + rate valid                                  */
    int32_t encoding;
    int32_t length;       /* PSDU bytes announced by SIGNAL                              */
    int32_t frame_symbols;
    int32_t n_rows;       /* data symbols the equalizer emitted                          */
    int32_t accepted;     /* decode_mac took the tag (n_sym<=511 && len<=1528)           */
    int32_t decoded;      /* decode_mac collected n_sym symbols and ran decode()         */
    int32_t crc_ok;
    double  snr;
    int64_t row_off;      /* first row (48 B each) of this frame in the rows array       */
    int64_t psdu_off;     /* byte offset of the decoded PSDU (incl. FCS) in the psdu blob, -1 if none */
} orc_frame;

typedef struct orc_rx_cfg {
    double threshold;     /* sync_short threshold (hier: sensitivity, 0.56)   */
    int32_t min_plateau;  /* 2                                                  */
    int32_t algo;         /* 0 LS 1 LMS 2 COMB 3 STA                            */
    double freq;          /* carrier frequency, Hz                              */
    double bw;            /* bandwidth, Hz                                      */
    int32_t final;        /* 1: the stream ends with this buffer                */
    int32_t want_carrier; /* keep equalised points                              */
    int32_t soft;         /* 1: max-log LLR demapper + soft-decision Viterbi (no reference counterpart, DESIGN.md 9) */
    int32_t hist;         /* resumed stream: valid samples stored before x[0] (front-end history), 0 at a stream start */
    int64_t min_pos;      /* resumed stream: first index sync_short may trigger on (previous trigger + MIN_GAP + 1), else 0 */
    float fo_carry;       /* resumed stream: sync_long's d_freq_offset entering the buffer, else 0 */
    int32_t pad;
} orc_rx_cfg;

/* ---- tables / small pieces (for known-answer tests) ---- */
int  orc_mcs(int enc, int *n_bpsc, int *n_cbps, int *n_dbps, int *rate_field, int *punct);
int  orc_n_sym(int enc, int psdu_len);
void orc_scramble(const uint8_t *in, uint8_t *out, int n, int seed);
void orc_conv_encode(const uint8_t *in, uint8_t *out, int n);              /* out 2n */
int  orc_puncture(const uint8_t *in, uint8_t *out, int n_mother, int enc); /* returns kept */
void orc_interleave(const uint8_t *in, uint8_t *out, int n_sym, int enc, int reverse);
void orc_signal_field(int enc, int len, uint8_t *out48);
void orc_polarity(float *out127);
void orc_long_taps(float *out128);   /* LONG[64] matched-filter taps, interleaved re,im */
void orc_lts_freq(float *out64);     /* LTS in shifted order                              */
void orc_constellation(int enc, float *out_pts /* 2*2^n_bpsc */);
int  orc_decide(int enc, float re, float im);
void orc_fft64(const float *in, float *out, int inverse);  /* natural order, unnormalised */
int  orc_viterbi(const uint8_t *depunctured, int n_avail, int n_bits, int ntraceback, uint8_t *out_bits);
uint32_t orc_crc32(const uint8_t *p, int n);

/* ---- TX ---- */
int  orc_mac_frame(const uint8_t *payload, int n, int seq, const uint8_t *src, const uint8_t *dst,
                   const uint8_t *bss, uint8_t *psdu_out);                  /* returns psdu len */
int  orc_tx_symbols(const uint8_t *psdu, int len, int enc, int seed, uint8_t *out /* n_sym*48 */);
int  orc_tx_frame(const uint8_t *psdu, int len, int enc, int seed, float *iq_out, int cap_samples);

/* ---- synthetic channel (Philox), see DESIGN.md ---- */
typedef struct orc_chan_cfg {
    float gain;            /* amplitude applied to the input                     */
    float cfo;             /* rad/sample                                         */
    float phase0;          /* rad                                                */
    float noise_sigma;     /* E|n|^2 = sigma^2 (utils/channel.py:50-53 convention) */
    int32_t n_taps;        /* <= 8                                               */
    int32_t delay[8];
    float tap_re[8], tap_im[8];
    uint64_t seed;         /* Philox key                                         */
    uint64_t stream;       /* Philox counter high words (link id)                */
} orc_chan_cfg;
void orc_channel(const float *in, float *out, int64_t n, int64_t n0, const orc_chan_cfg *cfg);
/* time-varying fading taps, same layout and meaning as wifi_b200_fading (include/wifi_b200.h, 112 bytes) */
typedef struct orc_fading_cfg {
    int32_t n_taps;        /* 1..8                                               */
    int32_t n_sin;         /* sinusoids per tap, 1..16                           */
    int32_t delay[8];      /* samples, >= 0                                      */
    float power[8];        /* E|h_t|^2, >= 0                                     */
    float k_factor;        /* Rician K of tap 0, >= 0                            */
    float doppler;         /* cycles/sample, 0 .. 0.25                           */
    float los_doppler;     /* cycles/sample, -0.25 .. 0.25                       */
    int32_t reserved;
    int64_t t0;            /* time index of output sample 0                      */
    uint64_t seed, stream; /* Philox key and counter words of the realisation    */
} orc_fading_cfg;
/* orc_channel with the taps of fad (seg->n_taps must be 0); -1 for out-of-range parameters, else 0 */
int  orc_channel_fading(const float *in, float *out, int64_t n, int64_t n0, const orc_chan_cfg *seg, const orc_fading_cfg *fad);

/* ---- RX ---- */
void orc_frontend(const float *x, int64_t n, float *a_out, float *p_out, float *c_out);
void orc_flags(const float *x, int64_t n, double threshold, uint8_t *out);   /* sync_short's plateau test per sample */
typedef struct orc_rx_result orc_rx_result;
orc_rx_result *orc_rx(const float *x, int64_t n, int link, const orc_rx_cfg *cfg);
/* many links, one std::thread per worker; link l is x + 2*off[l], length len[l] */
orc_rx_result *orc_rx_links(const float *x, const int64_t *off, const int64_t *len, int n_links,
                            const orc_rx_cfg *cfg, int n_threads);
int64_t orc_rx_n_frames(const orc_rx_result *r);
int64_t orc_rx_n_rows(const orc_rx_result *r);
int64_t orc_rx_psdu_bytes(const orc_rx_result *r);
void orc_rx_copy(const orc_rx_result *r, orc_frame *frames, uint8_t *rows, float *carrier, uint8_t *psdu);
/* soft mode: one int8 per coded bit, 288 per row (first N_CBPS used), bit order c*N_BPSC+k */
void orc_rx_copy_soft(const orc_rx_result *r, int8_t *soft);
int  orc_viterbi_soft(const int8_t *depunctured, int n_avail, int n_bits, int ntraceback, uint8_t *out_bits);
void orc_rx_free(orc_rx_result *r);
/* element-wise evaluation of the numerical contract (include/wifi_detmath.h wdm_selftest) for tests/test_detmath.py */
void orc_detmath(int fn, const float *a, const float *b, const float *c, const float *d, float *o0, float *o1, int64_t n);

#ifdef __cplusplus
}
#endif
#endif
