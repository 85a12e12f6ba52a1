// wifi_common.cuh -- shared device types, constant tables and the fp32 helper
// ops of libwifi_b200.so.  Numerical contract: every float expression here and
// in the kernels is written in the same order as oracle/wifi_oracle.cpp and the
// translation unit is compiled with -fmad=false (the only fused multiply-adds are
// the explicit fmaf() of include/wifi_detmath.h), so results are bit-identical
// to the oracle.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/wifi_b200.h"
#include "../../include/wifi_detmath.h"

#define WIFI_MAX_SYM 511        // [UPSTREAM] utils.h MAX_SYM
#define WIFI_MAX_PSDU 1528      // [UPSTREAM] utils.h MAX_PSDU_SIZE
#define SS_MIN_GAP 480          // [UPSTREAM] sync_short.cc MIN_GAP
#define SS_MAX_SAMPLES 43200    // [UPSTREAM] sync_short.cc MAX_SAMPLES = 540*80
#define SYNC_LENGTH 320         // wifi_phy_hier.grc:698-715 sync_length
#define FE_CHUNK 64             // running-sum re-seed period of the front-end (DESIGN.md)
#define DET_THREADS 128         // k_detect: one thread per chunk, one block per tile
#define DET_TILE (DET_THREADS * FE_CHUNK)   // 8192 samples
#define PSDU_STRIDE 1536        // bytes reserved per decode job in the psdu store
#define VIT_MAXW 1560           // 32-bit words (8 trellis steps each) reserved per decode job
#define SOFT_MAXW 6240          // soft mode: one word = 2 trellis steps x 2 int8 soft symbols
#define SOFT_ROW 288            // soft values reserved per data symbol (N_CBPS <= 288)

// complex products, multiply-accumulates and divisions are the fused sequences of include/wifi_detmath.h
typedef wdm_cf cf;
__device__ __forceinline__ cf cadd(cf a, cf b) { return {a.re + b.re, a.im + b.im}; }
__device__ __forceinline__ cf csub(cf a, cf b) { return {a.re - b.re, a.im - b.im}; }
__device__ __forceinline__ cf cmul(cf a, cf b) { return wdm_cmul(a, b); }
__device__ __forceinline__ cf cdiv(cf a, cf b) { return wdm_cdiv(a, b); }
__device__ __forceinline__ cf cscale(cf a, float s) { return {a.re * s, a.im * s}; }
__device__ __forceinline__ cf crot(float phase)
{
    cf w;
    wdm_sincosf(phase, &w.im, &w.re);
    return w;
}
__device__ __forceinline__ cf cshfl(cf v, int lane) { return {__shfl_sync(0xffffffffu, v.re, lane), __shfl_sync(0xffffffffu, v.im, lane)}; }
__device__ __forceinline__ cf cshfl_xor(cf v, int m) { return {__shfl_xor_sync(0xffffffffu, v.re, m), __shfl_xor_sync(0xffffffffu, v.im, m)}; }

struct McsDesc { int n_bpsc, n_cbps, n_dbps, rate_field, punct; };

struct DevTables {
    float lts[64];            // LTS, shifted order (index = subcarrier + 32)
    float polarity[127];      // pilot polarity, wifi_phy_hier.grc:350-376
    cf long_taps[64];         // sync_long matched filter LONG[]
    cf tw[32];                // exp(-j 2 pi k/64)
    cf sts[64];               // sync word 1/2
    cf lts_rot[64];           // sync word 3
    float win;                // 1/sqrt(52)
    uint16_t P[8][288];       // interleaver: out[k] = in[P[k]]
    uint16_t Pinv[8][288];    // Pinv[P[k]] = k
    cf cons[8][64];           // constellations
    McsDesc mcs[8];
    uint32_t crc_tab[256];
    uint16_t scr_tab[128];    // descrambler, 8 steps: low byte = 8 feedback bits (LSB first), high byte = next state
    int8_t carrier_of[64];    // shifted bin -> data carrier 0..47, -1 for pilots/null
};
__constant__ DevTables c_tab;   // single translation unit (wifi_b200.cu)

// per-link descriptor (device)
struct LinkDesc {
    int64_t x_off;        // first sample of the link in the iq buffer
    int64_t len;          // samples
    int64_t chunk_base;   // first FE_CHUNK chunk of the link (links start on a DET_TILE tile: multiple of DET_THREADS)
    int32_t frame_first;  // first frame record of the link
    int32_t frame_count;
    float fo_carry;       // sync_long d_freq_offset entering this buffer
    int32_t is_final;
    int32_t hist;         // valid samples stored before x_off (streaming history); older samples read as 0
    int32_t hold_last;    // streaming: the newest burst is held back while a later trigger could still cut it short
    int64_t min_pos;      // first sample index sync_short may trigger on (previous trigger + MIN_GAP + 1)
    int64_t row_base;     // first equalizer row reserved for the link
};

// per-frame equalizer state handed from the SIGNAL phase to the data phase
struct EqState {
    cf H[64];
    cf prev_pil[4];
    double d_er;
    double eps0;
    double snr;
    float havg;           // mean |H|^2 over the 52 used carriers after the LTS estimate
    float pad0;
    float w0[64];         // soft-bit weight per carrier: |H|^2 / havg frozen at the LTS estimate
    uint8_t sig_bits[48];
};

// decode job, stored at the index of its owner (tag) frame; n_sym == 0: no job
struct JobDesc {
    int32_t frame;        // owner (tag) frame
    int32_t enc, len, n_sym;
    int32_t n_seg;        // bursts the symbols were collected from; the first 4 are listed below
    int32_t seg_row[4];   // first row of each segment
    int32_t seg_cnt[4];   // rows in each segment
    int32_t need_pack;    // trellis words not already written by k_demod (gathered rows, BPSK 3/4)
    int32_t last_frame;   // frame that delivered the last symbol (n_seg > 4: the segments are found by walking the frames)
    int32_t pad0;
};

// Row of data symbol s of a decode job.  Up to four bursts are listed in the job; a collection that spans more
// (decode_mac keeps collecting through any number of bursts whose tags it refuses) is located by walking the frame
// records from the tag frame: every burst in between that delivered rows contributed all of them, in order.
__device__ __forceinline__ int64_t job_row(const JobDesc &J, const wifi_b200_frame *__restrict__ frames, int s)
{
    if (J.n_seg <= 4) {
        int seg = 0, sbase = 0;
        while (seg < J.n_seg - 1 && s >= sbase + J.seg_cnt[seg]) { sbase += J.seg_cnt[seg]; ++seg; }
        return (int64_t)J.seg_row[seg] + (s - sbase);
    }
    int left = s;
    for (int g = J.frame; g < J.last_frame; ++g) {
        const int nr = frames[g].n_rows;
        if (nr <= 0) continue;
        if (left < nr) return frames[g].row_off + left;
        left -= nr;
    }
    return frames[J.last_frame].row_off + left;
}

// One axis of a decision and of the decided constellation point.  The comparisons are those of upstream's
// decision_maker (the oracle's decide()), the point is the table value (float)(+-magnitude) * level picked by
// selects instead of rebuilt from the bits.
template <int H>   // bits per axis: 1, 2, 3
__device__ __forceinline__ void dev_axis(float v, int &bits, float &pt)
{
    const int sgn = v > 0;
    if (H == 1) {
        const float level = sqrtf(0.5f);
        bits = sgn;
        pt = sgn ? level : -level;                 // (float)(+-1) * level
    } else if (H == 2) {
        const float level = sqrtf(0.1f);
        const int inner = fabsf(v) < (2 * level);
        bits = sgn | (inner << 1);
        const float m = inner ? 1.0f * level : 3.0f * level;
        pt = sgn ? m : -m;
    } else {
        const float level = sqrtf(1.0f / 42.0f);
        const float ar = fabsf(v);
        const int b1 = ar < (4 * level);
        const int b2 = (ar < (6 * level)) && (ar > (2 * level));
        bits = sgn | (b1 << 1) | (b2 << 2);
        // Gray: (b1, b2) = 00 -> 7, 01 -> 5, 11 -> 3, 10 -> 1
        const float m = b1 ? (b2 ? 3.0f * level : 1.0f * level) : (b2 ? 5.0f * level : 7.0f * level);
        pt = sgn ? m : -m;
    }
}
// decision + decided point of one carrier, dispatched on the (warp-uniform) modulation
__device__ __forceinline__ void dev_decide_point(int nb, cf s, int &bits, cf &pt)
{
    int bi, bq;
    if (nb == 6) {
        dev_axis<3>(s.re, bi, pt.re); dev_axis<3>(s.im, bq, pt.im);
        bits = bi | (bq << 3);
    } else if (nb == 4) {
        dev_axis<2>(s.re, bi, pt.re); dev_axis<2>(s.im, bq, pt.im);
        bits = bi | (bq << 2);
    } else if (nb == 2) {
        dev_axis<1>(s.re, bi, pt.re); dev_axis<1>(s.im, bq, pt.im);
        bits = bi | (bq << 1);
    } else {
        bits = s.re > 0;
        pt = cf{bits ? 1.f : -1.f, 0.f};
    }
}

__device__ __forceinline__ int dev_bitrev5(int v) { return (int)(__brev((unsigned)v) >> 27); }

// Per-lane twiddles of the warp FFT, fetched once per kernel (the table index depends on the
// lane, so reading c_tab inside the symbol loop would serialise in the constant cache).
struct WarpTw { cf w[6]; };
__device__ __forceinline__ WarpTw warp_tw(int lane, bool inverse)
{
    WarpTw t;
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        const int half = 1 << s;
        t.w[s] = c_tab.tw[(lane & (half - 1)) * (32 >> s)];
    }
    t.w[5] = c_tab.tw[lane];
    if (inverse) {
#pragma unroll
        for (int s = 0; s < 6; ++s) t.w[s].im = -t.w[s].im;
    }
    return t;
}

// Input index of a in warp_fft64 on lane l: 2*bitrev5(r) with r = l rotated left by one bit (5 bits);
// b is the input right after it.
__device__ __forceinline__ int warp_fft_in(int lane)
{
    return 2 * dev_bitrev5(((lane << 1) | (lane >> 4)) & 31);
}

// Lanes l and l^m trade one value: afterwards the lane with (l & m) == 0 holds its lo and the partner's lo,
// the other one the partner's hi and its own hi.  This turns span-2^k butterfly pairs into span-2^k' pairs.
__device__ __forceinline__ void warp_fft_trade(cf &lo, cf &hi, int lane, int m)
{
    const bool up = (lane & m) != 0;
    const cf r = cshfl_xor(up ? lo : hi, m);
    lo = up ? r : lo;
    hi = up ? hi : r;
}

// 64-point FFT across one warp, one butterfly per lane and stage.  On entry lane l holds in[warp_fft_in(l)] (a)
// and the input after it (b): DIT positions r and r+32 after bit reversal, r = l rotated left by one bit.
// Before the stage of span 2^s (s < 5) the lane holds a span-2^s pair; one trade with lane l^m re-pairs the
// values for the next stage.  The trade masks 16, 1, 2, 4, 8, 16 rotate the lane-to-position map back by one bit,
// so that on exit a = X[l], b = X[l+32], and at every stage s the pair's twiddle is tw.w[s] of warp_tw.
// Each butterfly is t = w*hi, lo + t, lo - t: the operations, operands and rounding of oracle fft64().
__device__ __forceinline__ void warp_fft64(cf &a, cf &b, int lane, const WarpTw &tw)
{
    warp_fft_trade(a, b, lane, 16);
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        const cf t = cmul(tw.w[s], b);
        const cf u = a;
        a = cadd(u, t);
        b = csub(u, t);
        warp_fft_trade(a, b, lane, 1 << s);
    }
    const cf t = cmul(tw.w[5], b);
    const cf u = a;
    a = cadd(u, t);
    b = csub(u, t);
}

// max-log LLR of one axis bit, weighted and quantised exactly as oracle soft_q(): clamp(rint((l*w)*16), +-32)
__device__ __forceinline__ int dev_soft_q(float l, float w)
{
    float v = rintf((l * w) * 16.0f);
    if (v > 32.f) v = 32.f;
    if (v < -32.f) v = -32.f;
    if (!(v == v)) v = 0.f;   /* NaN input: no information (float -> int of NaN is not portable) */
    return (int)v;
}
// soft values of one carrier (oracle soft_demap).  q[u][t]: axis u (0 = I, 1 = Q), t = 0 sign bit,
// 1 inner-half bit, 2 ring bit; coded bit k = u * (nb/2) + t.  BPSK: q[0][0] only.
struct SoftQ { int q[2][3]; };
__device__ __forceinline__ SoftQ dev_soft_demap(int nb, cf s, float w)
{
    SoftQ r;
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int t = 0; t < 3; ++t) r.q[u][t] = 0;
    if (nb == 1) { r.q[0][0] = dev_soft_q(s.re, w); return r; }
    const int h = nb >> 1;
    const float level = (h == 1) ? sqrtf(0.5f) : (h == 2) ? sqrtf(0.1f) : sqrtf(1.0f / 42.0f);
    const float ax[2] = {s.re / level, s.im / level};
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const float a = ax[u], m = fabsf(a);
        r.q[u][0] = dev_soft_q(a, w);
        if (h == 2) r.q[u][1] = dev_soft_q(2.0f - m, w);
        if (h == 3) {
            r.q[u][1] = dev_soft_q(4.0f - m, w);
            r.q[u][2] = dev_soft_q(2.0f - fabsf(m - 4.0f), w);
        }
    }
    return r;
}
