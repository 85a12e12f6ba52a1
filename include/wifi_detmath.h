/*
 * wifi_detmath.h -- the numerical contract of the 802.11a/g baseband.
 *
 * Why this exists.  The reference PHY (gr-ieee802-11 behind
 * gnu_radio/wifi_phy_hier.grc) calls libm/libstdc++ for arg(), exp(j*phi) and
 * log() (sync_short.cc: arg(in_abs[i])/16 and exp(gr_complex(0,-f*n));
 * sync_long.cc: arg(first*conj(second))/64; frame_equalizer_impl.cc: arg()/exp()
 * per symbol).  libm results differ in the last ulp between glibc versions and
 * differ again from CUDA's device libm, so "same decisions as the reference"
 * could only be a statistical statement.  To make parity a *bit-exact*
 * statement we fix the elementary functions here, as plain IEEE-754 binary32
 * operation sequences (+, -, *, /, fmaf, rintf, sqrtf -- all correctly rounded
 * on x86-64 SSE/FMA and on sm_100a), and both the CPU oracle (oracle/) and the
 * CUDA library (gnuradio-wifi-imagetransfer_b200/csrc/) evaluate exactly these
 * sequences.  Each function stays within a few ulp of glibc (checked in
 * tests/test_detmath.py), i.e. inside the spread the reference itself shows
 * between machines.
 *
 * Rules for users of this header:
 *   - compile host code with  -ffp-contract=off -mfma  (no implicit FMA, real
 *     fmaf instruction), device code with  -fmad=false  (no implicit FMA);
 *   - never build with -ffast-math / --use_fast_math.
 *
 * Polynomials are the classic single-precision Cephes minimax sets
 * (public domain, S. Moshier), evaluated in the fixed order written below.
 */
#ifndef WIFI_DETMATH_H
#define WIFI_DETMATH_H

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define WDM_FN __host__ __device__ __forceinline__
#else
#define WDM_FN static inline
#endif

/* ---- complex arithmetic: fixed sequences of IEEE-754 multiplies and fused multiply-adds ----
 * The reference multiplies complex numbers through VOLK / std::complex, whose rounding depends on the SIMD kernel the
 * machine dispatches to (SSE: separate multiplies and adds; AVX2+FMA builds: fused).  The contract fixes ONE sequence
 * per operation -- the fused one: it is the more accurate of the two (one rounding less per term) and costs 4
 * instructions per complex multiply on the GPU instead of 6.  Every complex product, multiply-accumulate and division
 * of the oracle and of the CUDA library goes through these functions. */
typedef struct wdm_cf { float re, im; } wdm_cf;

/* a * b */
WDM_FN wdm_cf wdm_cmul(wdm_cf a, wdm_cf b)
{
    wdm_cf r;
    r.re = fmaf(a.re, b.re, -(a.im * b.im));
    r.im = fmaf(a.re, b.im, a.im * b.re);
    return r;
}
/* a * conj(b) */
WDM_FN wdm_cf wdm_cmulc(wdm_cf a, wdm_cf b)
{
    wdm_cf r;
    r.re = fmaf(a.re, b.re, a.im * b.im);
    r.im = fmaf(a.im, b.re, -(a.re * b.im));
    return r;
}
/* acc + a * b */
WDM_FN wdm_cf wdm_cmac(wdm_cf acc, wdm_cf a, wdm_cf b)
{
    wdm_cf r;
    r.re = fmaf(-a.im, b.im, fmaf(a.re, b.re, acc.re));
    r.im = fmaf(a.im, b.re, fmaf(a.re, b.im, acc.im));
    return r;
}
/* acc + a * conj(b) */
WDM_FN wdm_cf wdm_cmacc(wdm_cf acc, wdm_cf a, wdm_cf b)
{
    wdm_cf r;
    r.re = fmaf(a.im, b.im, fmaf(a.re, b.re, acc.re));
    r.im = fmaf(-a.re, b.im, fmaf(a.im, b.re, acc.im));
    return r;
}
/* acc - a * conj(b) */
WDM_FN wdm_cf wdm_cmsubc(wdm_cf acc, wdm_cf a, wdm_cf b)
{
    wdm_cf r;
    r.re = fmaf(-a.im, b.im, fmaf(-a.re, b.re, acc.re));
    r.im = fmaf(a.re, b.im, fmaf(-a.im, b.re, acc.im));
    return r;
}
/* |a|^2 */
WDM_FN float wdm_norm(wdm_cf a) { return fmaf(a.re, a.re, a.im * a.im); }
/* acc + |a|^2, acc - |a|^2 */
WDM_FN float wdm_norm_add(float acc, wdm_cf a) { return fmaf(a.im, a.im, fmaf(a.re, a.re, acc)); }
WDM_FN float wdm_norm_sub(float acc, wdm_cf a) { return fmaf(-a.im, a.im, fmaf(-a.re, a.re, acc)); }
/* a / b = a * conj(b) * (1 / |b|^2): one IEEE division */
WDM_FN wdm_cf wdm_cdiv(wdm_cf a, wdm_cf b)
{
    const float inv = 1.0f / wdm_norm(b);
    wdm_cf n = wdm_cmulc(a, b), r;
    r.re = n.re * inv;
    r.im = n.im * inv;
    return r;
}

/* sin and cos of x (radians).  |x| up to ~1e5 keeps abs error < 2e-7;
 * the PHY's largest argument is pi/16 * 43200 ~ 8.5e3.                      */
WDM_FN void wdm_sincosf(float x, float *s, float *c)
{
    /* Cody-Waite reduction to r in [-pi/4, pi/4] with k = nearest multiple of pi/2 */
    float k = rintf(x * 0.636619772f);
    float r = fmaf(k, -1.57079601e+00f, x);
    r = fmaf(k, -3.13916473e-07f, r);
    r = fmaf(k, -5.39030253e-15f, r);
    float z = r * r;
    /* sin(r) */
    float ps = fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f);
    ps = fmaf(ps, z, -1.6666654611e-1f);
    float sr = fmaf(ps * z, r, r);
    /* cos(r) */
    float pc = fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f);
    pc = fmaf(pc, z, 4.166664568298827e-2f);
    float cr = fmaf(pc * z, z, fmaf(z, -0.5f, 1.0f));
    int q = (int)k & 3; /* two's-complement & 3 == k mod 4 also for negative k */
    float so = (q & 1) ? cr : sr;
    float co = (q & 1) ? sr : cr;
    if (q & 2) so = -so;
    if ((q + 1) & 2) co = -co;
    *s = so;
    *c = co;
}

/* sin and cos of 2*pi*p/2^32: a phase in turns held as an unsigned 32-bit integer (the accumulator of a numerically
 * controlled oscillator).  The quadrant comes from the top bits and the remainder is a signed offset in [-pi/4, pi/4),
 * so no Cody-Waite step is needed and the error is below 3e-7 absolute for every phase.  The polynomials and the
 * quadrant swap are wdm_sincosf's; they are written out again because sharing them through a helper reschedules the
 * receiver kernels that call wdm_sincosf. */
WDM_FN void wdm_sincos_turn(uint32_t p, float *s, float *c)
{
    const uint32_t q = (p + 0x20000000u) >> 30;                                  /* nearest quarter turn, 0..3 */
    const float r = (float)(int32_t)(p - (q << 30)) * 1.46291807926715968e-9f;   /* x 2 pi / 2^32 */
    float z = r * r;
    float ps = fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f);
    ps = fmaf(ps, z, -1.6666654611e-1f);
    float sr = fmaf(ps * z, r, r);
    float pc = fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f);
    pc = fmaf(pc, z, 4.166664568298827e-2f);
    float cr = fmaf(pc * z, z, fmaf(z, -0.5f, 1.0f));
    float so = (q & 1) ? cr : sr;
    float co = (q & 1) ? sr : cr;
    if (q & 2) so = -so;
    if ((q + 1) & 2) co = -co;
    *s = so;
    *c = co;
}

/* atan2(y, x) in (-pi, pi].  atan2(0,0) = 0.  NaN inputs give NaN.
 * One division and no branches: with mn = min(|x|,|y|), mx = max(|x|,|y|) the angle of (mx, mn) lies in [0, pi/4];
 * above tan(pi/8) it is pi/4 + atan((mn - mx)/(mn + mx)), so the argument of the polynomial is formed as a quotient of
 * sums BEFORE the division (the classic form divides twice: mn/mx, then (q - 1)/(q + 1)); |t| <= tan(pi/8). */
WDM_FN float wdm_atan2f(float y, float x)
{
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const int hi = mn > 0.4142135623730950f * mx;
    const float num = hi ? mn - mx : mn;
    const float den = hi ? mn + mx : mx;
    float t = num / den;
    if (mx == 0.0f) t = 0.0f;                               /* atan2(0, 0) = 0 */
    const float z = t * t;
    float p = fmaf(z, 8.05374449538e-2f, -1.38776856032e-1f);
    p = fmaf(p, z, 1.99777106478e-1f);
    p = fmaf(p, z, -3.33329491539e-1f);
    float r = fmaf(p * z, t, t);
    if (hi) r = 0.7853981633974483f + r;
    if (ay > ax) r = 1.5707963267948966f - r;
    if (x < 0.0f) r = 3.14159265358979f - r;
    if (y < 0.0f) r = -r;
    if (x != x || y != y) r = x + y;
    return r;
}

/* natural log for finite x > 0 (used by the synthetic channel's Box-Muller) */
WDM_FN float wdm_logf(float x)
{
    /* x = m * 2^e, m in [sqrt(1/2), sqrt(2)) ; normal numbers only */
    union { float f; uint32_t u; } v;
    v.f = x;
    int e = (int)((v.u >> 23) & 0xff) - 126;
    v.u = (v.u & 0x007fffffu) | 0x3f000000u;   /* m in [0.5, 1) */
    float m = v.f;
    if (m < 0.707106781186547524f) {
        e -= 1;
        m = m + m;
    }
    m = m - 1.0f;
    float z = m * m;
    float p = fmaf(m, 7.0376836292e-2f, -1.1514610310e-1f);
    p = fmaf(p, m, 1.1676998740e-1f);
    p = fmaf(p, m, -1.2420140846e-1f);
    p = fmaf(p, m, 1.4249322787e-1f);
    p = fmaf(p, m, -1.6668057665e-1f);
    p = fmaf(p, m, 2.0000714765e-1f);
    p = fmaf(p, m, -2.4999993993e-1f);
    p = fmaf(p, m, 3.3333331174e-1f);
    float y = (m * z) * p;
    float fe = (float)e;
    y = fmaf(fe, -2.12194440e-4f, y);
    y = fmaf(z, -0.5f, y);
    float r = m + y;
    r = fmaf(fe, 0.693359375f, r);
    return r;
}

/* ---- Philox4x32-10 counter RNG (Salmon et al., SC'11); integer-exact ---- */
WDM_FN void wdm_philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                           uint32_t k0, uint32_t k1, uint32_t out[4])
{
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* one complex standard-normal pair (each component N(0,1)) from two words */
WDM_FN void wdm_box_muller(uint32_t w0, uint32_t w1, float *z0, float *z1)
{
    float u1 = ((float)(w0 >> 8) + 0.5f) * 5.9604644775390625e-8f; /* (0,1) */
    float u2 = ((float)(w1 >> 8) + 0.5f) * 5.9604644775390625e-8f;
    float rad = sqrtf(-2.0f * wdm_logf(u1));
    float s, c;
    wdm_sincosf(6.283185307179586f * u2, &s, &c);
    *z0 = rad * c;
    *z1 = rad * s;
}

/* ---- time-varying multipath fading: a sum of sinusoids per tap (DESIGN.md "fading channel") ----
 * Tap t of a realisation is  h_t(n) = sum_{m < n_sin} w_{t,m} exp(j 2 pi f_{t,m} n)  (+ the line-of-sight term on tap 0)
 * with w ~ CN(0, P_t / n_sin) and f_{t,m} = doppler cos(2 pi (m + u_{t,m}) / n_sin), u ~ U[0,1): given the frequencies the
 * tap is complex Gaussian at every n, and over realisations its autocorrelation is Clarke's J0(2 pi doppler tau).  Phases
 * are 32-bit NCO phases fq * n (mod 2^32), exact for every n, so the process is periodic in 2^32 samples.
 * The draws come from Philox with key = seed and counter (16 t + m, 0xFFFFFFFF, stream): word 1 of an AWGN counter is the
 * high half of a non-negative sample index and never 0xFFFFFFFF, so the fading and the noise of one key are independent. */
typedef struct wdm_fade_ent { float re, im; uint32_t fq, pad; } wdm_fade_ent;   /* weight w and NCO increment of one term */

/* cycles/sample -> NCO phase increment per sample; |f| <= 0.25 keeps rintf(f 2^32) inside int32 */
WDM_FN uint32_t wdm_nco_freq(float f) { return (uint32_t)(int32_t)rintf(f * 4294967296.0f); }

/* Term m of tap t of the realisation (seed, stream).  m < n_sin: scatter sinusoid m, with power E|w|^2 = P / n_sin, or
 * on tap 0 P / (n_sin (k + 1)) (Rician K = k).  m == n_sin, tap 0, k > 0 only: the line-of-sight term
 * sqrt(P k / (k + 1)) exp(j (2 pi los_doppler n + phi)), phi from its own counter (128, 0xFFFFFFFF, stream). */
WDM_FN wdm_fade_ent wdm_fading_entry(uint64_t seed, uint64_t stream, int t, int m, int n_sin, float power, float k,
                                     float doppler, float los_doppler)
{
    wdm_fade_ent e;
    uint32_t r[4];
    float s, c;
    wdm_philox4x32(m < n_sin ? (uint32_t)(16 * t + m) : 128u, 0xFFFFFFFFu, (uint32_t)stream, (uint32_t)(stream >> 32),
                   (uint32_t)seed, (uint32_t)(seed >> 32), r);
    if (m < n_sin) {
        const float kk = t == 0 ? k : 0.0f;
        const float amp = sqrtf(power / ((float)n_sin * (kk + 1.0f))) * 0.70710678f;   /* per component of CN(0, 1) */
        float z0, z1;
        wdm_box_muller(r[0], r[1], &z0, &z1);
        e.re = amp * z0;
        e.im = amp * z1;
        /* angle (m + u) / n_sin turns with u = (r2 >> 8) / 2^24, as a 32-bit phase: an exact integer division */
        const uint32_t p = (uint32_t)((((uint64_t)m << 32) | (r[2] & 0xFFFFFF00u)) / (uint64_t)n_sin);
        wdm_sincos_turn(p, &s, &c);
        e.fq = wdm_nco_freq(doppler * c);
    } else {
        const float amp = sqrtf(power * k / (k + 1.0f));
        wdm_sincos_turn(r[0], &s, &c);
        e.re = amp * c;
        e.im = amp * s;
        e.fq = wdm_nco_freq(los_doppler);
    }
    e.pad = 0u;
    return e;
}

/* acc + w exp(j 2 pi fq n / 2^32): one term of a tap at sample n */
WDM_FN wdm_cf wdm_fading_step(wdm_cf acc, wdm_fade_ent e, uint32_t n)
{
    wdm_cf w, g;
    wdm_sincos_turn(e.fq * n, &w.im, &w.re);
    g.re = e.re;
    g.im = e.im;
    return wdm_cmac(acc, g, w);
}

/* h_t(n): the terms of one tap summed in ascending order */
WDM_FN wdm_cf wdm_fading_tap(const wdm_fade_ent *e, int cnt, uint32_t n)
{
    wdm_cf h;
    h.re = 0.0f;
    h.im = 0.0f;
    for (int k = 0; k < cnt; ++k) h = wdm_fading_step(h, e[k], n);
    return h;
}

/* ---- self-test dispatch: one element of tests/test_detmath.py (host: orc_detmath, device: wifi_b200_selftest_detmath).
 * o0/o1 are in-out (the accumulator of the multiply-accumulate forms). ---- */
enum { WDM_T_SINCOS = 0, WDM_T_ATAN2, WDM_T_LOG, WDM_T_CMUL, WDM_T_CMULC, WDM_T_CDIV, WDM_T_BOX_MULLER, WDM_T_CMAC,
       WDM_T_CMACC, WDM_T_CMSUBC, WDM_T_NORM_ADD, WDM_T_NORM_SUB, WDM_T_PHILOX, WDM_T_SINCOS_TURN, WDM_T_FADING_ENTRY,
       WDM_T_FADING_FREQ, WDM_T_FADING_STEP, WDM_T_COUNT };
WDM_FN void wdm_selftest(int fn, float a, float b, float c, float d, float *o0, float *o1)
{
    wdm_cf x, y, acc, r;
    x.re = a; x.im = b; y.re = c; y.im = d; acc.re = *o0; acc.im = *o1;
    union { float f; uint32_t u; } ua, ub, uc, ud;
    ua.f = a; ub.f = b; uc.f = c; ud.f = d;
    switch (fn) {
    case WDM_T_SINCOS: wdm_sincosf(a, o0, o1); break;
    case WDM_T_ATAN2: *o0 = wdm_atan2f(a, b); break;
    case WDM_T_LOG: *o0 = wdm_logf(a); break;
    case WDM_T_CMUL: r = wdm_cmul(x, y); *o0 = r.re; *o1 = r.im; break;
    case WDM_T_CMULC: r = wdm_cmulc(x, y); *o0 = r.re; *o1 = r.im; break;
    case WDM_T_CDIV: r = wdm_cdiv(x, y); *o0 = r.re; *o1 = r.im; break;
    case WDM_T_BOX_MULLER: wdm_box_muller(ua.u, ub.u, o0, o1); break;           /* a, b carry the two 32-bit words */
    case WDM_T_CMAC: r = wdm_cmac(acc, x, y); *o0 = r.re; *o1 = r.im; break;
    case WDM_T_CMACC: r = wdm_cmacc(acc, x, y); *o0 = r.re; *o1 = r.im; break;
    case WDM_T_CMSUBC: r = wdm_cmsubc(acc, x, y); *o0 = r.re; *o1 = r.im; break;
    case WDM_T_NORM_ADD: *o0 = wdm_norm_add(acc.re, x); break;
    case WDM_T_NORM_SUB: *o0 = wdm_norm_sub(acc.re, x); break;
    case WDM_T_PHILOX: {                                                        /* counter (a, b), key (c, d) as bit patterns */
        uint32_t w[4];
        wdm_philox4x32(ua.u, ub.u, 0u, 0u, uc.u, ud.u, w);
        ua.u = w[0] ^ w[2]; ub.u = w[1] ^ w[3];
        *o0 = ua.f; *o1 = ub.f;
        break;
    }
    case WDM_T_SINCOS_TURN: wdm_sincos_turn(ua.u, o0, o1); break;                /* a carries the phase */
    case WDM_T_FADING_ENTRY:     /* a, b: bits of seed, stream; c: doppler (-c: LoS doppler); d: bits t | m << 4 | (n_sin - 1) << 12;  */
    case WDM_T_FADING_FREQ: {    /* in: o0 = power, o1 = k.  ENTRY: o0, o1 = weight; FREQ: o0 = bits of fq, o1 = 0               */
        const wdm_fade_ent e = wdm_fading_entry(ua.u, ub.u, (int)(ud.u & 7u), (int)((ud.u >> 4) & 31u), (int)((ud.u >> 12) & 15u) + 1,
                                                *o0, *o1, c, -c);
        if (fn == WDM_T_FADING_ENTRY) {
            *o0 = e.re;
            *o1 = e.im;
        } else {
            ua.u = e.fq;
            *o0 = ua.f;
            *o1 = 0.0f;
        }
        break;
    }
    case WDM_T_FADING_STEP: {    /* a, b: weight; c, d: bits of fq and n; o0, o1: accumulator */
        wdm_fade_ent e;
        e.re = a; e.im = b; e.fq = uc.u; e.pad = 0u;
        r = wdm_fading_step(acc, e, ud.u);
        *o0 = r.re; *o1 = r.im;
        break;
    }
    default: break;
    }
}

#endif /* WIFI_DETMATH_H */
