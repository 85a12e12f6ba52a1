/*
 * fading_oracle.cpp -- CPU reference of the time-varying fading channel (TEST INFRASTRUCTURE ONLY).
 *
 * The scalar restatement of k_channel_fading that tests/test_fading_channel.py checks the kernel against, in the style of
 * the oracle's channel() (oracle/wifi_oracle.cpp): the same loop with the fixed taps replaced by h_t(t0 + i).  The draws
 * and the evaluation of h_t are the wdm_fading_* functions of include/wifi_detmath.h, which the kernel calls too, so the
 * two agree bit for bit when both follow the numerical contract's build rules (-ffp-contract=off -mfma here, -fmad=false
 * on the device).  Built by tests/fading_oracle.py.
 */
#include "../include/wifi_detmath.h"

#include <cmath>
#include <cstdint>

typedef wdm_cf cf;

/* same layout and meaning as wifi_b200_fading (include/wifi_b200.h) */
struct fad_cfg {
    int32_t n_taps, n_sin;
    int32_t delay[8];
    float power[8];
    float k_factor, doppler, los_doppler;
    int32_t reserved;
    int64_t t0;
    uint64_t seed, stream;
};

/* the segment's remaining fields, as the oracle's orc_chan_cfg without its taps */
struct fad_seg {
    float gain, cfo, phase0, noise_sigma;
    uint64_t seed, stream;
};

extern "C" int fad_channel(const float *in_f, float *out_f, int64_t n, int64_t n0, const fad_seg *seg, const fad_cfg *fad)
{
    const fad_seg &c = *seg;
    const fad_cfg &f = *fad;
    if (f.n_taps < 1 || f.n_taps > 8 || f.n_sin < 1 || f.n_sin > 16 || !(f.k_factor >= 0.f) ||
        !(f.doppler >= 0.f && f.doppler <= 0.25f) || !(std::fabs(f.los_doppler) <= 0.25f))
        return -1;
    for (int t = 0; t < f.n_taps; ++t)
        if (f.delay[t] < 0 || !(f.power[t] >= 0.f)) return -1;
    const cf *in = (const cf *)in_f;
    cf *out = (cf *)out_f;
    /* tap t's terms in ascending order; tap 0's line-of-sight term follows its n_sin sinusoids */
    wdm_fade_ent ent[8][17];
    const int cnt0 = f.n_sin + (f.k_factor > 0.f ? 1 : 0);
    for (int t = 0; t < f.n_taps; ++t)
        for (int m = 0; m < (t == 0 ? cnt0 : f.n_sin); ++m)
            ent[t][m] = wdm_fading_entry(f.seed, f.stream, t, m, f.n_sin, f.power[t], f.k_factor, f.doppler, f.los_doppler);
    const float ns = c.noise_sigma * 0.70710678f;
    for (int64_t i = 0; i < n; ++i) {
        const uint32_t nn = (uint32_t)(f.t0 + i);
        cf acc = {0.f, 0.f};
        for (int t = 0; t < f.n_taps; ++t) {
            int64_t j = i - f.delay[t];
            if (j < 0 || j >= n) continue;
            acc = wdm_cmac(acc, wdm_fading_tap(ent[t], t == 0 ? cnt0 : f.n_sin, nn), in[j]);
        }
        acc = cf{acc.re * c.gain, acc.im * c.gain};
        cf w;
        wdm_sincosf(c.cfo * (float)i + c.phase0, &w.im, &w.re);
        cf y = wdm_cmul(acc, w);
        if (c.noise_sigma > 0.f) {
            uint64_t idx = (uint64_t)(n0 + i);
            uint32_t r[4];
            wdm_philox4x32((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)c.stream, (uint32_t)(c.stream >> 32),
                           (uint32_t)c.seed, (uint32_t)(c.seed >> 32), r);
            float z0, z1;
            wdm_box_muller(r[0], r[1], &z0, &z1);
            y.re = y.re + ns * z0;
            y.im = y.im + ns * z1;
        }
        out[i] = y;
    }
    return 0;
}
