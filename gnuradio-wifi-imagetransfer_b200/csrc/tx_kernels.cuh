// tx_kernels.cuh -- transmit chain of wifi_phy_hier and the synthetic test channel.
// Reference stages (gnu_radio/wifi_phy_hier.grc, SURVEY.md 8a T1-T6):
//   T1 ieee802_11_mapper (:570-586)   T2 packet_headergenerator + signal_field (:35-46,425-441)
//   T3 chunks_to_symbols x2 (:316-335,518-532)   T4 tagged_stream_mux + ofdm_carrier_allocator (:279-405)
//   T5 fft_vxx_0_0 inverse, shift, window 1/sqrt(52) (:459-479)   T6 ofdm_cyclic_prefixer cp 16 rolloff 2 (:406-424)
// One block per PSDU: scrambled bits are staged in shared memory, every coded bit is then a
// 5-tap XOR of them (the K=7 encoder is an FIR over GF(2)), so all OFDM symbols of the frame
// are produced independently, one warp per symbol, IFFT in registers + warp shuffles.
#pragma once
#include "wifi_common.cuh"

#define TX_MAX_BITS 12480

struct TxFrameDesc {
    uint32_t psdu_off, len;
    uint32_t enc, seed;
    uint64_t burst_off;   // first output sample
    uint64_t sym_off;     // first byte in the tx symbol store
};

__device__ __forceinline__ int tx_scr(const uint8_t *scr, int i) { return i >= 0 ? scr[i] : 0; }

__global__ void __launch_bounds__(128) k_tx(const uint8_t *__restrict__ psdu_blob, const TxFrameDesc *__restrict__ descs, int n_frames,
                                             cf *__restrict__ out, uint8_t *__restrict__ sym_out)
{
    __shared__ uint8_t scr[TX_MAX_BITS];
    __shared__ uint8_t seq[127];
    __shared__ uint8_t sig[48];
    const int f = blockIdx.x;
    if (f >= n_frames) return;
    const TxFrameDesc D = descs[f];
    const int enc = D.enc, L = D.len;
    const McsDesc m = c_tab.mcs[enc];
    const int n_sym = (16 + 8 * L + 6 + m.n_dbps - 1) / m.n_dbps;
    const int n_data = n_sym * m.n_dbps;
    const uint8_t *psdu = psdu_blob + D.psdu_off;
    const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
    if (tid == 0) {
        int state = D.seed;
        for (int i = 0; i < 127; ++i) {
            int fb = ((state >> 6) & 1) ^ ((state >> 3) & 1);
            seq[i] = (uint8_t)fb;
            state = ((state << 1) & 0x7e) | fb;
        }
    }
    if (tid == 32) {
        // SIGNAL: 24 header bits -> conv encode -> BPSK interleave
        uint8_t hdr[24], coded[48];
        int rf = m.rate_field;
        hdr[0] = (rf >> 3) & 1; hdr[1] = (rf >> 2) & 1; hdr[2] = (rf >> 1) & 1; hdr[3] = rf & 1; hdr[4] = 0;
        int sum = hdr[0] + hdr[1] + hdr[2] + hdr[3];
        for (int i = 0; i < 12; ++i) { hdr[5 + i] = (L >> i) & 1; sum += hdr[5 + i]; }
        hdr[17] = sum & 1;
        for (int i = 18; i < 24; ++i) hdr[i] = 0;
        int st = 0;
        for (int i = 0; i < 24; ++i) {
            st = ((st << 1) & 0x7e) | hdr[i];
            coded[2 * i] = __popc(st & 0155) & 1;
            coded[2 * i + 1] = __popc(st & 0117) & 1;
        }
        for (int k = 0; k < 48; ++k) sig[k] = coded[c_tab.P[0][k]];
    }
    __syncthreads();
    for (int i = tid; i < n_data; i += blockDim.x) {
        int d = 0;
        if (i >= 16 && i < 16 + 8 * L) d = (psdu[(i - 16) >> 3] >> ((i - 16) & 7)) & 1;
        int v = d ^ seq[i % 127];
        if (i >= 16 + 8 * L && i < 16 + 8 * L + 6) v = 0;   // reset_tail_bits
        scr[i] = (uint8_t)v;
    }
    __syncthreads();
    const int total_syms = 5 + n_sym;
    cf *o = out + D.burst_off;
    const int q0 = warp_fft_in(lane);
    const WarpTw tw = warp_tw(lane, true);
    for (int s = wib; s < total_syms; s += 4) {
        cf v[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            int i = (q0 + u + 32) & 63;   // shifted bin feeding natural IFFT input q0+u
            cf X;
            if (s < 2) X = c_tab.sts[i];
            else if (s == 2) X = c_tab.lts_rot[i];
            else if (s == 3) X = cf{c_tab.lts[i], 0.f};
            else {
                int n = s - 4;
                float p = c_tab.polarity[n % 127];
                int c = c_tab.carrier_of[i];
                if (i == 11 || i == 25 || i == 39) X = cf{p, 0.f};
                else if (i == 53) X = cf{-p, 0.f};
                else if (c < 0) X = cf{0.f, 0.f};
                else if (n == 0) X = cf{sig[c] ? 1.f : -1.f, 0.f};
                else {
                    int ds = n - 1, val = 0;
                    for (int k = 0; k < m.n_bpsc; ++k) {
                        int q = ds * m.n_cbps + c_tab.P[enc][c * m.n_bpsc + k];
                        int mi = m.punct == 0 ? q : (m.punct == 1 ? (q / 3) * 4 + q % 3 : (q / 4) * 6 + ((q & 3) == 3 ? 5 : (q & 3)));
                        int bi = mi >> 1;
                        int bit = (mi & 1) ? (tx_scr(scr, bi) ^ tx_scr(scr, bi - 1) ^ tx_scr(scr, bi - 2) ^ tx_scr(scr, bi - 3) ^ tx_scr(scr, bi - 6))
                                           : (tx_scr(scr, bi) ^ tx_scr(scr, bi - 2) ^ tx_scr(scr, bi - 3) ^ tx_scr(scr, bi - 5) ^ tx_scr(scr, bi - 6));
                        val |= bit << k;
                    }
                    X = c_tab.cons[enc][val];
                    if (sym_out) sym_out[D.sym_off + (uint64_t)ds * 48 + c] = (uint8_t)val;
                }
            }
            v[u] = cscale(X, c_tab.win);
        }
        cf a = v[0], b = v[1];
        warp_fft64(a, b, lane, tw);
        cf *os = o + (int64_t)s * 80;
        os[16 + lane] = a;
        os[48 + lane] = b;
        if (lane >= 16) os[lane - 16] = b;
    }
    __syncthreads();
    for (int s = tid; s <= total_syms; s += blockDim.x) {
        if (s == total_syms) {
            o[(int64_t)s * 80] = cscale(o[(int64_t)(s - 1) * 80 + 16], 0.5f);
        } else {
            cf d = s > 0 ? cscale(o[(int64_t)(s - 1) * 80 + 16], 0.5f) : cf{0.f, 0.f};
            o[(int64_t)s * 80] = cadd(cscale(o[(int64_t)s * 80], 0.5f), d);
        }
    }
}

// synthetic channel, mirrors the oracle's channel(): y(i) = gain * sum_t tap(t, t0 + i) * x(i - delay[t]), then the CFO
// rotation and Philox AWGN at counter n0 + i.  One grid row per segment.  tap(t, n) is tap t's coefficient at time n
// (a 32-bit NCO time, computed once per sample here; the fixed taps ignore it).
template <class Tap>
__device__ __forceinline__ void channel_body(const cf *__restrict__ in, cf *__restrict__ out, const wifi_b200_chan_seg &S, int n_taps,
                                             const int32_t *delay, int64_t t0, Tap tap)
{
    const float ns = S.noise_sigma * 0.70710678f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < S.n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t n = (uint32_t)(t0 + i);
        cf acc = {0.f, 0.f};
        for (int t = 0; t < n_taps; ++t) {
            int64_t j = i - delay[t];
            if (j < 0 || j >= S.in_len) continue;
            acc = wdm_cmac(acc, tap(t, n), in[S.in_off + j]);
        }
        acc = cscale(acc, S.gain);
        cf w = crot(S.cfo * (float)i + S.phase0);
        cf y = cmul(acc, w);
        if (S.noise_sigma > 0.f) {
            uint64_t idx = (uint64_t)(S.n0 + i);
            uint32_t r[4];
            wdm_philox4x32((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)S.stream, (uint32_t)(S.stream >> 32),
                           (uint32_t)S.seed, (uint32_t)(S.seed >> 32), r);
            float z0, z1;
            wdm_box_muller(r[0], r[1], &z0, &z1);
            y.re = y.re + ns * z0;
            y.im = y.im + ns * z1;
        }
        out[S.out_off + i] = y;
    }
}

// fixed taps (wifi_b200_channel_dev)
__global__ void __launch_bounds__(256) k_channel(const cf *__restrict__ in, cf *__restrict__ out, const wifi_b200_chan_seg *__restrict__ segs, int n_segs)
{
    const int sidx = blockIdx.y;
    if (sidx >= n_segs) return;
    const wifi_b200_chan_seg S = segs[sidx];
    channel_body(in, out, S, S.n_taps, S.delay, 0, [&](int t, uint32_t) { return cf{S.tap_re[t], S.tap_im[t]}; });
}

// time-varying fading channel (wifi_b200_channel_fading_dev): the taps are h_t(t0 + i) of include/wifi_detmath.h.  The
// block first draws its segment's terms into shared memory (tap t at slots t * FADE_SLOTS ..; tap 0's line-of-sight term
// follows its n_sin sinusoids), then every sample evaluates one NCO sincos and one complex multiply-accumulate per term.
#define FADE_SLOTS 17
__global__ void __launch_bounds__(256) k_channel_fading(const cf *__restrict__ in, cf *__restrict__ out, const wifi_b200_chan_seg *__restrict__ segs,
                                                        const wifi_b200_fading *__restrict__ fades, int n_segs)
{
    __shared__ wdm_fade_ent ent[8 * FADE_SLOTS];
    const int sidx = blockIdx.y;
    if (sidx >= n_segs) return;
    const wifi_b200_chan_seg S = segs[sidx];
    const wifi_b200_fading F = fades[sidx];
    const int cnt0 = F.n_sin + (F.k_factor > 0.f ? 1 : 0);
    for (int k = threadIdx.x; k < F.n_taps * FADE_SLOTS; k += blockDim.x) {
        const int t = k / FADE_SLOTS, m = k - t * FADE_SLOTS;
        if (m < (t == 0 ? cnt0 : F.n_sin))
            ent[k] = wdm_fading_entry(F.seed, F.stream, t, m, F.n_sin, F.power[t], F.k_factor, F.doppler, F.los_doppler);
    }
    __syncthreads();
    channel_body(in, out, S, F.n_taps, F.delay, F.t0,
                 [&](int t, uint32_t n) { return wdm_fading_tap(ent + t * FADE_SLOTS, t == 0 ? cnt0 : F.n_sin, n); });
}
