"""Time-varying Rayleigh/Rician multipath fading (wifi_b200_channel_fading[_dev]) and its CPU reference
(tests/fading_oracle.cpp, the oracle's channel() loop with the fading taps).

The CPU half checks the model through that reference and the oracle's contract self-test: the NCO sincos of include/wifi_detmath.h, the Rayleigh / Rician
marginals, Clarke's autocorrelation, the power-delay profile and the determinism a user builds on (same realisation for the
same (seed, stream, t0), a segment split in time equals the unsplit one).  Statistics average over realisations (streams),
not over time: a realisation with a finite number of sinusoids is not ergodic.  The GPU half asks for bit equality with
the oracle, for the static channel's arithmetic at zero Doppler, and for decode parity of all four equalizers on a
capture that fades inside its frames."""
import numpy as np
import pytest

import fading_oracle as F
from util import assert_frames_equal

SINCOS_TURN, FADING_ENTRY, FADING_FREQ, FADING_STEP = 13, 14, 15, 16


def _h(n, **fad):
    """The realisation itself: all-ones input, one tap at delay 0, gain 1, no noise -> the output is h_0(t0 + i)."""
    return F.channel(np.ones(n, np.complex64), fading=dict(taps=fad.pop("taps", ((0, 1.0),)), **fad))


# ---------------------------------------------------------------------------------------------------------- CPU (oracle)
def test_turn_sincos_accuracy(O):
    edges = [(k * 2 ** 30 + d) % 2 ** 32 for k in range(4) for d in (-2, -1, 0, 1, 2)]
    edges += [((2 * k + 1) * 2 ** 29 + d) % 2 ** 32 for k in range(4) for d in (-2, -1, 0, 1, 2)]   # where the quadrant changes
    p = np.concatenate([np.array(edges, np.uint32), np.random.default_rng(0).integers(0, 2 ** 32, 10 ** 6, dtype=np.uint32)])
    s, c = O.detmath(SINCOS_TURN, p.view(np.float32))
    ang = 2 * np.pi * p.astype(np.float64) / 2 ** 32
    assert np.abs(s - np.sin(ang)).max() <= 3e-7 and np.abs(c - np.cos(ang)).max() <= 3e-7
    z = int(np.nonzero(p == 0)[0][0])
    assert s[z] == 0.0 and c[z] == 1.0                       # zero phase is exactly (0, 1): a static tap stays exact


def test_block_rayleigh():
    from scipy import stats
    h = _h(64, taps=((0, 2.0),), seed=5, stream=0)
    assert np.all(h == h[0])                                   # doppler 0: one value per segment, exactly
    h = np.array([_h(1, taps=((0, 2.0),), seed=5, stream=s)[0] for s in range(4000)])
    e = np.abs(h.astype(np.complex128)) ** 2
    assert abs(e.mean() - 2.0) < 5 * 2.0 / np.sqrt(e.size)
    assert stats.kstest(e, "expon", args=(0, 2.0)).pvalue > 1e-3


def test_rician_k_by_moments():
    h = np.array([_h(1, k_factor=4.0, doppler=1e-3, los_doppler=2e-4, seed=9, stream=s)[0] for s in range(4000)])
    e = np.abs(h.astype(np.complex128)) ** 2
    q = np.sqrt(2 - np.mean(e ** 2) / np.mean(e) ** 2)        # m4 / m2^2 = 2 - (K / (K + 1))^2
    assert abs(q / (1 - q) - 4.0) < 0.2 * 4.0
    assert abs(e.mean() - 1.0) < 0.05


def test_strong_line_of_sight_without_doppler_keeps_its_phase():
    h = _h(20000, k_factor=1e5, doppler=1e-3, los_doppler=0.0, seed=1, stream=7)
    d = np.angle(h * np.conj(h[0]))
    assert np.abs(d).max() < 0.05
    g = _h(20000, k_factor=1e5, doppler=1e-3, los_doppler=1e-4, seed=1, stream=7)
    assert np.abs(np.angle(g * np.conj(g[0]))).max() > 1.0      # a LoS Doppler does turn it


def test_clarke_autocorrelation():
    from scipy import special
    fd = 0.01
    lags = np.rint(np.array([0.5, 1.0, 2.405, 3.8]) / (2 * np.pi * fd)).astype(int)
    H = np.array([_h(200, doppler=fd, seed=2, stream=s) for s in range(4000)]).astype(np.complex128)
    for L in lags:
        r = np.mean(H[:, :200 - L] * np.conj(H[:, L:]))
        assert abs(r.real - special.j0(2 * np.pi * fd * L)) < 0.08 and abs(r.imag) < 0.08, (L, r)


def test_no_frequency_beyond_the_doppler(O):
    rng = np.random.default_rng(4)
    n = 200_000
    for fd in (1e-4, 5e-4, 0.25):
        seed, stream = rng.integers(0, 2 ** 32, n, dtype=np.uint32), rng.integers(0, 2 ** 32, n, dtype=np.uint32)
        t, m, M = rng.integers(0, 8, n), rng.integers(0, 16, n), rng.integers(1, 17, n)
        m = np.minimum(m, M - 1)
        d = (t | (m << 4) | ((M - 1) << 12)).astype(np.uint32)
        fq, _ = O.detmath(FADING_FREQ, seed.view(np.float32), stream.view(np.float32), np.full(n, fd, np.float32),
                          d.view(np.float32), np.ones(n, np.float32), np.zeros(n, np.float32))
        f = fq.view(np.int32).astype(np.int64)
        assert np.abs(f).max() <= np.rint(np.float32(fd) * np.float32(2 ** 32)), fd
        assert f.max() > 0.9 * fd * 2 ** 32 and f.min() < -0.9 * fd * 2 ** 32


def test_taps_follow_the_power_delay_profile_and_are_uncorrelated():
    pdp = ((0, 0.6), (2, 0.3), (5, 0.1))
    x = np.zeros(8, np.complex64)
    x[0] = 1
    H = np.array([F.channel(x, fading=dict(taps=pdp, n_sin=4, seed=3, stream=s))[[0, 2, 5]] for s in range(4000)]).astype(np.complex128)
    N = H.shape[0]
    for k, (_, p) in enumerate(pdp):
        assert abs(np.mean(np.abs(H[:, k]) ** 2) - p) < 5 * p / np.sqrt(N), k
    for a in range(3):
        for b in range(a + 1, 3):
            assert abs(np.mean(H[:, a] * np.conj(H[:, b]))) / np.sqrt(pdp[a][1] * pdp[b][1]) < 5 / np.sqrt(N), (a, b)


def test_determinism_streams_and_split_segments():
    rng = np.random.default_rng(8)
    x = (rng.standard_normal(3000) + 1j * rng.standard_normal(3000)).astype(np.complex64)
    fad = dict(taps=((0, 1.0),), k_factor=2.0, doppler=1e-3, los_doppler=-3e-4, seed=11, stream=4)
    kw = dict(gain=0.8, noise_sigma=0.05, seed=99, stream=2)
    a = F.channel(x, fading=fad, **kw)
    assert np.array_equal(a, F.channel(x, fading=fad, **kw))
    assert not np.array_equal(a, F.channel(x, fading=dict(fad, stream=5), **kw))
    N = 1234
    first = F.channel(x[:N], fading=fad, **kw)
    second = F.channel(x[N:], n0=N, fading=dict(fad, t0=N), **kw)
    assert np.array_equal(np.concatenate([first, second]), a)


def test_out_of_range_parameters_are_refused_by_the_oracle():
    x = np.ones(4, np.complex64)
    for bad in (dict(taps=()), dict(n_sin=0), dict(n_sin=17), dict(k_factor=-1.0), dict(doppler=0.3), dict(doppler=-1e-3),
                dict(los_doppler=0.26), dict(taps=((-1, 1.0),)), dict(taps=((0, -1.0),))):
        with pytest.raises(ValueError):
            F.channel(x, fading=dict(dict(taps=((0, 1.0),)), **bad))


# ------------------------------------------------------------------------------------------------------------------- GPU
def _seg_pair(W, n, seg, fad):
    """A segment of n samples with no static taps (keywords of chan_seg in `seg`) and its fading record (keywords of fading)."""
    w = W.wifi_b200
    return w.chan_seg(in_len=n, n=n, taps=(), **seg), w.fading(**fad)


def _oracle_seg(x, s, f):
    return F.channel(x, f, n0=int(s["n0"][0]), gain=float(s["gain"][0]), cfo=float(s["cfo"][0]), phase0=float(s["phase0"][0]),
                     noise_sigma=float(s["noise_sigma"][0]), seed=int(s["seed"][0]), stream=int(s["stream"][0]))


CASES = {
    "flat_rayleigh_block": dict(taps=((0, 1.0),)),
    "three_taps_rician_doppler": dict(taps=((0, 0.6), (1, 0.3), (3, 0.1)), k_factor=4.0, doppler=1e-3, los_doppler=3e-4, seed=7, stream=3),
    "eight_taps_sixteen_sinusoids": dict(taps=tuple((2 * t, 1.0 / (t + 1)) for t in range(8)), n_sin=16, doppler=5e-4, seed=12),
    "nco_wraps_inside": dict(taps=((0, 1.0), (4, 0.5)), doppler=2e-3, k_factor=1.0, los_doppler=-1e-3, t0=2 ** 32 - 100, stream=9),
    "cfo_gain_noise_n0_stream": dict(taps=((0, 0.7), (2, 0.3)), doppler=1e-3, seed=2 ** 40 + 5, stream=2 ** 35 + 1,
                                     seg=dict(gain=0.7, cfo=0.013, phase0=0.5, noise_sigma=0.2, n0=1234, seed=77, stream=3)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_kernel_equals_oracle(W, case):
    import torch
    kw = dict(CASES[case])
    segkw = kw.pop("seg", {})
    x = (np.random.default_rng(41).standard_normal(5000) + 1j * np.random.default_rng(42).standard_normal(5000)).astype(np.complex64)
    s, f = _seg_pair(W, x.size, segkw, kw)
    h = W.Handle(max_samples=1 << 16)
    try:
        tx = torch.from_numpy(x.view(np.float32)).cuda()
        ty = torch.zeros_like(tx)
        h.channel_fading_dev(tx.data_ptr(), ty.data_ptr(), s, f)
        got = ty.cpu().numpy().view(np.complex64)
        assert np.array_equal(got, _oracle_seg(x, s, f))
        assert np.array_equal(h.channel(x, fading=f, **segkw), got)    # host-buffer twin
    finally:
        h.close()


@pytest.mark.gpu
def test_many_segments_over_several_launches(W):
    """70000 segments: more than one launch of 65535 grid rows, every one its own stream, t0 and n0."""
    import torch
    w = W.wifi_b200
    n_seg, L = 70000, 48
    rng = np.random.default_rng(5)
    x = (rng.standard_normal(n_seg * L) + 1j * rng.standard_normal(n_seg * L)).astype(np.complex64)
    segs = np.zeros(n_seg, w.CHANSEG_DTYPE)
    fades = np.zeros(n_seg, w.FADING_DTYPE)
    segs["in_off"] = segs["out_off"] = np.arange(n_seg) * L
    segs["in_len"] = segs["n"] = L
    segs["n0"] = segs["in_off"] + 17
    segs["gain"], segs["noise_sigma"], segs["seed"] = 0.9, 0.1, 4
    segs["cfo"] = rng.uniform(-0.01, 0.01, n_seg)
    fades["n_taps"], fades["n_sin"] = 2, 8
    fades["delay"][:, 1] = 1
    fades["power"][:, 0], fades["power"][:, 1] = 0.8, 0.2
    fades["doppler"], fades["k_factor"] = 5e-4, np.where(np.arange(n_seg) % 3 == 0, 2.0, 0.0)
    fades["t0"] = rng.integers(0, 2 ** 33, n_seg)
    fades["seed"], fades["stream"] = 21, np.arange(n_seg)
    h = W.Handle(max_samples=1 << 16)
    try:
        tx = torch.from_numpy(x.view(np.float32)).cuda()
        ty = torch.zeros_like(tx)
        h.channel_fading_dev(tx.data_ptr(), ty.data_ptr(), segs, fades)
        got = ty.cpu().numpy().view(np.complex64).reshape(n_seg, L)
    finally:
        h.close()
    for i in list(range(0, 600)) + list(range(65400, 65700)) + list(range(n_seg - 300, n_seg)):
        want = _oracle_seg(x[i * L:(i + 1) * L], segs[i:i + 1], fades[i:i + 1])
        assert np.array_equal(got[i], want), i
    assert len({got[i, 0] for i in range(0, n_seg, 97)}) > 700      # distinct streams, distinct realisations


@pytest.mark.gpu
def test_zero_doppler_runs_the_static_channels_arithmetic(W):
    """At doppler 0 every tap is one constant: read it off an impulse, hand it to k_channel, get the same bits."""
    taps = ((0, 0.6), (1, 0.25), (3, 0.15))
    fad = dict(taps=taps, n_sin=8, k_factor=3.0, seed=31, stream=8)
    h = W.Handle(max_samples=1 << 16)
    try:
        imp = np.zeros(16, np.complex64)
        imp[0] = 1
        r = h.channel(imp, fading=fad)
        drawn = [(d, complex(r[d])) for d, _ in taps]
        assert all(abs(v) > 0 for _, v in drawn)
        x = (np.random.default_rng(3).standard_normal(4000) + 1j * np.random.default_rng(4).standard_normal(4000)).astype(np.complex64)
        kw = dict(gain=0.8, cfo=0.02, phase0=0.1, noise_sigma=0.05, n0=77, seed=5, stream=6)
        assert np.array_equal(h.channel(x, fading=fad, **kw), h.channel(x, taps=drawn, **kw))
    finally:
        h.close()


@pytest.mark.gpu
def test_decode_parity_under_fading_all_equalizers(O, W):
    """Frames that fade while they are received, through k_channel_fading, decoded by every equalizer (and soft LS) on
    the GPU and by the oracle: identical frame tables, PSDUs, rows and equalised carrier points."""
    import os
    import torch
    from util import make_psdu
    w = W.wifi_b200
    rng = np.random.default_rng(77)
    n_links, fpl, gap, lead = 4, 64, 900, 200
    encs = [0, 2, 4, 7]
    specs = [(encs[f % 4], int(rng.integers(1200, 1529))) for f in range(n_links * fpl)]
    psdus = [make_psdu(O, rng, ln, seq=i) for i, (_, ln) in enumerate(specs)]
    h = W.Handle(max_samples=1 << 23, max_frames=4096, want_carrier=True)
    try:
        iq, boff = h.tx(psdus, enc=np.array([e for e, _ in specs], np.uint8))
        flen = np.diff(boff.astype(np.int64))
        strides = flen + gap
        link_len = [lead + int(strides[l * fpl:(l + 1) * fpl].sum()) for l in range(n_links)]
        link_off = np.concatenate([[0], np.cumsum(link_len)]).astype(np.int64)
        n = n_links * fpl
        segs = np.zeros(n, w.CHANSEG_DTYPE)
        fades = np.zeros(n, w.FADING_DTYPE)
        for f in range(n):
            l, k = divmod(f, fpl)
            segs["out_off"][f] = link_off[l] + lead + int(strides[l * fpl:f].sum())
        segs["in_off"], segs["in_len"], segs["n"] = boff[:-1].astype(np.int64), flen, strides
        segs["n0"] = segs["out_off"]
        segs["gain"], segs["noise_sigma"], segs["seed"] = 0.6, 0.6 * 10 ** (-25 / 20), 5
        segs["cfo"] = rng.uniform(-0.01, 0.01, n)
        fades["n_taps"], fades["n_sin"] = 3, 8
        fades["delay"][:, 1], fades["delay"][:, 2] = 1, 3
        fades["power"][:, :3] = np.array([0.6, 0.3, 0.1], np.float32)
        fades["doppler"], fades["seed"], fades["stream"] = 5e-4, 123, np.arange(n)
        fades["t0"] = segs["out_off"]
        tx = torch.from_numpy(iq.view(np.float32)).cuda()
        cap = torch.zeros(2 * int(link_off[-1]), dtype=torch.float32, device="cuda")
        h.channel_fading_dev(tx.data_ptr(), cap.data_ptr(), segs, fades)
        y = cap.cpu().numpy().view(np.complex64)
        lo = link_off.astype(np.uint64)
        threads = max(1, min(n_links, os.cpu_count() or 1))
        for algo, soft in ((0, False), (1, False), (2, False), (3, False), (0, True)):
            h.set_param(w.P_CHAN_EST, algo)
            h.set_param(w.P_SOFT_DECISION, int(soft))
            res = h.rx_batch(y, lo)
            ref = O.rx_links(y, link_off[:-1], np.diff(link_off), n_threads=threads, algo=algo, soft=soft)
            assert_frames_equal(res, ref)
            assert res.pdus() == ref.pdus()
            rows, car = h.rows(carrier=True)
            for i in range(len(ref.frames)):
                f, g = ref.frames[i], res.frames[i]
                assert np.array_equal(rows[g["row_off"]:g["row_off"] + g["n_rows"]], ref.rows[f["row_off"]:f["row_off"] + f["n_rows"]]), (algo, soft, i)
                assert np.array_equal(car[g["row_off"]:g["row_off"] + g["n_rows"]], ref.carrier[f["row_off"]:f["row_off"] + f["n_rows"]]), (algo, soft, i)
            assert ref.frames["sig_ok"].sum() > n // 2, (algo, soft)      # the frames were found; their data fades
            assert set(res.pdus()) <= {p[:-4] for p in psdus}
    finally:
        h.close()


@pytest.mark.gpu
def test_out_of_range_fading_is_refused_and_writes_nothing(W):
    import torch
    w = W.wifi_b200
    h = W.Handle(max_samples=1 << 16)
    try:
        x = torch.ones(2 * 256, dtype=torch.float32, device="cuda")
        y = torch.full_like(x, 7.0)
        good_s, good_f = _seg_pair(W, 256, {}, dict(taps=((0, 1.0),)))
        h.channel_fading_dev(x.data_ptr(), y.data_ptr(), good_s, good_f)
        assert not torch.all(y == 7.0)
        y.fill_(7.0)
        bad = [("n_taps", 0), ("n_taps", 9), ("n_sin", 0), ("n_sin", 17), ("k_factor", -1.0), ("k_factor", np.nan),
               ("doppler", 0.26), ("doppler", -1e-4), ("doppler", np.nan), ("los_doppler", 0.3), ("los_doppler", -0.3)]
        cases = []
        for field, v in bad:
            f = good_f.copy()
            f[field] = v
            cases.append((good_s, f))
        for field, v in (("delay", -1), ("power", -0.5), ("power", np.inf)):
            f = good_f.copy()
            f[field][0, 0] = v
            cases.append((good_s, f))
        s = good_s.copy()
        s["n_taps"] = 1                                   # a static segment handed to the fading entry point
        cases.append((s, good_f))
        two = np.concatenate([good_s, good_s])            # one bad record among good ones still refuses the whole call
        f2 = np.concatenate([good_f, good_f])
        f2["n_sin"][1] = 99
        cases.append((two, f2))
        for s, f in cases:
            with pytest.raises(w.WifiB200Error) as e:
                h.channel_fading_dev(x.data_ptr(), y.data_ptr(), s, f)
            assert e.value.code == w.E_ARG, (s, f)
            assert torch.all(y == 7.0)
            out = np.full(256, 7 + 7j, np.complex64)
            rc = h._L.wifi_b200_channel_fading(h._h, w._p(np.ones(256, np.complex64)), 256, w._p(out), 256, w._p(s), w._p(f), s.size)
            assert rc == w.E_ARG and np.all(out == 7 + 7j)
        assert h._L.wifi_b200_channel_fading_dev(h._h, x.data_ptr(), y.data_ptr(), w._p(good_s), None, 1) == w.E_ARG
    finally:
        h.close()


@pytest.mark.gpu
def test_device_evaluates_the_fading_contract_bit_for_bit(O, W):
    rng = np.random.default_rng(9)
    n = 1_000_000
    h = W.Handle(max_samples=1 << 16)
    try:
        p = rng.integers(0, 2 ** 32, n, dtype=np.uint32).view(np.float32)
        for got, want in zip(h.detmath(SINCOS_TURN, p), O.detmath(SINCOS_TURN, p)):
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
        seed, stream = [rng.integers(0, 2 ** 32, n, dtype=np.uint32).view(np.float32) for _ in range(2)]
        fd = rng.uniform(0, 0.25, n).astype(np.float32)
        M = rng.integers(1, 17, n)
        m = rng.integers(0, 17, n) % (M + 1)                      # m == n_sin: the line-of-sight term
        d = (rng.integers(0, 8, n) | (m << 4) | ((M - 1) << 12)).astype(np.uint32).view(np.float32)
        pw, kf = rng.uniform(0, 4, n).astype(np.float32), rng.uniform(0, 10, n).astype(np.float32)
        for fn in (FADING_ENTRY, FADING_FREQ):
            got, want = h.detmath(fn, seed, stream, fd, d, pw, kf), O.detmath(fn, seed, stream, fd, d, pw, kf)
            assert np.array_equal(got[0].view(np.uint32), want[0].view(np.uint32)) and np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32)), fn
        a, b, e, f = [rng.standard_normal(n).astype(np.float32) for _ in range(4)]
        fq, nn = [rng.integers(0, 2 ** 32, n, dtype=np.uint32).view(np.float32) for _ in range(2)]
        got, want = h.detmath(FADING_STEP, a, b, fq, nn, e, f), O.detmath(FADING_STEP, a, b, fq, nn, e, f)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    finally:
        h.close()


@pytest.mark.gpu
def test_loopback_runner_over_a_continuous_fading_channel(W):
    """--doppler-hz / --k-factor: the datagrams cross one flat Rician channel that keeps fading from burst to burst."""
    import pickle
    import socket
    import struct
    out = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    out.bind(("127.0.0.1", 0))
    out.settimeout(5)
    t = W.loopback_runner.IrsTransceiver(in_port=0, out_addr=("127.0.0.1", out.getsockname()[1]), snr=30.0, encoding=3,
                                         doppler_hz=300.0, k_factor=3.0, seed=4)
    seen = []
    chan = t.phy.handle.channel

    def recording(x, **kw):
        y = chan(x, **kw)
        seen.append((x.copy(), kw, y.copy()))
        return y
    t.phy.handle.channel = recording
    rng = np.random.default_rng(82)
    pieces = [((int(rng.integers(0, 30)), int(rng.integers(0, 30)), 0), rng.integers(0, 256, (10, 10, 1), dtype=np.uint8)) for _ in range(4)]
    sent = [pickle.dumps(p) for p in pieces]
    try:
        for data in sent:
            t.handle_datagram(struct.pack("=L", len(data)) + data)
        got = []
        while True:
            try:
                got.append(out.recvfrom(2048)[0])
            except socket.timeout:
                break
        assert got and all(g in sent for g in got)
        assert [kw["fading"]["t0"] for _, kw, _ in seen] == [kw["n0"] for _, kw, _ in seen]
        assert seen[1][1]["fading"]["t0"] == seen[0][2].size
        assert seen[0][1]["fading"]["doppler"] == 300.0 / 20e6 and seen[0][1]["fading"]["k_factor"] == 3.0
        # one channel call over both bursts gives exactly the two calls the runner made: the second continues the first
        x = np.concatenate([seen[0][0], seen[1][0]])
        kw = dict(seen[0][1], fading=dict(seen[0][1]["fading"], t0=0), n0=0)
        kw.pop("n_out")
        assert np.array_equal(chan(x, **kw), np.concatenate([seen[0][2], seen[1][2]]))
    finally:
        t.close()
        out.close()
