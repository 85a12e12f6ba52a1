"""The receiver, stage by stage, against the float64 model of tests/ref_model.py.

Every other receive-side test holds the CUDA library to the CPU oracle; both follow include/wifi_detmath.h and the same
restatement of gr-ieee802-11, so an error they share is invisible there.  Here the device under test -- the oracle
(CPU suite) or the library (GPU suite) -- is compared with the model computed from the formulas in float64: the plateau
flags, sync_short's triggers, freq_short, sync_long's frame start and freq_long, the SNR, the equalised points, the
decisions and the soft values.  Each model stage is fed the device's outputs of the stage before (its frame start, its
frequency offsets, its decisions for the decision-directed equalizers), so one point near a boundary cannot fork the
model away from the device.  Tolerances are those of SURVEY.md 8c where it states one.
"""
import functools
import warnings

import numpy as np
import pytest

import ref_model as M
from util import make_capture, make_psdu

FLAG_REL = 1e-5        # a flag may differ from the float64 decision only where ||a| - thr p| <= FLAG_REL * E
FREQ_TOL = 1e-5        # rad/sample, freq_short and freq_long
TIE_REL = 1e-6         # sync_long magnitudes this close make the top-4 ranking a coin toss: reported, not asserted
SNR_TOL = 0.01         # dB
POINT_TOL = 2e-3       # equalised points of frames with SNR >= 15 dB, and the decision-boundary guard
POINT_TOL_LOW = 1e-4   # frames below 15 dB: observed maximum 5.2e-6 (the 6-10 dB LMS capture), 19x headroom
TAPS3 = ((0, 1.0), (1, 0.4 * np.exp(1j * 1.0)), (3, 0.2 * np.exp(-2j)))


# ------------------------------------------------------------------------------------------------ devices under test
class Out:
    def __init__(self, frames, flags, rows, carrier, soft, pdus):
        self.frames, self.flags, self.rows, self.carrier, self.soft, self.pdus = frames, flags, rows, carrier, soft, pdus


class OracleDev:
    name = "oracle"

    def __init__(self, O):
        self.O = O

    def run(self, y, algo=0, soft=False, sc16=None):
        if sc16 is not None:
            y = dequantise(*sc16)
        r = self.O.rx(y, algo=algo, soft=soft)
        return Out(r.frames, self.O.flags(y, 0.56), r.rows, r.carrier, r.soft, r.pdus())


class LibraryDev:
    name = "library"

    def __init__(self, W, h):
        self.W, self.h = W, h

    def run(self, y, algo=0, soft=False, sc16=None):
        h, w = self.h, self.W.wifi_b200
        h.set_param(w.P_CHAN_EST, algo)
        h.set_param(w.P_SOFT_DECISION, int(soft))
        res = h.rx_batch(y) if sc16 is None else h.rx_batch_sc16(*sc16)
        rows, car = h.rows(carrier=True)
        return Out(res.frames, h.flags(0, y.size), rows, car, h.soft_rows() if soft else None, res.pdus())


@pytest.fixture(scope="module", params=["oracle", pytest.param("library", marks=pytest.mark.gpu)])
def dev(request, O):
    if request.param == "oracle":
        yield OracleDev(O)
        return
    W = request.getfixturevalue("W")
    h = W.Handle(max_samples=1 << 21, max_frames=4096, want_carrier=True)
    yield LibraryDev(W, h)
    h.close()


# ------------------------------------------------------------------------------------------------ captures (seeded)
def quantise(y, scale):
    return np.clip(np.rint(y.view(np.float32) / scale), -32768, 32767).astype(np.int16)


def dequantise(q, scale):
    return (q.astype(np.float32) * np.float32(scale)).view(np.complex64)


@functools.lru_cache(maxsize=None)
def digests_capture(O):
    """The capture of tests/golden/oracle_regression.json: every MCS plus a 1528-byte 64-QAM frame, 3 taps, 24 dB."""
    specs = [(e, 60 + 90 * e) for e in range(8)] + [(7, 1528), (3, 296)]
    return make_capture(O, np.random.default_rng(7), specs, snr_db=24, cfo=0.009, taps=TAPS3, seed=5, gap=900)[0]


@functools.lru_cache(maxsize=None)
def marginal_capture(O):
    """24 frames at 6 to 10 dB through 3 taps: decision-directed estimates under noise."""
    rng = np.random.default_rng(31)
    parts = [make_capture(O, rng, [(int(rng.integers(0, 8)), int(rng.integers(30, 400))) for _ in range(8)], snr_db=s,
                          cfo=0.004, taps=TAPS3, seed=40 + k, gap=700)[0] for k, s in enumerate((6, 8, 10))]
    return np.concatenate(parts).astype(np.complex64)


@functools.lru_cache(maxsize=None)
def cfo_capture(O, cfo):
    rng = np.random.default_rng(int(abs(cfo) * 1000))
    specs = [(e, int(rng.integers(60, 500))) for e in range(8)]
    return make_capture(O, rng, specs, snr_db=28, cfo=cfo, taps=TAPS3, seed=50, gap=800)[0]


@functools.lru_cache(maxsize=None)
def long_capture(O):
    """1528-byte BPSK 1/2 (511 symbols, 41281 samples) and 64-QAM 3/4 at CFO 0.02, 30 dB: the largest rotation phases."""
    return make_capture(O, np.random.default_rng(61), [(0, 1528), (7, 1528)], snr_db=30, cfo=0.02, seed=61, gap=1500)[0]


@functools.lru_cache(maxsize=None)
def gain_capture(O, gain):
    rng = np.random.default_rng(71)
    specs = [(e, int(rng.integers(60, 400))) for e in range(8)]
    return make_capture(O, rng, specs, snr_db=26, cfo=-0.007, seed=71, gap=700, gain=gain)[0]


@functools.lru_cache(maxsize=None)
def silence_capture(O):
    """Noise-free frames between exact zeros (100 before, 1000 after each frame, as IRS_tranceiver pads its bursts):
    every MCS, six PSDU lengths, gains 1e-3 / 0.6 / 37.  Returns (iq, psdus)."""
    rng = np.random.default_rng(1)
    parts, psdus = [], []
    for gain in (1e-3, 0.6, 37.0):
        for enc in range(8):
            for ln in (30, 100, 250, 480, 700, 900):
                p = make_psdu(O, rng, ln, seq=len(psdus))
                psdus.append(p)
                parts += [np.zeros(100, np.complex64), np.complex64(gain) * O.tx_frame(p, enc, seed=1 + len(psdus) % 127),
                          np.zeros(1000, np.complex64)]
    return np.concatenate(parts).astype(np.complex64), psdus


# ------------------------------------------------------------------------------------------------ stage checks
def check_frontend(y, out, rep):
    """Flags against the float64 decision; the triggers against sync_short's state machine run on the device's flags
    (exact) and on the model's (the same set up to in-band flags); freq_short.  rep collects the largest deviation of
    every stage (for reporting)."""
    a, p, flags, margin, E = M.frontend(y)
    got = np.asarray(out.flags, bool)
    assert got.size == y.size
    assert not (got & (p == 0)).any(), ("flag in a window of exact zeros", np.flatnonzero(got & (p == 0))[:10])
    diff = np.flatnonzero(got != flags)
    inband = margin <= FLAG_REL * E
    assert inband[diff].all(), ("flag differs from the float64 decision", diff[~inband[diff]][:10])
    rep["flag_diffs"] = rep.get("flag_diffs", 0) + diff.size
    F = out.frames
    t, blen, fs = M.sync_short(got, a, y.size)
    assert np.array_equal(t, F["trigger"]), (t[:10], F["trigger"][:10])
    assert np.array_equal(blen, F["burst_len"])
    t2, _, _ = M.sync_short(flags, a, y.size)
    for u in np.setxor1d(t, t2):
        lo, hi = max(0, u - 3), min(y.size, u + 4)                # min_plateau + 1 = 3 samples either side
        assert inband[lo:hi].any(), ("trigger not explained by an in-band flag", u)
    if t.size:
        d = np.abs(fs - F["freq_short"].astype(np.float64))
        rep["freq_short"] = max(rep.get("freq_short", 0.0), float(d.max()))
        assert d.max() <= FREQ_TOL, ("freq_short", int(np.argmax(d)), d.max())


def check_chain(y, out, algo, soft, rep):
    """sync_long, the equaliser, the decisions and the soft values of every frame, each stage on the device's outputs
    of the stage before."""
    F = out.frames
    fo = 0.0
    n_checked = 0
    for i, f in enumerate(F):
        t, bl = int(f["trigger"]), int(f["burst_len"])
        s = M.sync_long(y, t, bl, f["freq_short"], fo)
        if s["tie"] < TIE_REL:
            warnings.warn("sync_long ranking tie at trigger %d (relative gap %.1e): frame_start not compared" % (t, s["tie"]))
        else:
            assert (s["frame_start"], s["found"]) == (int(f["frame_start"]), int(f["found"])), (i, s, f)
        fo = float(f["freq_long"])
        dfl = abs(s["freq_long"] - fo)
        rep["freq_long"] = max(rep.get("freq_long", 0.0), dfl)
        assert dfl <= FREQ_TOL, ("freq_long", i, s["freq_long"], fo)
        if not f["sig_ok"]:
            continue
        enc, nr = int(f["encoding"]), int(f["n_rows"])
        sy = M.symbols(y, t, bl, f["freq_short"], f["freq_long"], int(f["frame_start"]), 3 + nr)
        rows = out.rows[f["row_off"]:f["row_off"] + nr]
        q = M.equalize(sy, enc, algo, f["freq_short"], f["freq_long"], rows=rows)
        dsnr = abs(q["snr"] - float(f["snr"]))
        rep["snr"] = max(rep.get("snr", 0.0), dsnr)
        assert dsnr <= SNR_TOL, ("snr", i, q["snr"], f["snr"])
        if not nr:
            continue
        n_checked += 1
        car = out.carrier[f["row_off"]:f["row_off"] + nr].astype(np.complex128)
        dp = float(np.abs(q["points"] - car).max())
        key = "points" if q["snr"] >= 15 else "points_low_snr"
        rep[key] = max(rep.get(key, 0.0), dp)
        assert dp <= (POINT_TOL if q["snr"] >= 15 else POINT_TOL_LOW), ("points", i, algo, q["snr"], dp)
        near, dist = M.decide_nearest(enc, q["points"])
        clear = dist > POINT_TOL
        assert np.array_equal(rows[clear], near[clear]), ("decisions", i, np.argwhere((rows != near) & clear)[:5])
        if soft:
            nb = M.N_BPSC[enc]
            sv = out.soft[f["row_off"]:f["row_off"] + nr, :48 * nb].astype(np.int64)
            want = np.clip(np.rint(q["soft"]), -32, 32)
            dq = np.abs(sv - want)
            assert dq.max() <= 1, ("soft", i, dq.max())
            firm = np.abs(np.abs(q["soft"] - np.floor(q["soft"])) - 0.5) >= 0.05
            assert np.array_equal(sv[firm], want[firm]), ("soft", i, np.argwhere((sv != want) & firm)[:5])
            rep["soft_off_by_one"] = rep.get("soft_off_by_one", 0) + int((dq > 0).sum())
    return n_checked


def check_capture(y, out, algo=0, soft=False, rep=None):
    rep = {} if rep is None else rep
    check_frontend(y, out, rep)
    return check_chain(y, out, algo, soft, rep), rep


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("algo", range(4))
def test_digests_capture_stage_by_stage(dev, O, algo):
    """The workload of the committed digests, under every equalizer, hard and soft, now with tolerances from outside."""
    y = digests_capture(O)
    for soft in (False, True):
        out = dev.run(y, algo=algo, soft=soft)
        n, rep = check_capture(y, out, algo, soft)
        assert n == 10, n                                    # every frame's SIGNAL decoded: the whole chain was compared


def test_marginal_frames_lms(dev, O):
    """Frames at 6 to 10 dB with LMS: the model's channel estimate follows the device's decisions."""
    y = marginal_capture(O)
    out = dev.run(y, algo=1)
    n, rep = check_capture(y, out, algo=1)
    assert n >= 12 and len(out.frames) >= 20, (n, len(out.frames))


@pytest.mark.parametrize("cfo", [-0.03, 0.04])
def test_large_frequency_offsets(dev, O, cfo):
    y = cfo_capture(O, cfo)
    for algo in (0, 3):
        out = dev.run(y, algo=algo)
        n, rep = check_capture(y, out, algo)
        assert n == 8 and sum(out.frames["crc_ok"]) == 8


def test_longest_frames_hard_and_soft(dev, O):
    """511 BPSK symbols and a 1528-byte 64-QAM 3/4 frame at CFO 0.02: the largest rotation phases.  In soft mode the
    BPSK frame is 12264 trellis steps of confident soft values (|q| near 16 throughout, the metric spread growing at its
    largest sustained rate), and two in five of the 64-QAM values sit at the +-32 clamp."""
    y = long_capture(O)
    for soft in (False, True):
        out = dev.run(y, algo=0, soft=soft)
        n, rep = check_capture(y, out, 0, soft)
        assert n == 2 and list(out.frames["crc_ok"]) == [1, 1] and list(out.frames["length"]) == [1528, 1528]
        assert int(out.frames["n_rows"][0]) == 511
        if soft:
            F = out.frames
            bpsk = out.soft[F["row_off"][0]:F["row_off"][0] + 511, :48]
            qam = out.soft[F["row_off"][1]:F["row_off"][1] + int(F["n_rows"][1]), :288]
            assert np.abs(bpsk).min() >= 8 and (np.abs(qam) == 32).mean() > 0.3


@pytest.mark.parametrize("gain", [1e-4, 3e3])
def test_amplitude_extremes(dev, O, gain):
    y = gain_capture(O, gain)
    out = dev.run(y, algo=2)
    n, rep = check_capture(y, out, 2)
    assert n == 8 and sum(out.frames["crc_ok"]) == 8


@pytest.mark.parametrize("fmt", ["fc32", "sc16"])
def test_silence_does_not_cut_frames_short(dev, O, fmt):
    """Noise-free frames between exact zeros: a window of zeros is never over the threshold, whatever residue the
    running sums keep, so no trigger falls into the silence behind a frame and truncates it.  Every frame decodes,
    and no record without a SIGNAL field appears.  sc16: each gain's 48 frames as a 16-bit recording whose full scale
    is four times that gain (the frames peak at 3.6 times it)."""
    x, psdus = silence_capture(O)
    n = x.size // 3
    if fmt == "fc32":
        runs = [(x, None, psdus)]
    else:
        runs = []
        for g, gain in enumerate((1e-3, 0.6, 37.0)):
            scale = np.float32(gain * 4 / 32768)
            q = quantise(x[g * n:(g + 1) * n], scale)
            runs.append((dequantise(q, scale), (q, scale), psdus[48 * g:48 * (g + 1)]))
    for y, sc16, want in runs:
        out = dev.run(y, sc16=sc16)
        check_frontend(y, out, {})
        F = out.frames
        assert F["sig_ok"].all(), ("record without a SIGNAL field", F[F["sig_ok"] == 0]["trigger"][:5], F[F["sig_ok"] == 0]["burst_len"][:5])
        assert len(F) == len(want) and F["crc_ok"].all(), np.flatnonzero(F["crc_ok"] == 0)
        assert out.pdus == [p[:-4] for p in want]
