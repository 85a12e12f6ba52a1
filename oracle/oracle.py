"""ctypes binding of the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY -- imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  The product package never
imports this module (tests/test_abi_and_host.py::test_product_never_touches_the_oracle greps for it).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

FRAME_DTYPE = np.dtype([
    ("trigger", "<i8"), ("link", "<i4"), ("burst_len", "<i4"), ("freq_short", "<f4"), ("freq_long", "<f4"),
    ("found", "<i4"), ("frame_start", "<i4"), ("n_syms", "<i4"), ("sig_ok", "<i4"), ("encoding", "<i4"),
    ("length", "<i4"), ("frame_symbols", "<i4"), ("n_rows", "<i4"), ("accepted", "<i4"), ("decoded", "<i4"),
    ("crc_ok", "<i4"), ("snr", "<f8"), ("row_off", "<i8"), ("psdu_off", "<i8"),
], align=True)


class RxCfg(C.Structure):
    _fields_ = [("threshold", C.c_double), ("min_plateau", C.c_int32), ("algo", C.c_int32), ("freq", C.c_double),
                ("bw", C.c_double), ("final", C.c_int32), ("want_carrier", C.c_int32), ("soft", C.c_int32), ("hist", C.c_int32),
                ("min_pos", C.c_int64), ("fo_carry", C.c_float), ("pad", C.c_int32)]


class ChanCfg(C.Structure):
    _fields_ = [("gain", C.c_float), ("cfo", C.c_float), ("phase0", C.c_float), ("noise_sigma", C.c_float),
                ("n_taps", C.c_int32), ("delay", C.c_int32 * 8), ("tap_re", C.c_float * 8), ("tap_im", C.c_float * 8),
                ("seed", C.c_uint64), ("stream", C.c_uint64)]


class FadingCfg(C.Structure):
    """Same layout and meaning as wifi_b200_fading (include/wifi_b200.h)."""
    _fields_ = [("n_taps", C.c_int32), ("n_sin", C.c_int32), ("delay", C.c_int32 * 8), ("power", C.c_float * 8),
                ("k_factor", C.c_float), ("doppler", C.c_float), ("los_doppler", C.c_float), ("reserved", C.c_int32),
                ("t0", C.c_int64), ("seed", C.c_uint64), ("stream", C.c_uint64)]


def build(force=False):
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, "wifi_oracle.cpp"), os.path.join(_HERE, "wifi_oracle.h"),
            os.path.join(_HERE, "..", "include", "wifi_detmath.h")]
    have_src = all(os.path.exists(s) for s in srcs)
    hfile = so + ".srchash"
    digest = None
    if have_src:
        import hashlib
        hh = hashlib.sha256()
        for s in srcs + [os.path.join(_HERE, "Makefile")]:
            hh.update(open(s, "rb").read())
        digest = hh.hexdigest()
    try:
        stale = have_src and open(hfile).read().strip() != digest   # content, not mtimes: the tree is copied to the GPU box
    except OSError:
        stale = have_src
    if force or not os.path.exists(so) or stale:
        subprocess.check_call(["make", "-C", _HERE, "-B", "liboracle.so"])
        if digest:
            with open(hfile, "w") as f:
                f.write(digest)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        L = _LIB
        L.orc_rx.restype = C.c_void_p
        L.orc_rx_links.restype = C.c_void_p
        L.orc_rx_n_frames.restype = C.c_int64
        L.orc_rx_n_rows.restype = C.c_int64
        L.orc_rx_psdu_bytes.restype = C.c_int64
        L.orc_crc32.restype = C.c_uint32
        for f in ("orc_rx_n_frames", "orc_rx_n_rows", "orc_rx_psdu_bytes", "orc_rx_free"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.orc_rx_copy.argtypes = [C.c_void_p] * 5
        L.orc_rx_copy_soft.argtypes = [C.c_void_p] * 2
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def mcs(enc):
    v = [C.c_int() for _ in range(5)]
    if lib().orc_mcs(enc, *[C.byref(x) for x in v]):
        raise ValueError(enc)
    return dict(zip(("n_bpsc", "n_cbps", "n_dbps", "rate_field", "punct"), [x.value for x in v]))


def n_sym(enc, psdu_len):
    return lib().orc_n_sym(enc, psdu_len)


def scramble(bits, seed):
    b = np.ascontiguousarray(bits, np.uint8)
    o = np.empty_like(b)
    lib().orc_scramble(_p(b), _p(o), C.c_int(b.size), C.c_int(seed))
    return o


def conv_encode(bits):
    b = np.ascontiguousarray(bits, np.uint8)
    o = np.empty(2 * b.size, np.uint8)
    lib().orc_conv_encode(_p(b), _p(o), C.c_int(b.size))
    return o


def puncture(bits, enc):
    b = np.ascontiguousarray(bits, np.uint8)
    o = np.empty(b.size, np.uint8)
    n = lib().orc_puncture(_p(b), _p(o), C.c_int(b.size), C.c_int(enc))
    return o[:n].copy()


def interleave(bits, enc, reverse=False):
    b = np.ascontiguousarray(bits, np.uint8)
    ncb = mcs(enc)["n_cbps"]
    assert b.size % ncb == 0
    o = np.empty_like(b)
    lib().orc_interleave(_p(b), _p(o), C.c_int(b.size // ncb), C.c_int(enc), C.c_int(int(reverse)))
    return o


def signal_field(enc, length):
    o = np.empty(48, np.uint8)
    lib().orc_signal_field(C.c_int(enc), C.c_int(length), _p(o))
    return o


def polarity():
    o = np.empty(127, np.float32)
    lib().orc_polarity(_p(o))
    return o


def long_taps():
    o = np.empty(128, np.float32)
    lib().orc_long_taps(_p(o))
    return o.view(np.complex64)


def lts_freq():
    o = np.empty(64, np.float32)
    lib().orc_lts_freq(_p(o))
    return o


def constellation(enc):
    n = 1 << mcs(enc)["n_bpsc"]
    o = np.empty(2 * n, np.float32)
    lib().orc_constellation(C.c_int(enc), _p(o))
    return o.view(np.complex64)


def decide(enc, z):
    return lib().orc_decide(C.c_int(enc), C.c_float(z.real), C.c_float(z.imag))


def fft64(x, inverse=False):
    a = np.ascontiguousarray(x, np.complex64)
    o = np.empty(64, np.complex64)
    lib().orc_fft64(_p(a), _p(o), C.c_int(int(inverse)))
    return o


def viterbi(depunctured, n_bits, ntraceback):
    d = np.ascontiguousarray(depunctured, np.uint8)
    o = np.zeros(n_bits + 8, np.uint8)
    lib().orc_viterbi(_p(d), C.c_int(d.size), C.c_int(n_bits), C.c_int(ntraceback), _p(o))
    return o[:n_bits]


def viterbi_soft(depunctured, n_bits, ntraceback):
    d = np.ascontiguousarray(depunctured, np.int8)
    o = np.zeros(n_bits + 8, np.uint8)
    lib().orc_viterbi_soft(_p(d), C.c_int(d.size), C.c_int(n_bits), C.c_int(ntraceback), _p(o))
    return o[:n_bits]


def crc32(data):
    d = np.frombuffer(bytes(data), np.uint8)
    return lib().orc_crc32(_p(d), C.c_int(d.size))


def mac_frame(payload, seq, src=b"\x23" * 6, dst=b"\x42" * 6, bss=b"\xff" * 6):
    pl = np.frombuffer(bytes(payload), np.uint8)
    o = np.empty(pl.size + 28, np.uint8)
    n = lib().orc_mac_frame(_p(pl), C.c_int(pl.size), C.c_int(seq), C.c_char_p(src), C.c_char_p(dst), C.c_char_p(bss), _p(o))
    if n < 0:
        raise ValueError("payload too large")
    return o[:n].tobytes()


def tx_symbols(psdu, enc, seed):
    p = np.frombuffer(bytes(psdu), np.uint8)
    o = np.empty(511 * 48, np.uint8)
    ns = lib().orc_tx_symbols(_p(p), C.c_int(p.size), C.c_int(enc), C.c_int(seed), _p(o))
    if ns < 0:
        raise ValueError("psdu too large")
    return o[:ns * 48].reshape(ns, 48).copy()


def tx_frame(psdu, enc, seed):
    p = np.frombuffer(bytes(psdu), np.uint8)
    cap = 80 * (5 + 511) + 1
    o = np.empty(cap, np.complex64)
    n = lib().orc_tx_frame(_p(p), C.c_int(p.size), C.c_int(enc), C.c_int(seed), _p(o), C.c_int(cap))
    if n < 0:
        raise ValueError("psdu too large")
    return o[:n].copy()


def chan_cfg(gain=1.0, cfo=0.0, phase0=0.0, noise_sigma=0.0, taps=((0, 1.0 + 0j),), seed=0, stream=0):
    c = ChanCfg()
    c.gain, c.cfo, c.phase0, c.noise_sigma = gain, cfo, phase0, noise_sigma
    c.n_taps = len(taps)
    for i, (d, h) in enumerate(taps):
        c.delay[i] = int(d)
        c.tap_re[i] = np.float32(complex(h).real)
        c.tap_im[i] = np.float32(complex(h).imag)
    c.seed, c.stream = seed, stream
    return c


def fading_cfg(taps=((0, 1.0),), n_sin=8, k_factor=0.0, doppler=0.0, los_doppler=0.0, t0=0, seed=0, stream=0):
    """taps = ((delay, power), ...); the rest as wifi_b200_fading."""
    f = FadingCfg()
    f.n_taps, f.n_sin = len(taps), n_sin
    for i, (d, p) in enumerate(taps):
        f.delay[i], f.power[i] = int(d), float(p)
    f.k_factor, f.doppler, f.los_doppler = k_factor, doppler, los_doppler
    f.t0, f.seed, f.stream = t0, seed, stream
    return f


def channel(x, n0=0, fading=None, **kw):
    """Gain, taps, CFO rotation and Philox AWGN keyed by seed / stream at counter n0 + i (keywords of chan_cfg).
    fading: the time-varying taps instead of the fixed ones, as a FadingCfg, a FADING_DTYPE record or a dict of
    fading_cfg keywords; out-of-range parameters raise ValueError."""
    a = np.ascontiguousarray(x, np.complex64)
    o = np.empty_like(a)
    if fading is None:
        cfg = kw.pop("cfg", None) or chan_cfg(**kw)
        lib().orc_channel(_p(a), _p(o), C.c_int64(a.size), C.c_int64(n0), C.byref(cfg))
        return o
    if isinstance(fading, dict):
        fading = fading_cfg(**fading)
    elif isinstance(fading, np.ndarray):
        fading = FadingCfg.from_buffer_copy(np.ascontiguousarray(fading).tobytes())
    kw.setdefault("taps", ())
    cfg = chan_cfg(**kw)
    if lib().orc_channel_fading(_p(a), _p(o), C.c_int64(a.size), C.c_int64(n0), C.byref(cfg), C.byref(fading)):
        raise ValueError("fading parameters out of range")
    return o


def frontend(x):
    a = np.ascontiguousarray(x, np.complex64)
    ao = np.empty(a.size, np.complex64)
    po = np.empty(a.size, np.float32)
    co = np.empty(a.size, np.float32)
    lib().orc_frontend(_p(a), C.c_int64(a.size), _p(ao), _p(po), _p(co))
    return ao, po, co


def flags(x, threshold=0.56):
    """sync_short's per-sample plateau test as the numerical contract states it (squares, see wifi_oracle.cpp rx_link)."""
    a = np.ascontiguousarray(x, np.complex64)
    o = np.zeros(a.size, np.uint8)
    lib().orc_flags(_p(a), C.c_int64(a.size), C.c_double(threshold), _p(o))
    return o.astype(bool)


class RxResult:
    def __init__(self, frames, rows, carrier, psdu):
        self.frames, self.rows, self.carrier, self.psdu_blob = frames, rows, carrier, psdu

    def psdu(self, i):
        f = self.frames[i]
        if f["psdu_off"] < 0:
            return None
        return self.psdu_blob[f["psdu_off"]:f["psdu_off"] + f["length"]].tobytes()

    def pdus(self):
        """What decode_mac publishes on 'out': PSDU without FCS for CRC-ok frames."""
        return [self.psdu(i)[:-4] for i in range(len(self.frames)) if self.frames[i]["crc_ok"]]


def rx_cfg(threshold=0.56, min_plateau=2, algo=0, freq=5.89e9, bw=10e6, final=True, want_carrier=True, soft=False,
           hist=0, min_pos=0, fo_carry=0.0):
    return RxCfg(threshold, min_plateau, algo, freq, bw, int(final), int(want_carrier), int(soft), int(hist), int(min_pos), float(fo_carry), 0)


def _collect(h, want_carrier, soft=False):
    L = lib()
    nf, nr, nb = L.orc_rx_n_frames(h), L.orc_rx_n_rows(h), L.orc_rx_psdu_bytes(h)
    frames = np.zeros(nf, FRAME_DTYPE)
    rows = np.zeros((nr, 48), np.uint8)
    carrier = np.zeros((nr, 48), np.complex64) if want_carrier else None
    psdu = np.zeros(nb, np.uint8)
    L.orc_rx_copy(h, _p(frames), _p(rows), _p(carrier) if want_carrier else None, _p(psdu))
    res = RxResult(frames, rows, carrier, psdu)
    res.soft = None
    if soft:
        res.soft = np.zeros((nr, 288), np.int8)
        L.orc_rx_copy_soft(h, _p(res.soft))
    L.orc_rx_free(h)
    return res


def rx(x, link=0, **kw):
    """hist > 0: the first `hist` samples of x are history in front of the stream's sample 0 (a resumed stream)."""
    cfg = rx_cfg(**kw)
    a = np.ascontiguousarray(x, np.complex64)
    h = lib().orc_rx(C.c_void_p(a.ctypes.data + 8 * cfg.hist), C.c_int64(a.size - cfg.hist), C.c_int(link), C.byref(cfg))
    return _collect(C.c_void_p(h), bool(cfg.want_carrier), bool(cfg.soft))


def detmath(fn, a, b=None, c=None, d=None, o0=None, o1=None):
    """Element-wise wdm_selftest(fn, ...) of include/wifi_detmath.h on the host; returns (o0, o1)."""
    a = np.ascontiguousarray(a, np.float32)
    z = np.zeros_like(a)
    b, c, d = [z if v is None else np.ascontiguousarray(v, np.float32) for v in (b, c, d)]
    o0 = np.zeros_like(a) if o0 is None else np.array(o0, np.float32)
    o1 = np.zeros_like(a) if o1 is None else np.array(o1, np.float32)
    lib().orc_detmath(C.c_int(fn), _p(a), _p(b), _p(c), _p(d), _p(o0), _p(o1), C.c_int64(a.size))
    return o0, o1


def rx_links(x, offsets, lengths, n_threads=1, **kw):
    cfg = rx_cfg(**kw)
    a = np.ascontiguousarray(x, np.complex64)
    off = np.ascontiguousarray(offsets, np.int64)
    ln = np.ascontiguousarray(lengths, np.int64)
    h = lib().orc_rx_links(_p(a), _p(off), _p(ln), C.c_int(off.size), C.byref(cfg), C.c_int(n_threads))
    return _collect(C.c_void_p(h), bool(cfg.want_carrier), bool(cfg.soft))
