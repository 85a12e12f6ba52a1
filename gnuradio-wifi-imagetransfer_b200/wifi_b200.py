"""ctypes binding of libwifi_b200.so (include/wifi_b200.h).  There is no CPU path in this
module: every compute call goes to the CUDA library and raises WifiB200Error if it fails."""
import ctypes as C
import os

import numpy as np

from . import build as _build

FRAME_DTYPE = np.dtype([
    ("trigger", "<i8"), ("link", "<i4"), ("burst_len", "<i4"), ("freq_short", "<f4"), ("freq_long", "<f4"),
    ("found", "<i4"), ("frame_start", "<i4"), ("n_syms", "<i4"), ("sig_ok", "<i4"), ("encoding", "<i4"),
    ("length", "<i4"), ("frame_symbols", "<i4"), ("n_rows", "<i4"), ("accepted", "<i4"), ("decoded", "<i4"),
    ("crc_ok", "<i4"), ("snr", "<f8"), ("row_off", "<i8"), ("psdu_off", "<i8"),
], align=True)
PSDU_STRIDE = 1536
vp_t = C.c_void_p

ENCODINGS = ("BPSK_1_2", "BPSK_3_4", "QPSK_1_2", "QPSK_3_4", "QAM16_1_2", "QAM16_3_4", "QAM64_2_3", "QAM64_3_4")
EQUALIZERS = ("LS", "LMS", "COMB", "STA")
P_BANDWIDTH, P_FREQUENCY, P_SENSITIVITY, P_CHAN_EST, P_ENCODING, P_MIN_PLATEAU, P_WANT_CARRIER, P_SOFT_DECISION, P_STREAM_BATCH, P_HOST_GROUP_SAMPLES, P_VITERBI_FORM = range(11)
E_ARG, E_TOO_LARGE, E_CUDA, E_NOMEM, E_OVERFLOW, E_NODEVICE = -1, -2, -3, -4, -5, -6


class Cfg(C.Structure):
    _fields_ = [("bandwidth", C.c_double), ("frequency", C.c_double), ("sensitivity", C.c_double),
                ("chan_est", C.c_int32), ("encoding", C.c_int32), ("min_plateau", C.c_int32), ("device", C.c_int32),
                ("want_carrier", C.c_int32), ("soft_decision", C.c_int32), ("max_samples", C.c_int64), ("max_frames", C.c_int64)]


class ChanSeg(C.Structure):
    _fields_ = [("in_off", C.c_int64), ("in_len", C.c_int64), ("out_off", C.c_int64), ("n", C.c_int64), ("n0", C.c_int64),
                ("gain", C.c_float), ("cfo", C.c_float), ("phase0", C.c_float), ("noise_sigma", C.c_float),
                ("n_taps", C.c_int32), ("delay", C.c_int32 * 8), ("tap_re", C.c_float * 8), ("tap_im", C.c_float * 8),
                ("seed", C.c_uint64), ("stream", C.c_uint64)]


CHANSEG_DTYPE = np.dtype([
    ("in_off", "<i8"), ("in_len", "<i8"), ("out_off", "<i8"), ("n", "<i8"), ("n0", "<i8"),
    ("gain", "<f4"), ("cfo", "<f4"), ("phase0", "<f4"), ("noise_sigma", "<f4"), ("n_taps", "<i4"),
    ("delay", "<i4", (8,)), ("tap_re", "<f4", (8,)), ("tap_im", "<f4", (8,)), ("seed", "<u8"), ("stream", "<u8")], align=True)
assert CHANSEG_DTYPE.itemsize == C.sizeof(ChanSeg), (CHANSEG_DTYPE.itemsize, C.sizeof(ChanSeg))


class Fading(C.Structure):
    _fields_ = [("n_taps", C.c_int32), ("n_sin", C.c_int32), ("delay", C.c_int32 * 8), ("power", C.c_float * 8),
                ("k_factor", C.c_float), ("doppler", C.c_float), ("los_doppler", C.c_float), ("reserved", C.c_int32),
                ("t0", C.c_int64), ("seed", C.c_uint64), ("stream", C.c_uint64)]


FADING_DTYPE = np.dtype([
    ("n_taps", "<i4"), ("n_sin", "<i4"), ("delay", "<i4", (8,)), ("power", "<f4", (8,)), ("k_factor", "<f4"), ("doppler", "<f4"),
    ("los_doppler", "<f4"), ("reserved", "<i4"), ("t0", "<i8"), ("seed", "<u8"), ("stream", "<u8")], align=True)
assert FADING_DTYPE.itemsize == C.sizeof(Fading) == 112, (FADING_DTYPE.itemsize, C.sizeof(Fading))


LINK_STATE_DTYPE = np.dtype([("min_pos", "<i8"), ("fo_carry", "<f4"), ("hist", "<i4")], align=True)


class Stats(C.Structure):
    _fields_ = [("samples", C.c_int64), ("frames_detected", C.c_int64), ("signal_ok", C.c_int64), ("decoded", C.c_int64),
                ("crc_ok", C.c_int64), ("pdu_bytes", C.c_int64), ("per_mcs_crc_ok", C.c_int64 * 8)]


class WifiB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libwifi_b200: %s (code %d)" % (msg, code))
        self.code = code


EXPORTS = [
    "wifi_b200_abi_version", "wifi_b200_device_count", "wifi_b200_create", "wifi_b200_destroy", "wifi_b200_set_param",
    "wifi_b200_get_param", "wifi_b200_last_error", "wifi_b200_strerror", "wifi_b200_stream", "wifi_b200_sync",
    "wifi_b200_mac_frame", "wifi_b200_n_sym", "wifi_b200_frame_samples", "wifi_b200_tx", "wifi_b200_tx_dev",
    "wifi_b200_tx_symbols", "wifi_b200_channel_dev", "wifi_b200_channel", "wifi_b200_channel_fading_dev", "wifi_b200_channel_fading", "wifi_b200_rx_batch", "wifi_b200_rx_batch_dev", "wifi_b200_rx_batch_dev_state", "wifi_b200_rx_batch_sc16", "wifi_b200_rx_counts",
    "wifi_b200_rx_frames", "wifi_b200_rx_rows", "wifi_b200_rx_psdus", "wifi_b200_rx_soft", "wifi_b200_rx_flags", "wifi_b200_rx_push",
    "wifi_b200_rx_pop", "wifi_b200_rx_reset", "wifi_b200_rx_push_links", "wifi_b200_get_stats", "wifi_b200_stage_times", "wifi_b200_stage_name",
    "wifi_b200_selftest_detmath", "wifi_b200_alu_peak", "wifi_b200_rx_push_links_async", "wifi_b200_rx_push_links_sc16_async", "wifi_b200_rx_push_wait", "wifi_b200_rx_pop_view",
    "wifi_b200_host_alloc", "wifi_b200_host_free",
]

_LIB = None


def lib():
    """Loads (building if stale) the CUDA library.  Raises if it cannot be built or loaded."""
    global _LIB
    if _LIB is None:
        so = _build.build()
        L = C.CDLL(so)
        vp, i64, u64p = C.c_void_p, C.c_int64, C.POINTER(C.c_uint64)
        L.wifi_b200_create.argtypes = [C.POINTER(Cfg), C.POINTER(vp)]
        L.wifi_b200_destroy.argtypes = [vp]
        L.wifi_b200_destroy.restype = None
        L.wifi_b200_set_param.argtypes = [vp, C.c_int, C.c_double]
        L.wifi_b200_get_param.argtypes = [vp, C.c_int]
        L.wifi_b200_get_param.restype = C.c_double
        L.wifi_b200_last_error.argtypes = [vp]
        L.wifi_b200_last_error.restype = C.c_char_p
        L.wifi_b200_strerror.restype = C.c_char_p
        L.wifi_b200_stream.argtypes = [vp]
        L.wifi_b200_stream.restype = vp
        L.wifi_b200_sync.argtypes = [vp]
        L.wifi_b200_mac_frame.argtypes = [vp, C.c_int, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, vp]
        for f in ("wifi_b200_tx", "wifi_b200_tx_dev"):
            getattr(L, f).argtypes = [vp, vp, vp, vp, vp, vp, C.c_int, vp, C.c_size_t, vp]
            getattr(L, f).restype = i64
        L.wifi_b200_tx_symbols.argtypes = [vp, vp, C.c_size_t]
        L.wifi_b200_tx_symbols.restype = i64
        L.wifi_b200_channel_dev.argtypes = [vp, vp, vp, vp, C.c_int]
        L.wifi_b200_channel.argtypes = [vp, vp, i64, vp, i64, vp, C.c_int]
        L.wifi_b200_channel_fading_dev.argtypes = [vp, vp, vp, vp, vp, C.c_int]
        L.wifi_b200_channel_fading.argtypes = [vp, vp, i64, vp, i64, vp, vp, C.c_int]
        for f in ("wifi_b200_rx_batch", "wifi_b200_rx_batch_dev"):
            getattr(L, f).argtypes = [vp, vp, vp, C.c_int, C.c_int]
        L.wifi_b200_rx_batch_dev_state.argtypes = [vp, vp, vp, C.c_int, C.c_int, vp]
        L.wifi_b200_rx_batch_sc16.argtypes = [vp, vp, C.c_float, vp, C.c_int, C.c_int]
        L.wifi_b200_rx_counts.argtypes = [vp, vp, vp, vp, vp]
        L.wifi_b200_rx_frames.argtypes = [vp, vp, i64]
        L.wifi_b200_rx_rows.argtypes = [vp, vp, vp, i64]
        L.wifi_b200_rx_psdus.argtypes = [vp, vp, C.c_size_t]
        L.wifi_b200_rx_soft.argtypes = [vp, vp, i64]
        L.wifi_b200_rx_flags.argtypes = [vp, C.c_int, vp, i64]
        L.wifi_b200_rx_push.argtypes = [vp, vp, C.c_size_t, C.c_int]
        L.wifi_b200_rx_push_links.argtypes = [vp, vp, vp, C.c_int, C.c_int]
        L.wifi_b200_rx_push_links_async.argtypes = [vp, vp, vp, C.c_int, C.c_int]
        L.wifi_b200_rx_push_links_sc16_async.argtypes = [vp, vp, C.c_float, vp, C.c_int, C.c_int]
        L.wifi_b200_rx_push_wait.argtypes = [vp]
        L.wifi_b200_rx_pop.argtypes = [vp, vp, C.c_int, vp, C.c_size_t, C.POINTER(C.c_int)]
        L.wifi_b200_rx_pop_view.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
        L.wifi_b200_rx_reset.argtypes = [vp]
        L.wifi_b200_get_stats.argtypes = [vp, C.POINTER(Stats)]
        L.wifi_b200_stage_times.argtypes = [vp, vp, C.c_int]
        L.wifi_b200_stage_name.restype = C.c_char_p
        L.wifi_b200_selftest_detmath.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, i64]
        L.wifi_b200_alu_peak.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.wifi_b200_host_alloc.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
        L.wifi_b200_host_free.argtypes = [vp, vp]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def device_count():
    return lib().wifi_b200_device_count()


def mac_frame(payload, seq, src=b"\x23" * 6, dst=b"\x42" * 6, bss=b"\xff" * 6):
    """[UPSTREAM] ieee802_11.mac framing; defaults are the addresses of IRS_tranceiver.py:271."""
    pl = np.frombuffer(bytes(payload), np.uint8)
    o = np.empty(pl.size + 28, np.uint8)
    n = lib().wifi_b200_mac_frame(_p(pl) if pl.size else None, pl.size, seq, bytes(src), bytes(dst), bytes(bss), _p(o))
    if n < 0:
        raise WifiB200Error(n, lib().wifi_b200_strerror(n).decode())
    return o[:n].tobytes()


def n_sym(enc, psdu_len):
    return lib().wifi_b200_n_sym(enc, psdu_len)


def frame_samples(enc, psdu_len):
    return lib().wifi_b200_frame_samples(enc, psdu_len)


def chan_seg(in_off=0, in_len=0, out_off=0, n=0, n0=0, gain=1.0, cfo=0.0, phase0=0.0, noise_sigma=0.0, taps=((0, 1.0),),
             seed=0, stream=0):
    s = np.zeros(1, CHANSEG_DTYPE)
    s["in_off"], s["in_len"], s["out_off"], s["n"], s["n0"] = in_off, in_len, out_off, n, n0
    s["gain"], s["cfo"], s["phase0"], s["noise_sigma"] = gain, cfo, phase0, noise_sigma
    s["n_taps"] = len(taps)
    for i, (d, hh) in enumerate(taps):
        s["delay"][0, i], s["tap_re"][0, i], s["tap_im"][0, i] = d, np.float32(complex(hh).real), np.float32(complex(hh).imag)
    s["seed"], s["stream"] = seed, stream
    return s


def fading(taps=((0, 1.0),), n_sin=8, k_factor=0.0, doppler=0.0, los_doppler=0.0, t0=0, seed=0, stream=0):
    """One wifi_b200_fading record: taps = ((delay, power), ...) with power = E|h_t|^2; doppler and los_doppler in
    cycles/sample; the realisation is (seed, stream), placed in time by t0."""
    f = np.zeros(1, FADING_DTYPE)
    f["n_taps"], f["n_sin"] = len(taps), n_sin
    for i, (d, p) in enumerate(taps):
        f["delay"][0, i], f["power"][0, i] = d, p
    f["k_factor"], f["doppler"], f["los_doppler"] = k_factor, doppler, los_doppler
    f["t0"], f["seed"], f["stream"] = t0, seed, stream
    return f


_fading = fading     # Handle.channel's keyword of the same name hides it there


class RxResult:
    """All sync_short triggers of one rx call plus the decoded PSDU store."""

    def __init__(self, frames, store):
        self.frames, self.store = frames, store

    def psdu(self, i):
        f = self.frames[i]
        if f["psdu_off"] < 0:
            return None
        return self.store[f["psdu_off"]:f["psdu_off"] + f["length"]].tobytes()

    def pdus(self):
        """What mac_out carries: PSDU without FCS for every CRC-ok frame, in frame-table order."""
        return [self.psdu(i)[:-4] for i in range(len(self.frames)) if self.frames[i]["crc_ok"]]


class Handle:
    def __init__(self, bandwidth=10e6, frequency=5.89e9, sensitivity=0.56, chan_est=0, encoding=0, min_plateau=2,
                 device=0, want_carrier=False, max_samples=1 << 22, max_frames=0, soft_decision=False):
        self._L = lib()
        cfg = Cfg(bandwidth, frequency, sensitivity, int(chan_est), int(encoding), min_plateau, device, int(want_carrier), int(soft_decision),
                  int(max_samples), int(max_frames))
        h = C.c_void_p()
        rc = self._L.wifi_b200_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise WifiB200Error(rc, self._L.wifi_b200_strerror(rc).decode())
        self._h = h
        self.max_frames = int(max_frames) if max_frames else int(max_samples) // 1000 + 64
        # test hook: WIFI_B200_VITERBI_FORM=1|2|3 pins the Viterbi kernel form of every handle (the three forms are one decoder:
        # the whole GPU suite must pass under each)
        if os.environ.get("WIFI_B200_VITERBI_FORM"):
            self.set_param(P_VITERBI_FORM, int(os.environ["WIFI_B200_VITERBI_FORM"]))

    def close(self):
        if getattr(self, "_h", None):
            self._L.wifi_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc < 0:
            raise WifiB200Error(rc, self._L.wifi_b200_last_error(self._h).decode() or self._L.wifi_b200_strerror(rc).decode())
        return rc

    def set_param(self, pid, value):
        self._ck(self._L.wifi_b200_set_param(self._h, pid, float(value)))

    def get_param(self, pid):
        return self._L.wifi_b200_get_param(self._h, pid)

    @property
    def stream(self):
        return self._L.wifi_b200_stream(self._h)

    # ---- TX ----
    def _tx_args(self, psdus, enc, seed):
        n = len(psdus)
        blob = np.frombuffer(b"".join(psdus), np.uint8) if n else np.zeros(0, np.uint8)
        lens = np.array([len(p) for p in psdus], np.uint32)
        offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint32) if n else np.zeros(0, np.uint32)
        e = None if enc is None else np.broadcast_to(np.asarray(enc, np.uint8), (n,)).copy()
        s = None if seed is None else np.broadcast_to(np.asarray(seed, np.uint8), (n,)).copy()
        return n, blob, offs, lens, e, s

    def tx(self, psdus, enc=None, seed=None):
        """mac_in -> samp_out: list of PSDUs (bytes, FCS included) -> (iq complex64, burst offsets)."""
        n, blob, offs, lens, e, s = self._tx_args(psdus, enc, seed)
        encs = e if e is not None else np.full(n, int(self.get_param(P_ENCODING)), np.uint8)
        for ln in lens:
            if ln > 1528:
                raise WifiB200Error(E_TOO_LARGE, "PSDU too large")
        cap = int(sum(frame_samples(int(encs[i]), int(lens[i])) for i in range(n)))
        iq = np.empty(cap, np.complex64)
        boff = np.zeros(n + 1, np.uint64)
        tot = self._ck(self._L.wifi_b200_tx(self._h, _p(blob), _p(offs), _p(lens), _p(e), _p(s), n, _p(iq), cap, _p(boff)))
        return iq[:tot], boff

    def tx_dev(self, psdus, out_ptr, cap_samples, enc=None, seed=None):
        n, blob, offs, lens, e, s = self._tx_args(psdus, enc, seed)
        boff = np.zeros(n + 1, np.uint64)
        tot = self._ck(self._L.wifi_b200_tx_dev(self._h, _p(blob), _p(offs), _p(lens), _p(e), _p(s), n, C.c_void_p(out_ptr), cap_samples, _p(boff)))
        return tot, boff

    def tx_symbols(self):
        buf = np.empty(self.max_frames * 511 * 48 if self.max_frames < 64 else 64 * 511 * 48, np.uint8)
        n = self._ck(self._L.wifi_b200_tx_symbols(self._h, _p(buf), buf.size))
        return buf[:n].copy()

    def channel_dev(self, in_ptr, out_ptr, segs):
        segs = np.ascontiguousarray(segs, CHANSEG_DTYPE)
        self._ck(self._L.wifi_b200_channel_dev(self._h, C.c_void_p(in_ptr), C.c_void_p(out_ptr), _p(segs), segs.size))

    def channel_fading_dev(self, in_ptr, out_ptr, segs, fades):
        """Fading channel on device buffers: one FADING_DTYPE record per CHANSEG_DTYPE segment (whose n_taps is 0)."""
        segs = np.ascontiguousarray(segs, CHANSEG_DTYPE)
        fades = np.ascontiguousarray(fades, FADING_DTYPE)
        if fades.size != segs.size:
            raise ValueError("one fading record per segment")
        self._ck(self._L.wifi_b200_channel_fading_dev(self._h, C.c_void_p(in_ptr), C.c_void_p(out_ptr), _p(segs), _p(fades), segs.size))

    def channel(self, x, n_out=None, fading=None, **kw):
        """One-segment convenience form of the test channel on host arrays (keywords as chan_seg()).  fading: None for the
        fixed taps, or a FADING_DTYPE record / a dict of fading() keywords for time-varying taps (then `taps` is not given)."""
        a = np.ascontiguousarray(x, np.complex64)
        n_out = a.size if n_out is None else int(n_out)
        out = np.empty(n_out, np.complex64)
        if fading is None:
            seg = chan_seg(in_len=a.size, n=n_out, **kw)
            self._ck(self._L.wifi_b200_channel(self._h, _p(a), a.size, _p(out), n_out, _p(seg), 1))
            return out
        seg = chan_seg(in_len=a.size, n=n_out, taps=(), **kw)
        f = np.ascontiguousarray(fading if isinstance(fading, np.ndarray) else _fading(**fading), FADING_DTYPE)
        self._ck(self._L.wifi_b200_channel_fading(self._h, _p(a), a.size, _p(out), n_out, _p(seg), _p(f), 1))
        return out

    # ---- RX ----
    def rx_batch(self, iq, link_off=None, final=True, fetch=True):
        a = np.ascontiguousarray(iq, np.complex64)
        lo = np.array([0, a.size], np.uint64) if link_off is None else np.ascontiguousarray(link_off, np.uint64)
        self._ck(self._L.wifi_b200_rx_batch(self._h, _p(a), _p(lo), lo.size - 1, int(final)))
        return self.results() if fetch else None

    def rx_batch_sc16(self, iq16, scale, link_off=None, final=True, fetch=True):
        """Wire-format capture: interleaved int16 I/Q (2 values per sample); x = float32(i16) * float32(scale) on the GPU."""
        a = np.ascontiguousarray(iq16, np.int16).reshape(-1)
        lo = np.array([0, a.size // 2], np.uint64) if link_off is None else np.ascontiguousarray(link_off, np.uint64)
        self._ck(self._L.wifi_b200_rx_batch_sc16(self._h, _p(a), C.c_float(scale), _p(lo), lo.size - 1, int(final)))
        return self.results() if fetch else None

    def rx_batch_dev(self, iq_ptr, link_off, final=True, fetch=False):
        lo = np.ascontiguousarray(link_off, np.uint64)
        self._ck(self._L.wifi_b200_rx_batch_dev(self._h, C.c_void_p(iq_ptr), _p(lo), lo.size - 1, int(final)))
        return self.results() if fetch else None

    def rx_batch_dev_state(self, iq_ptr, link_off, state, final=True, fetch=False):
        """Resumed streams: `state` is a LINK_STATE_DTYPE array (min_pos, fo_carry, hist) with one entry per link."""
        lo = np.ascontiguousarray(link_off, np.uint64)
        st = np.ascontiguousarray(state, LINK_STATE_DTYPE)
        assert st.size == lo.size - 1
        self._ck(self._L.wifi_b200_rx_batch_dev_state(self._h, C.c_void_p(iq_ptr), _p(lo), lo.size - 1, int(final), _p(st)))
        return self.results() if fetch else None

    def counts(self):
        v = [C.c_int64() for _ in range(4)]
        self._ck(self._L.wifi_b200_rx_counts(self._h, *[C.byref(x) for x in v]))
        return dict(zip(("n_frames", "n_rows", "n_pdus", "psdu_store_bytes"), [x.value for x in v]))

    def results(self):
        c = self.counts()
        frames = np.zeros(c["n_frames"], FRAME_DTYPE)
        store = np.zeros(c["psdu_store_bytes"], np.uint8)
        if c["n_frames"]:
            self._ck(self._L.wifi_b200_rx_frames(self._h, _p(frames), frames.size))
        if c["psdu_store_bytes"]:
            self._ck(self._L.wifi_b200_rx_psdus(self._h, _p(store), store.size))
        return RxResult(frames, store)

    def frames(self, reuse=False):
        """The frame table of the last rx call alone (96 bytes per trigger; the PSDU store stays on the device).
        reuse=True returns a view of a buffer the wrapper keeps (no fresh pages to fault in for a large table): valid until
        the next frames(reuse=True)."""
        n = self.counts()["n_frames"]
        if reuse:
            if getattr(self, "_frames_buf", None) is None or self._frames_buf.size < n:
                self._frames_buf = np.empty(max(n, 1024), FRAME_DTYPE)
            frames = self._frames_buf[:n]
        else:
            frames = np.zeros(n, FRAME_DTYPE)
        if n:
            self._ck(self._L.wifi_b200_rx_frames(self._h, _p(frames), n))
        return frames

    def rows(self, carrier=False):
        c = self.counts()
        rows = np.zeros((c["n_rows"], 48), np.uint8)
        car = np.zeros((c["n_rows"], 48), np.complex64) if carrier else None
        self._ck(self._L.wifi_b200_rx_rows(self._h, _p(rows), _p(car), c["n_rows"]))
        return (rows, car) if carrier else rows

    def soft_rows(self):
        c = self.counts()
        s = np.zeros((c["n_rows"], 288), np.int8)
        self._ck(self._L.wifi_b200_rx_soft(self._h, _p(s), c["n_rows"]))
        return s

    def flags(self, link, n_samples):
        w = np.zeros((n_samples + 31) // 32, np.uint32)
        self._ck(self._L.wifi_b200_rx_flags(self._h, link, _p(w), w.size))
        return np.unpackbits(w.view(np.uint8), bitorder="little")[:n_samples].astype(bool)

    def rx_push(self, iq, flush=False):
        a = np.ascontiguousarray(iq, np.complex64)
        self._ck(self._L.wifi_b200_rx_push(self._h, _p(a) if a.size else None, a.size, int(flush)))

    def rx_push_links(self, chunks, flush=False):
        """chunks: one array of new complex samples per stream (empty arrays allowed)."""
        arrs = [np.ascontiguousarray(c, np.complex64).reshape(-1) for c in chunks]
        off = np.zeros(len(arrs) + 1, np.uint64)
        off[1:] = np.cumsum([a.size for a in arrs])
        blob = np.concatenate(arrs) if arrs and off[-1] else np.zeros(0, np.complex64)
        self._ck(self._L.wifi_b200_rx_push_links(self._h, _p(blob) if blob.size else None, _p(off), len(arrs), int(flush)))

    def rx_push_links_blob(self, blob, link_off, flush=False):
        """Zero-copy form: `blob` holds every link's new samples back to back (complex64, ideally pinned memory),
        link l = blob[link_off[l]:link_off[l+1]]."""
        a = blob if (isinstance(blob, np.ndarray) and blob.dtype == np.complex64 and blob.flags.c_contiguous) else np.ascontiguousarray(blob, np.complex64)
        off = np.ascontiguousarray(link_off, np.uint64)
        self._ck(self._L.wifi_b200_rx_push_links(self._h, _p(a) if a.size else None, _p(off), off.size - 1, int(flush)))

    def rx_push_links_async(self, blob, link_off, flush=False):
        """Queues the copy of this push and returns; `blob` (page-locked complex64) must stay untouched until the
        rx_push_wait() that completes it.  At most three pushes may be pending."""
        assert isinstance(blob, np.ndarray) and blob.dtype == np.complex64 and blob.flags.c_contiguous
        off = np.ascontiguousarray(link_off, np.uint64)
        self._ck(self._L.wifi_b200_rx_push_links_async(self._h, _p(blob) if blob.size else None, _p(off), off.size - 1, int(flush)))

    def rx_push_links_sc16_async(self, blob16, scale, link_off, flush=False):
        """The asynchronous push in the wire format: `blob16` is page-locked int16, I/Q interleaved (2 values per sample);
        link_off counts complex samples.  x = float32(i16) * float32(scale) on the GPU, as rx_batch_sc16."""
        assert isinstance(blob16, np.ndarray) and blob16.dtype == np.int16 and blob16.flags.c_contiguous
        off = np.ascontiguousarray(link_off, np.uint64)
        self._ck(self._L.wifi_b200_rx_push_links_sc16_async(self._h, _p(blob16) if blob16.size else None, C.c_float(scale), _p(off), off.size - 1, int(flush)))

    def rx_push_wait(self):
        """Completes the oldest pending asynchronous push (copy done, pipeline run); True if there was one."""
        return self._ck(self._L.wifi_b200_rx_push_wait(self._h)) == 1

    def rx_pop(self, cap=256):
        meta = np.zeros(cap, FRAME_DTYPE)
        buf = np.zeros(cap * 1528, np.uint8)
        n = C.c_int()
        self._ck(self._L.wifi_b200_rx_pop(self._h, _p(meta), cap, _p(buf), buf.size, C.byref(n)))
        out = []
        for i in range(n.value):
            f = meta[i]
            out.append((f.copy(), buf[f["psdu_off"]:f["psdu_off"] + f["length"] - 4].tobytes()))
        return out

    def rx_pop_arrays(self, cap=4096, copy=True):
        """Bulk form of rx_pop for many live links: (frame records, PSDU bytes); record i's PSDU is
        blob[rec["psdu_off"] : rec["psdu_off"] + rec["length"] - 4].  No per-frame Python objects.  copy=True packs up to
        `cap` frames back to back into fresh arrays; copy=False returns views of the library's own (page-locked) result
        buffers -- the frames of ONE pipeline run per call, `cap` ignored, valid until the next call on this handle
        (wifi_b200_rx_pop_view).  Call until no records come back."""
        if not copy:
            pm, pb, nb, n = vp_t(), vp_t(), C.c_size_t(), C.c_int()
            self._ck(self._L.wifi_b200_rx_pop_view(self._h, C.byref(pm), C.byref(pb), C.byref(nb), C.byref(n)))
            if not n.value:
                return np.zeros(0, FRAME_DTYPE), np.zeros(0, np.uint8)
            meta = np.frombuffer((C.c_char * (n.value * FRAME_DTYPE.itemsize)).from_address(pm.value), FRAME_DTYPE)
            blob = np.frombuffer((C.c_char * nb.value).from_address(pb.value), np.uint8) if nb.value else np.zeros(0, np.uint8)
            return meta, blob
        if getattr(self, "_pop_meta", None) is None or self._pop_meta.size < cap:
            self._pop_meta = np.zeros(cap, FRAME_DTYPE)
            self._pop_buf = np.zeros(cap * 1528, np.uint8)
        n = C.c_int()
        self._ck(self._L.wifi_b200_rx_pop(self._h, _p(self._pop_meta), cap, _p(self._pop_buf), self._pop_buf.size, C.byref(n)))
        k = n.value
        used = int(self._pop_meta["psdu_off"][k - 1] + self._pop_meta["length"][k - 1] - 4) if k else 0
        return self._pop_meta[:k].copy(), self._pop_buf[:used].copy()

    def rx_reset(self):
        self._ck(self._L.wifi_b200_rx_reset(self._h))

    def stats(self):
        s = Stats()
        self._ck(self._L.wifi_b200_get_stats(self._h, C.byref(s)))
        d = {k: getattr(s, k) for k, _ in Stats._fields_ if k != "per_mcs_crc_ok"}
        d["per_mcs_crc_ok"] = list(s.per_mcs_crc_ok)
        return d

    def detmath(self, fn, a, b=None, c=None, d=None, o0=None, o1=None):
        """wdm_selftest(fn, ...) of include/wifi_detmath.h evaluated element-wise on the GPU; returns (o0, o1)."""
        a = np.ascontiguousarray(a, np.float32)
        z = np.zeros_like(a)
        b, c, d = [z if v is None else np.ascontiguousarray(v, np.float32) for v in (b, c, d)]
        o0 = np.zeros_like(a) if o0 is None else np.array(o0, np.float32)
        o1 = np.zeros_like(a) if o1 is None else np.array(o1, np.float32)
        self._ck(self._L.wifi_b200_selftest_detmath(self._h, int(fn), _p(a), _p(b), _p(c), _p(d), _p(o0), _p(o1), a.size))
        return o0, o1

    def host_alloc(self, n, dtype=np.complex64):
        """Page-locked host array of n elements, allocated and first touched on the GPU's side of the machine
        (wifi_b200_host_alloc).  Free it with host_free(array) before closing the handle."""
        dt = np.dtype(dtype)
        p = C.c_void_p()
        self._ck(self._L.wifi_b200_host_alloc(self._h, int(n) * dt.itemsize, C.byref(p)))
        buf = (C.c_char * (int(n) * dt.itemsize)).from_address(p.value)
        a = np.frombuffer(buf, dtype=dt)
        self._host_ptrs = getattr(self, "_host_ptrs", {})
        self._host_ptrs[a.ctypes.data] = p
        return a

    def host_free(self, a):
        p = getattr(self, "_host_ptrs", {}).pop(a.ctypes.data, None)
        if p is not None:
            self._ck(self._L.wifi_b200_host_free(self._h, p))

    def alu_peak(self, iters=4096):
        """Measured issue rate of the integer ALU pipe: (warp-instructions per second, milliseconds of the probe)."""
        v, ms = C.c_double(), C.c_double()
        self._ck(self._L.wifi_b200_alu_peak(self._h, int(iters), C.byref(v), C.byref(ms)))
        return v.value, ms.value

    def stage_times(self):
        ms = np.zeros(16, np.float32)
        n = self._ck(self._L.wifi_b200_stage_times(self._h, _p(ms), 16))
        return {self._L.wifi_b200_stage_name(i).decode(): float(ms[i]) for i in range(n)}
