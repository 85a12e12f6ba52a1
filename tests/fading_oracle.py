"""ctypes binding of tests/fading_oracle.cpp, the CPU reference of the fading channel (TEST INFRASTRUCTURE ONLY).

The library is compiled once per process into a temporary directory, with the numerical contract's host flags (those of
oracle/Makefile), and removed at exit; nothing is written into the tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
CXXFLAGS = ["-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-mfma", "-mavx2", "-fno-math-errno", "-Wall", "-shared"]


class FadingCfg(C.Structure):
    """Same layout and meaning as wifi_b200_fading (include/wifi_b200.h)."""
    _fields_ = [("n_taps", C.c_int32), ("n_sin", C.c_int32), ("delay", C.c_int32 * 8), ("power", C.c_float * 8),
                ("k_factor", C.c_float), ("doppler", C.c_float), ("los_doppler", C.c_float), ("reserved", C.c_int32),
                ("t0", C.c_int64), ("seed", C.c_uint64), ("stream", C.c_uint64)]


class SegCfg(C.Structure):
    _fields_ = [("gain", C.c_float), ("cfo", C.c_float), ("phase0", C.c_float), ("noise_sigma", C.c_float),
                ("seed", C.c_uint64), ("stream", C.c_uint64)]


def lib():
    global _LIB
    if _LIB is None:
        d = tempfile.mkdtemp(prefix="fading_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libfading_oracle.so")
        subprocess.check_call([os.environ.get("CXX", "g++")] + CXXFLAGS + ["-o", so, os.path.join(_HERE, "fading_oracle.cpp")])
        _LIB = C.CDLL(so)
        _LIB.fad_channel.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(SegCfg), C.POINTER(FadingCfg)]
    return _LIB


def fading_cfg(taps=((0, 1.0),), n_sin=8, k_factor=0.0, doppler=0.0, los_doppler=0.0, t0=0, seed=0, stream=0):
    """taps = ((delay, power), ...); the rest as wifi_b200_fading."""
    f = FadingCfg()
    f.n_taps, f.n_sin = len(taps), n_sin
    for i, (d, p) in enumerate(taps):
        f.delay[i], f.power[i] = int(d), float(p)
    f.k_factor, f.doppler, f.los_doppler = k_factor, doppler, los_doppler
    f.t0, f.seed, f.stream = t0, seed, stream
    return f


def channel(x, fading, n0=0, gain=1.0, cfo=0.0, phase0=0.0, noise_sigma=0.0, seed=0, stream=0):
    """The oracle's channel() (gain, CFO rotation, Philox AWGN keyed by seed / stream at counter n0 + i) with the fading taps
    `fading`: a FadingCfg, a FADING_DTYPE record, or a dict of fading_cfg keywords."""
    if isinstance(fading, dict):
        f = fading_cfg(**fading)
    elif isinstance(fading, np.ndarray):
        f = FadingCfg.from_buffer_copy(np.ascontiguousarray(fading).tobytes())
    else:
        f = fading
    a = np.ascontiguousarray(x, np.complex64)
    o = np.empty_like(a)
    s = SegCfg(gain, cfo, phase0, noise_sigma, seed, stream)
    if lib().fad_channel(a.ctypes.data, o.ctypes.data, a.size, n0, C.byref(s), C.byref(f)):
        raise ValueError("fading parameters out of range")
    return o
