"""Independent float64 numpy model of the 802.11a/g OFDM PHY, written from the formulas of
IEEE 802.11-2012 clause 18 (not from the oracle, not from gr-ieee802-11): used to cross-check
the oracle's TX bit pipeline / waveform and its RX decisions.  It deliberately uses the
standard's own formulation where that differs from upstream's (forward interleaver
permutations 18-17/18-18, Gray tables, numpy FFT, full-traceback Viterbi)."""
import numpy as np

N_BPSC = [1, 1, 2, 2, 4, 4, 6, 6]
N_CBPS = [48, 48, 96, 96, 192, 192, 288, 288]
N_DBPS = [24, 36, 48, 72, 96, 144, 192, 216]
RATE_BITS = ["1101", "1111", "0101", "0111", "1001", "1011", "0001", "0011"]   # R1..R4
PUNCT = [(1, 1), (1, 1, 1, 0, 0, 1), (1, 1), (1, 1, 1, 0, 0, 1), (1, 1), (1, 1, 1, 0, 0, 1), (1, 1, 1, 0), (1, 1, 1, 0, 0, 1)]

LTS = np.array([1, 1, -1, -1, 1, 1, -1, 1, -1, 1, 1, 1, 1, 1, 1, -1, -1, 1, 1, -1, 1, -1, 1, 1, 1, 1, 0,
                1, -1, -1, 1, 1, -1, 1, -1, 1, -1, -1, -1, -1, -1, 1, 1, -1, -1, 1, -1, 1, -1, 1, 1, 1, 1], float)
STS_POS = {-24: 1, -20: -1, -16: 1, -12: -1, -8: -1, -4: 1, 4: -1, 8: -1, 12: 1, 16: 1, 20: 1, 24: 1}
DATA_SC = [k for k in range(-26, 27) if k not in (-21, -7, 0, 7, 21)]


def scrambler_seq(seed, n):
    s = [(seed >> (6 - i)) & 1 for i in range(7)]   # x7..x1
    out = []
    for _ in range(n):
        fb = s[0] ^ s[3]                            # x7 xor x4
        out.append(fb)
        s = s[1:] + [fb]
    return np.array(out, np.uint8)


PILOT_POLARITY = 1 - 2 * scrambler_seq(0x7f, 127).astype(int)


def conv_encode(bits):
    g0, g1 = 0o133, 0o171
    reg = 0
    out = []
    for b in bits:
        reg = ((reg << 1) | int(b)) & 0x7f          # newest bit at LSB
        # taps counted from the newest bit: g = 1 + D^2 + D^3 + D^5 + D^6 etc.
        a = sum(((reg >> d) & 1) for d in range(7) if (g0 >> (6 - d)) & 1) & 1
        c = sum(((reg >> d) & 1) for d in range(7) if (g1 >> (6 - d)) & 1) & 1
        out += [a, c]
    return np.array(out, np.uint8)


def puncture(coded, enc):
    pat = np.array(PUNCT[enc], bool)
    keep = np.resize(pat, coded.size)
    return coded[keep]


def interleave_perm(enc):
    """Standard 18-17 / 18-18: bit k of the encoder output goes to position j."""
    n, s = N_CBPS[enc], max(N_BPSC[enc] // 2, 1)
    k = np.arange(n)
    i = (n // 16) * (k % 16) + k // 16
    j = s * (i // s) + (i + n - (16 * i) // n) % s
    return j


def gray_axis(bits):
    table = {1: {(0,): -1, (1,): 1},
             2: {(0, 0): -3, (0, 1): -1, (1, 1): 1, (1, 0): 3},
             3: {(0, 0, 0): -7, (0, 0, 1): -5, (0, 1, 1): -3, (0, 1, 0): -1, (1, 1, 0): 1, (1, 1, 1): 3, (1, 0, 1): 5, (1, 0, 0): 7}}
    return table[len(bits)][tuple(int(b) for b in bits)]


def map_bits(bits, enc):
    nb = N_BPSC[enc]
    b = np.asarray(bits).reshape(-1, nb)
    if nb == 1:
        return (2.0 * b[:, 0] - 1).astype(complex)
    h = nb // 2
    norm = {1: np.sqrt(2), 2: np.sqrt(10), 3: np.sqrt(42)}[h]
    return np.array([(gray_axis(r[:h]) + 1j * gray_axis(r[h:])) / norm for r in b])


def signal_bits(enc, length):
    b = [int(c) for c in RATE_BITS[enc]] + [0] + [(length >> i) & 1 for i in range(12)]
    b.append(sum(b) & 1)
    return np.array(b + [0] * 6, np.uint8)


def data_bits(psdu, enc, seed):
    n_sym = -(-(16 + 8 * len(psdu) + 6) // N_DBPS[enc])
    n_data = n_sym * N_DBPS[enc]
    bits = np.zeros(n_data, np.uint8)
    bits[16:16 + 8 * len(psdu)] = np.unpackbits(np.frombuffer(bytes(psdu), np.uint8), bitorder="little")
    scr = bits ^ scrambler_seq(seed, n_data)
    scr[16 + 8 * len(psdu):16 + 8 * len(psdu) + 6] = 0
    return scr, n_sym


def ofdm_symbol(data48, pilot_pol):
    X = np.zeros(64, complex)                      # index = subcarrier mod 64
    for v, k in zip(data48, DATA_SC):
        X[k % 64] = v
    for k, sgn in zip((-21, -7, 7, 21), (1, 1, 1, -1)):
        X[k % 64] = pilot_pol * sgn
    return X


def time_symbol(X):
    return np.fft.ifft(X) * 64 / np.sqrt(52)


def tx_frame(psdu, enc, seed):
    """Returns (samples, per-symbol carrier indices as the mapper numbers them: bit k = b_k)."""
    scr, n_sym = data_bits(psdu, enc, seed)
    coded = puncture(conv_encode(scr), enc)
    perm = interleave_perm(enc)
    ncb, nb = N_CBPS[enc], N_BPSC[enc]
    syms_f = []
    S = np.zeros(64, complex)
    for k, s in STS_POS.items():
        S[k % 64] = s * np.sqrt(13 / 6) * (1 + 1j)
    L = np.zeros(64, complex)
    for i, k in enumerate(range(-26, 27)):
        L[k % 64] = LTS[i]
    sts_t, lts_t = time_symbol(S), time_symbol(L)
    parts = [np.tile(sts_t, 3)[:160], np.concatenate([lts_t[32:], lts_t, lts_t])]
    sig = np.zeros(48, np.uint8)
    sig[interleave_perm(0)] = conv_encode(signal_bits(enc, len(psdu)))
    t = time_symbol(ofdm_symbol(map_bits(sig, 0), PILOT_POLARITY[0]))
    parts.append(np.concatenate([t[48:], t]))
    idx = np.zeros((n_sym, 48), np.uint8)
    for n in range(n_sym):
        blk = np.zeros(ncb, np.uint8)
        blk[perm] = coded[n * ncb:(n + 1) * ncb]
        idx[n] = (blk.reshape(48, nb) << np.arange(nb)).sum(1)
        t = time_symbol(ofdm_symbol(map_bits(blk, enc), PILOT_POLARITY[(n + 1) % 127]))
        parts.append(np.concatenate([t[48:], t]))
    # time windowing as the GNU Radio cyclic prefixer does it (rolloff 2): symbol boundaries are
    # the average of the incoming symbol's first CP sample and the periodic extension of the previous one
    out = np.concatenate(parts + [np.zeros(1, complex)])
    starts = list(range(0, 80 * (5 + n_sym) + 1, 80))
    # periodic extension of each 80-sample symbol = its sample 16 (x[0] of the 64-point body)
    bodies = np.concatenate(parts).reshape(-1, 80)
    for s_i, st in enumerate(starts):
        prev = bodies[s_i - 1][16] if s_i > 0 else 0.0
        cur = bodies[s_i][0] if s_i < len(bodies) else 0.0
        out[st] = 0.5 * cur + 0.5 * prev
    return out, idx


# ---------------------------------------------------------------- receive side (genie timing)
def viterbi_full(sym):
    """Hard-decision ML decoder, erasures = 2, full traceback from the best end state."""
    n = len(sym) // 2
    nxt = np.zeros((64, 2), int)
    outb = np.zeros((64, 2, 2), int)
    for s in range(64):
        for b in range(2):
            reg = ((s << 1) | b) & 0x7f
            nxt[s, b] = reg & 0x3f
            outb[s, b, 0] = bin(reg & 0o155).count("1") & 1
            outb[s, b, 1] = bin(reg & 0o117).count("1") & 1
    metric = np.zeros(64)
    back = np.zeros((n, 64), np.int8)
    prev_of = [[(s2 >> 1), (s2 >> 1) | 32] for s2 in range(64)]
    for t in range(n):
        r0, r1 = sym[2 * t], sym[2 * t + 1]
        new = np.full(64, -1e9)
        for s2 in range(64):
            b = s2 & 1
            for which, s in enumerate(prev_of[s2]):
                m = metric[s]
                if r0 != 2:
                    m += outb[s, b, 0] == r0
                if r1 != 2:
                    m += outb[s, b, 1] == r1
                if m > new[s2]:
                    new[s2] = m
                    back[t, s2] = which
        metric = new
    s = int(np.argmax(metric))
    bits = np.zeros(n, np.uint8)
    for t in range(n - 1, -1, -1):
        bits[t] = s & 1
        s = prev_of[s][back[t, s]]
    return bits


def rx_frame(samples, frame_start, enc=None):
    """Genie-timed LS receiver: returns (enc, length, psdu bytes or None)."""
    x = np.asarray(samples, complex)
    l1 = np.fft.fft(x[frame_start + 192:frame_start + 256]) * np.sqrt(52) / 64
    l2 = np.fft.fft(x[frame_start + 256:frame_start + 320]) * np.sqrt(52) / 64
    Lf = np.zeros(64)
    for i, k in enumerate(range(-26, 27)):
        Lf[k % 64] = LTS[i]
    used = Lf != 0
    H = np.ones(64, complex)
    H[used] = (l1[used] + l2[used]) / 2 / Lf[used]

    def demod(n_sym_index, enc_):
        st = frame_start + 320 + 80 * n_sym_index + 16
        Y = np.fft.fft(x[st:st + 64]) * np.sqrt(52) / 64 / H
        pil = sum(Y[k % 64] * sgn for k, sgn in zip((-21, -7, 7, 21), (1, 1, 1, -1))) * PILOT_POLARITY[n_sym_index % 127]
        Y = Y * np.exp(-1j * np.angle(pil))
        d = np.array([Y[k % 64] for k in DATA_SC])
        nb = N_BPSC[enc_]
        if nb == 1:
            return (d.real > 0).astype(np.uint8).reshape(48, 1)
        h = nb // 2
        norm = {1: np.sqrt(2), 2: np.sqrt(10), 3: np.sqrt(42)}[h]
        levels = {1: [-1, 1], 2: [-3, -1, 1, 3], 3: [-7, -5, -3, -1, 1, 3, 5, 7]}[h]
        inv = {gray_axis(b): b for b in [tuple((v >> (h - 1 - i)) & 1 for i in range(h)) for v in range(1 << h)]}
        out = np.zeros((48, nb), np.uint8)
        for c in range(48):
            for ax, val in enumerate((d[c].real * norm, d[c].imag * norm)):
                lv = min(levels, key=lambda q: abs(q - val))
                out[c, ax * h:(ax + 1) * h] = inv[lv]
        return out

    sig = demod(0, 0).reshape(-1)
    dec = viterbi_full(sig[interleave_perm(0)])
    rate = "".join(str(b) for b in dec[:4])
    if rate not in RATE_BITS or (dec[:17].sum() & 1) != dec[17]:
        return None, None, None
    enc_ = RATE_BITS.index(rate)
    length = int(sum(int(dec[5 + i]) << i for i in range(12)))
    n_sym = -(-(16 + 8 * length + 6) // N_DBPS[enc_])
    perm = interleave_perm(enc_)
    coded = np.concatenate([demod(1 + n, enc_).reshape(-1)[perm] for n in range(n_sym)])
    pat = np.resize(np.array(PUNCT[enc_], bool), 2 * n_sym * N_DBPS[enc_])
    dep = np.full(pat.size, 2, np.uint8)
    dep[pat] = coded
    bits = viterbi_full(dep)
    seq_state = bits[:7]
    seed = int(sum(int(b) << (6 - i) for i, b in enumerate(seq_state)))
    # the first 7 scrambled SERVICE bits are the scrambler output itself: regenerate the sequence
    for cand in range(1, 128):
        if np.array_equal(scrambler_seq(cand, 7), seq_state):
            seed = cand
            break
    plain = bits ^ scrambler_seq(seed, bits.size)
    return enc_, length, np.packbits(plain[16:16 + 8 * length], bitorder="little").tobytes()


# ---------------------------------------------------------------- receiver stages in float64
# The receive chain of wifi_phy_hier (gr-ieee802-11's sync_short, sync_long and frame_equalizer, as SURVEY.md 8a and
# Appendix A restate them), computed in float64 from the formulas: exact window sums, numpy's FFT, exp() rotations,
# each upstream rotation applied on its own.  Every stage takes its inputs explicitly, so a test can feed it either
# the previous model stage or what the device under test reported.
SS_MIN_GAP, SS_MAX_SAMPLES, SYNC_LENGTH = 480, 540 * 80, 320
LEVEL = {1: np.sqrt(0.5), 2: np.sqrt(0.1), 3: np.sqrt(1 / 42)}       # per-axis unit of QPSK / 16-QAM / 64-QAM
USED = np.array([i for i in range(6, 59) if i != 32])                  # the 52 used carriers, shifted order (index = k + 32)
PILOT_IDX = np.array([11, 25, 39, 53])
DATA_IDX = np.array([i for i in USED if i not in PILOT_IDX])


def lts_shifted():
    L = np.zeros(64)
    L[6:59] = LTS
    return L


def long_taps():
    """sync_long's matched filter LONG[63 - n] = conj(lts_t[n]) rounded to 4 decimals, lts_t the LTS time symbol."""
    L = np.zeros(64, complex)
    for i, k in enumerate(range(-26, 27)):
        L[k % 64] = LTS[i]
    lt = time_symbol(L)
    return np.round(np.conj(lt[::-1]).real, 4) + 1j * np.round(np.conj(lt[::-1]).imag, 4)


def constellation(enc):
    """Point of every carrier index v (bit k of v = coded bit b_k, b_0 first on air)."""
    nb = N_BPSC[enc]
    return map_bits([(v >> k) & 1 for v in range(1 << nb) for k in range(nb)], enc)


def frontend(x, thr=0.56):
    """Exact window sums of the autocorrelation front end; samples before index 0 are zeros.
    a[i] = sum of x[j] conj(x[j-16]) over j = i-47 .. i, p[i] = sum of |x[j]|^2 over j = i-63 .. i.
    Returns (a, p, flags, margin, E): flags = p > 0 and |a| > thr p, margin = ||a| - thr p|, E[i] = sum of |x|^2 over the
    last 128 samples (the scale of the margin)."""
    from numpy.lib.stride_tricks import sliding_window_view as win
    x = np.asarray(x, np.complex128)
    n = x.size
    xz = np.concatenate([np.zeros(127, complex), x])
    pw = xz.real ** 2 + xz.imag ** 2
    prod = np.zeros(xz.size, complex)
    prod[16:] = xz[16:] * np.conj(xz[:-16])
    a = win(prod[80:], 48).sum(axis=1)[:n]
    p = win(pw[64:], 64).sum(axis=1)[:n]
    cs = np.concatenate([[0.0], np.cumsum(pw)])
    E = np.maximum(cs[128:128 + n] - cs[:n], 0.0)
    flags = (p > 0) & (np.abs(a) > thr * p)
    return a, p, flags, np.abs(np.abs(a) - thr * p), E


def sync_short(flags, a, n=None, min_plateau=2, min_pos=0):
    """sync_short's SEARCH / COPY state machine on a flag array (the port of its per-sample loop, stepped from flag to
    flag: an unflagged sample only resets the plateau counter).  Returns (triggers, burst_len, freq_short) with
    freq_short = angle(a[t]) / 16."""
    n = len(flags) if n is None else n
    trig = []
    search, plateau, c0, last = True, 0, 0, -2
    for i in np.flatnonzero(flags):
        i = int(i)
        if i != last + 1:
            plateau = 0
        last = i
        if not search and i >= c0 + SS_MAX_SAMPLES:
            search = True                     # the copy ended on sample c0 + MAX_SAMPLES - 1
        if search:
            if plateau < min_plateau:
                plateau += 1
                continue
            if i < min_pos:
                continue
            search, plateau, c0 = False, 0, i
            trig.append(i)                    # falls through to COPY with the same sample
        if plateau < min_plateau:
            plateau += 1
        elif i - c0 > SS_MIN_GAP:
            trig.append(i)
            c0, plateau = i, 1
    t = np.array(trig, np.int64)
    nxt = np.concatenate([t[1:], [n]])
    blen = np.minimum(np.minimum(nxt, t + SS_MAX_SAMPLES), n) - t
    fs = np.angle(a[t]) / 16 if t.size else np.zeros(0)
    return t, blen, fs


def _burst(x, t, j, hist=0):
    src = t + np.asarray(j) - 16
    ok = src >= -hist
    out = np.zeros(src.shape, complex)
    out[ok] = np.asarray(x, np.complex128)[src[ok] + hist]
    return out


def sync_long(x, t, burst_len, freq_short, fo_carry=0.0, hist=0, taps=None):
    """The LTS matched filter over 320 lags of sync_short's derotated burst, the top four |corr|^2 (stable order) and the
    63/64/65 pair rule preferring 64.  x[hist] is the stream's sample 0.  Returns a dict: frame_start, found, freq_long
    (fo_carry where no pair is found: sync_long keeps its offset across bursts), tie (relative gap between the fourth and
    fifth largest magnitudes, and between equal-rank neighbours: a tie below 1e-6 makes the ranking fragile)."""
    r = {"frame_start": SYNC_LENGTH, "found": 0, "freq_long": float(fo_carry), "tie": np.inf}
    if burst_len < SYNC_LENGTH + 63:
        return r
    taps = long_taps() if taps is None else taps
    j = np.arange(SYNC_LENGTH + 63)
    b = _burst(x, t, j, hist) * np.exp(-1j * float(freq_short) * j)
    from numpy.lib.stride_tricks import sliding_window_view as win
    corr = win(b, 64)[:SYNC_LENGTH] @ taps[::-1]          # corr[i] = sum_m LONG[63 - m] b[i + m]
    mag = np.abs(corr) ** 2
    order = np.argsort(-mag, kind="stable")
    top = order[:4]
    srt = mag[order[:5]]
    r["tie"] = float(np.min(np.abs(np.diff(srt)) / srt[0])) if srt[0] > 0 else 0.0
    done = False
    for i in range(3):
        if done:
            break
        for k in range(i + 1, 4):
            lo, hi = min(top[i], top[k]), max(top[i], top[k])
            d = hi - lo
            if d in (63, 64, 65):
                r.update(frame_start=int(lo), found=int(d), freq_long=float(np.angle(corr[lo] * np.conj(corr[hi])) / d))
                if d == 64:
                    done = True
                    break
    return r


def symbols(x, t, burst_len, freq_short, freq_long, frame_start, n_syms, hist=0, final=True, last=False):
    """sync_long's COPY output cut into 64-sample symbols (CP dropped): LTS1, LTS2, SIGNAL, data ...  Each sample gets
    sync_short's exp(-j fs j) and sync_long's exp(+j fl j), j its burst position; a partial symbol is zero-padded."""
    avail = burst_len - SYNC_LENGTH
    R = avail - frame_start
    E = 0 if R <= 0 else (R if R <= 128 else 128 + 64 * ((R - 128) // 80) + max(0, ((R - 128) % 80) - 16))
    k = np.arange(n_syms * 64)
    nn, m = k // 64, k % 64
    j = frame_start + np.where(nn < 2, 64 * nn + m, 128 + 80 * (nn - 2) + 16 + m)
    s = _burst(x, t, j, hist) * np.exp(-1j * float(freq_short) * j) * np.exp(1j * float(freq_long) * j)
    s[k >= E] = 0
    return s.reshape(n_syms, 64)


def decide_nearest(enc, z):
    """Index of the nearest constellation point of every z, and its distance to the closest decision boundary."""
    z = np.asarray(z, complex)
    pts = constellation(enc)
    idx = np.argmin(np.abs(z[..., None] - pts), axis=-1)
    h = N_BPSC[enc] // 2
    if N_BPSC[enc] == 1:
        return idx, np.abs(z.real)
    lv = LEVEL[h]
    bnd = lv * np.arange(-(2 ** h) + 2, 2 ** h - 1, 2)     # midpoints between adjacent levels
    dist = np.minimum(np.abs(z.real[..., None] - bnd).min(-1), np.abs(z.imag[..., None] - bnd).min(-1))
    return idx, dist


def llr(enc, z):
    """Max-log LLR per coded bit in units of the axis level (positive = bit 1), 48 * N_BPSC values per symbol in the
    order of the carrier index bits."""
    nb = N_BPSC[enc]
    if nb == 1:
        return z.real[:, None]
    h = nb // 2
    out = []
    for a in (z.real / LEVEL[h], z.imag / LEVEL[h]):
        m = np.abs(a)
        out.append(a)
        if h == 2:
            out.append(2 - m)
        if h == 3:
            out += [4 - m, 2 - np.abs(m - 4)]
    return np.stack(out, axis=-1)


def equalize(sy, enc, algo, freq_short, freq_long, rows=None, bw=10e6, freq=5.89e9):
    """frame_equalizer on the symbols of one frame (sy: LTS1, LTS2, SIGNAL, data ...): FFT and +-32 shift, the
    sampling-offset ramp 2 pi n 80 (eps0 + d_er)(i - 32) / 64 with eps0 from the frequency offset sync_long tagged,
    the pilot phase beta, the pilot phase-drift term er through the 0.1 IIR, then LS / LMS / COMB / STA.
    rows: the data decisions (carrier indices) the decision-directed updates use, one row per data symbol; None = the
    model's own nearest points.  SIGNAL is decided by the model (BPSK).
    Returns dict: snr (dB, from the LTS pair), points (n_data x 48), w (soft weight per data carrier), soft (16 l w)."""
    n_syms = sy.shape[0]
    pol = PILOT_POLARITY.astype(float)
    lts = lts_shifted()
    eps0 = (float(freq_short) - float(freq_long)) * bw / (2 * np.pi * freq)
    d_er, prev = 0.0, None
    H = np.zeros(64, complex)
    snr, w0 = np.nan, np.ones(64)
    pts, soft = [], []
    ph_i = np.arange(64) - 32
    for nn in range(n_syms):
        cur = np.fft.fft(sy[nn])[(np.arange(64) + 32) & 63]
        cur = cur * np.exp(1j * 2 * np.pi * nn * 80 * (eps0 + d_er) * ph_i / 64)
        if nn < 2:
            pil = cur[PILOT_IDX] * np.array([1, -1, 1, 1])
        else:
            p = pol[(nn - 2) % 127]
            pil = cur[PILOT_IDX] * np.array([p, p, p, -p])
        beta = np.angle(pil.sum())
        er = 0.0
        if nn >= 2:
            er = np.angle(np.sum(pil * np.conj(prev))) * bw / (2 * np.pi * freq * 80)
        prev = pil
        cur = cur * np.exp(-1j * beta)
        if nn >= 2:
            d_er = 0.9 * d_er + 0.1 * er
        e = 0 if nn == 2 else enc
        if algo == 2:                                       # comb: divide by the pilot-interpolated gain first
            if nn < 2:
                cp = cur[PILOT_IDX] * np.array([1, -1, 1, 1])
            else:
                p = pol[(nn - 2) % 127]
                cp = cur[PILOT_IDX] * np.array([p, p, p, -p])
            knots_x = [0, 11, 25, 39, 53, 64]
            knots_y = [cp.mean(), cp[0], cp[1], cp[2], cp[3], cp.mean()]
            G = np.zeros(64, complex)
            for s in range(5):
                x0, x1 = knots_x[s], knots_x[s + 1]
                i = np.arange(x0 + (s > 0), x1 + 1) if s < 4 else np.arange(54, 64)
                G[i] = (knots_y[s] * (x1 - i) + knots_y[s + 1] * (i - x0)) / (x1 - x0)
            cur = cur / G
        if nn == 0:
            H = cur.copy()
            continue
        if nn == 1:
            d, s = H[USED] - cur[USED], H[USED] + cur[USED]
            snr = 10 * np.log10(np.sum(np.abs(s) ** 2) / np.sum(np.abs(d) ** 2) / 2)
            H = H.copy()
            H[USED] = s / (2 * lts[USED])
            w0 = np.abs(H) ** 2 / np.mean(np.abs(H[USED]) ** 2)
            continue
        z = cur[DATA_IDX] / H[DATA_IDX]
        if nn == 2 or rows is None:
            dec = decide_nearest(e, z)[0]
        else:
            dec = np.asarray(rows[nn - 3], int)
        if nn > 2:
            pts.append(z)
            soft.append(16 * llr(e, z) * w0[DATA_IDX][:, None])
        q = cur[DATA_IDX] / constellation(e)[dec]
        if algo == 1:                                       # lms, alpha 0.5
            H[DATA_IDX] = 0.5 * H[DATA_IDX] + 0.5 * q
        elif algo == 3:                                     # sta, alpha 0.5, beta 2
            p = pol[(nn - 2) % 127]
            Hu = np.zeros(64, complex)
            Hu[DATA_IDX] = q
            Hu[PILOT_IDX] = cur[PILOT_IDX] * np.array([p, p, p, -p])
            used = np.zeros(64, bool)
            used[USED] = True
            Hn = H.copy()
            for i in USED:
                k = np.arange(i - 2, i + 3)
                k = k[used[k]]
                Hn[i] = 0.5 * H[i] + 0.5 * Hu[k].mean()
            H = Hn
    nd = len(pts)
    return {"snr": snr, "points": np.array(pts).reshape(nd, 48), "w": w0[DATA_IDX],
            "soft": np.array(soft).reshape(nd, 48 * N_BPSC[enc]) if nd else np.zeros((0, 48 * N_BPSC[enc]))}
