"""GPU parity tests: libwifi_b200.so (through its C ABI) against the CPU oracle on the same
seeded inputs.  Integer/index/byte results must be identical; fp32 results are identical too
because both sides follow include/wifi_detmath.h (only the double-precision log10 of the SNR
estimate is compared with a tolerance, 1e-9 relative)."""
import os

import numpy as np
import pytest

from util import (adversarial_stream, assert_frames_equal, capture_with_collection_over_many_bursts, gpu_segment_decoder, make_capture,
                  make_psdu)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def H(W):
    h = W.Handle(max_samples=1 << 21, max_frames=4096, want_carrier=True)
    yield h
    h.close()


@pytest.mark.parametrize("enc", range(8))
def test_tx_bit_exact(H, O, W, enc):
    rng = np.random.default_rng(enc)
    lens = [28, 100, 333, 1528, int(rng.integers(29, 1528))]
    psdus = [make_psdu(O, rng, n, seq=i) for i, n in enumerate(lens)]
    seeds = [1, 127, 93, 45, 7]
    iq, off = H.tx(psdus, enc=enc, seed=seeds)
    syms = H.tx_symbols()
    spos = 0
    for i, p in enumerate(psdus):
        ref = O.tx_frame(p, enc, seeds[i])
        got = iq[int(off[i]):int(off[i + 1])]
        assert got.size == ref.size == W.wifi_b200.frame_samples(enc, len(p))
        assert np.array_equal(got, ref), (enc, i, np.abs(got - ref).max())
        rs = O.tx_symbols(p, enc, seeds[i]).reshape(-1)
        assert np.array_equal(syms[spos:spos + rs.size], rs)
        spos += rs.size


def test_tx_running_seed_and_errors(H, O, W):
    h = W.Handle(encoding=3, max_samples=1 << 16)
    rng = np.random.default_rng(0)
    p = make_psdu(O, rng, 64)
    for i in range(130):   # [UPSTREAM] mapper: seed 1,2,..,127,1,..
        iq, _ = h.tx([p])
        if i in (0, 1, 126, 127, 129):
            assert np.array_equal(iq, O.tx_frame(p, 3, 1 + i % 127)), i
    with pytest.raises(W.WifiB200Error) as e:
        h.tx([bytes(1529)])
    assert e.value.code == W.wifi_b200.E_TOO_LARGE
    h.close()


@pytest.mark.parametrize("algo", range(4))
def test_rx_all_mcs(H, O, W, algo):
    rng = np.random.default_rng(100 + algo)
    specs = [(e, int(rng.integers(40, 700))) for e in range(8)] + [(7, 1528), (0, 200), (4, 1500)]
    y, psdus = make_capture(O, rng, specs, snr_db=32, cfo=0.011, seed=algo)
    H.set_param(W.wifi_b200.P_CHAN_EST, algo)
    res = H.rx_batch(y)
    ref = O.rx(y, algo=algo)
    assert_frames_equal(res, ref)
    rows, car = H.rows(carrier=True)
    for i in range(len(ref.frames)):
        f = ref.frames[i]
        g = res.frames[i]
        a = rows[g["row_off"]:g["row_off"] + g["n_rows"]]
        b = ref.rows[f["row_off"]:f["row_off"] + f["n_rows"]]
        assert np.array_equal(a, b), ("rows", i)
        ca = car[g["row_off"]:g["row_off"] + g["n_rows"]]
        cb = ref.carrier[f["row_off"]:f["row_off"] + f["n_rows"]]
        assert np.array_equal(ca, cb), ("carrier", i, np.abs(ca - cb).max())
    assert res.pdus() == ref.pdus()
    assert sum(ref.frames["crc_ok"]) >= 9   # the capture is decodable


@pytest.mark.parametrize("form", [1, 2, 3])
def test_viterbi_kernel_forms_are_one_decoder(O, W, form):
    """One trellis per warp, per four lanes and per thread (WIFI_P_VITERBI_FORM): every MCS and traceback depth, lengths that
    differ inside a warp, frames that fail their FCS at a marginal SNR, several links -- the same bytes as the oracle's decoder."""
    rng = np.random.default_rng(4242)
    caps = []
    for l in range(3):
        specs = [(int(rng.integers(0, 8)), int(rng.integers(20, 1529))) for _ in range(14)] + [(l, 1), (7 - l, 1528)]
        caps.append(make_capture(O, rng, specs, snr_db=[30, 19, 13][l], cfo=float(rng.uniform(-0.01, 0.01)), seed=300 + l, gap=600)[0])
    off = np.concatenate([[0], np.cumsum([c.size for c in caps])]).astype(np.uint64)
    h = W.Handle(max_samples=1 << 22, max_frames=512)
    try:
        h.set_param(W.wifi_b200.P_VITERBI_FORM, form)
        assert h.get_param(W.wifi_b200.P_VITERBI_FORM) == form
        res = h.rx_batch(np.concatenate(caps), link_off=off)
        k = 0
        n_bad = 0
        for l, c in enumerate(caps):
            ref = O.rx(c, algo=0, want_carrier=False)
            for i in range(len(ref.frames)):
                g = res.frames[k + i]
                assert int(g["link"]) == l and int(g["trigger"]) == int(ref.frames[i]["trigger"])
                assert int(g["decoded"]) == int(ref.frames[i]["decoded"]) and int(g["crc_ok"]) == int(ref.frames[i]["crc_ok"]), (l, i)
                if ref.frames[i]["decoded"]:
                    assert res.psdu(k + i) == ref.psdu(i), (l, i)
                    n_bad += not ref.frames[i]["crc_ok"]
            k += len(ref.frames)
        assert k == len(res.frames) >= 40 and n_bad >= 3
        with pytest.raises(W.WifiB200Error):
            h.set_param(W.wifi_b200.P_VITERBI_FORM, 4)
    finally:
        h.close()


def test_flags_match_frontend(H, O, W):
    rng = np.random.default_rng(5)
    y, _ = make_capture(O, rng, [(2, 100), (5, 300)], snr_db=15, cfo=-0.02)
    H.rx_batch(y)
    ref = O.flags(y, 0.56)
    assert np.array_equal(H.flags(0, y.size), ref)
    # the contract compares squares; sync_short's literal c > threshold differs from it only where c sits within a
    # rounding of the threshold
    _, _, c = O.frontend(y)
    lit = c.astype(np.float64) > 0.56
    assert np.all(np.abs(c[lit != ref] - 0.56) < 1e-6) and (lit != ref).mean() < 1e-4


@pytest.mark.parametrize("snr_db", [3, 8, 14, 20])
def test_rx_low_snr_marginal_frames(H, O, W, snr_db):
    """Marginal and failing frames must fail the same way (identical frame table)."""
    rng = np.random.default_rng(snr_db)
    specs = [(int(rng.integers(0, 8)), int(rng.integers(30, 400))) for _ in range(24)]
    taps = ((0, 1.0), (1, 0.4 * np.exp(1j * 1.0)), (3, 0.2 * np.exp(-2j)))
    y, _ = make_capture(O, rng, specs, snr_db=snr_db, cfo=0.004, taps=taps, seed=snr_db, gap=700)
    H.set_param(W.wifi_b200.P_CHAN_EST, 1)
    res = H.rx_batch(y)
    ref = O.rx(y, algo=1)
    assert_frames_equal(res, ref)


def test_rx_noise_only_and_empty(H, O, W):
    rng = np.random.default_rng(9)
    y = (rng.standard_normal(20000) + 1j * rng.standard_normal(20000)).astype(np.complex64)
    res = H.rx_batch(y)
    ref = O.rx(y)
    assert_frames_equal(res, ref)
    res = H.rx_batch(np.zeros(0, np.complex64))
    assert len(res.frames) == 0


def test_rx_truncated_and_back_to_back(H, O, W):
    """Frames closer than sync_long's 320-sample delay truncate their predecessor; a capture
    that ends mid-frame leaves an incomplete burst."""
    rng = np.random.default_rng(11)
    y, _ = make_capture(O, rng, [(3, 120), (3, 120), (6, 500), (0, 60)], snr_db=28, gap=150, seed=3)
    y = y[:-700]
    for algo in (0, 3):
        H.set_param(W.wifi_b200.P_CHAN_EST, algo)
        assert_frames_equal(H.rx_batch(y), O.rx(y, algo=algo))
    for final in (True, False):
        assert_frames_equal(H.rx_batch(y, final=final), O.rx(y, algo=3, final=final))


def test_short_final_burst_carries_the_frequency_offset(H, O, W):
    """A capture that ends less than 320 + 63 samples behind its last trigger: sync_long never completes for that burst,
    and its record carries the frequency offset of the last burst that matched (found by the time-sharding fuzz)."""
    rng = np.random.default_rng(77)
    y, _ = make_capture(O, rng, [(3, 120), (5, 200), (2, 90)], snr_db=28, cfo=0.006, gap=400, seed=9)
    ref_all = O.rx(y, algo=0)
    t_last = int(ref_all.frames["trigger"][-1])
    H.set_param(W.wifi_b200.P_CHAN_EST, 0)
    for cut in (t_last + 60, t_last + 300, t_last + 382, t_last + 383):
        ref = O.rx(y[:cut], algo=0)
        assert ref.frames["burst_len"][-1] == cut - t_last and ref.frames["freq_long"][-2] != 0
        assert_frames_equal(H.rx_batch(y[:cut]), ref)
        assert_frames_equal(H.rx_batch(y[:cut], final=False), O.rx(y[:cut], algo=0, final=False))


def test_rx_multi_link(H, O, W):
    rng = np.random.default_rng(21)
    links, offs = [], [0]
    for l in range(5):
        y, _ = make_capture(O, rng, [(int(rng.integers(0, 8)), int(rng.integers(40, 300))) for _ in range(3)],
                            snr_db=25, cfo=float(rng.uniform(-0.01, 0.01)), seed=l, lead=int(rng.integers(20, 300)))
        links.append(y)
        offs.append(offs[-1] + y.size)
    x = np.concatenate(links)
    H.set_param(W.wifi_b200.P_CHAN_EST, 0)
    res = H.rx_batch(x, np.array(offs, np.uint64))
    ref = O.rx_links(x, offs[:-1], np.diff(offs), algo=0)
    # the library allocates frame slots per link with an atomic: order by (link, trigger)
    order = np.lexsort((res.frames["trigger"], res.frames["link"]))
    res.frames = res.frames[order]
    assert_frames_equal(res, ref)


def test_rx_streaming_equals_batch(O, W):
    rng = np.random.default_rng(31)
    y, psdus = make_capture(O, rng, [(int(rng.integers(0, 8)), int(rng.integers(40, 600))) for _ in range(12)],
                            snr_db=30, cfo=0.006, seed=4)
    ref = O.rx(y, algo=0)
    h = W.Handle(max_samples=1 << 18)
    got = []
    pos = 0
    while pos < y.size:
        n = int(rng.integers(1, 9000))
        h.rx_push(y[pos:pos + n], flush=(pos + n >= y.size))
        got += h.rx_pop()
        pos += n
    want = [(int(f["trigger"]), ref.psdu(i)[:-4]) for i, f in enumerate(ref.frames) if f["crc_ok"]]
    assert [(int(f["trigger"]), d) for f, d in got] == want
    h.close()


def test_channel_matches_oracle(H, O, W):
    import torch
    rng = np.random.default_rng(41)
    x = (rng.standard_normal(5000) + 1j * rng.standard_normal(5000)).astype(np.complex64)
    taps = ((0, 0.9 + 0.1j), (2, -0.3j), (5, 0.1))
    ref = O.channel(x, n0=1234, gain=0.7, cfo=0.013, phase0=0.5, noise_sigma=0.2, taps=taps, seed=77, stream=3)
    tx = torch.from_numpy(x.view(np.float32)).cuda()
    ty = torch.zeros_like(tx)
    seg = np.zeros(1, W.wifi_b200.CHANSEG_DTYPE)
    seg["in_len"], seg["n"], seg["n0"] = x.size, x.size, 1234
    seg["gain"], seg["cfo"], seg["phase0"], seg["noise_sigma"] = 0.7, 0.013, 0.5, 0.2
    seg["n_taps"] = 3
    for i, (d, hh) in enumerate(taps):
        seg["delay"][0, i], seg["tap_re"][0, i], seg["tap_im"][0, i] = d, np.float32(complex(hh).real), np.float32(complex(hh).imag)
    seg["seed"], seg["stream"] = 77, 3
    H.channel_dev(tx.data_ptr(), ty.data_ptr(), seg)
    got = ty.cpu().numpy().view(np.complex64)
    assert np.array_equal(got, ref), np.abs(got - ref).max()
    assert np.array_equal(H.channel(x, n0=1234, gain=0.7, cfo=0.013, phase0=0.5, noise_sigma=0.2, taps=taps, seed=77, stream=3), got)


def test_full_size_roundtrip_property(O, W):
    """BASELINE config 3 shape (64-QAM 3/4, 1528-byte PSDUs) at a size the oracle does not run:
    encode -> channel -> decode round trip, every PSDU must come back bit-exact."""
    import torch
    n = 2048
    rng = np.random.default_rng(51)
    h = W.Handle(max_samples=n * 6100 + 4096, max_frames=n + 64, chan_est=1, encoding=7)
    psdus = [make_psdu(O, rng, 1528, seq=i) for i in range(n)]
    flen = W.wifi_b200.frame_samples(7, 1528)
    tx = torch.zeros(2 * n * flen, dtype=torch.float32, device="cuda")
    tot, off = h.tx_dev(psdus, tx.data_ptr(), n * flen)
    assert tot == n * flen
    stride = flen + 1100
    cap = torch.zeros(2 * (n * stride + 200), dtype=torch.float32, device="cuda")
    seg = np.zeros(n, W.wifi_b200.CHANSEG_DTYPE)
    seg["in_off"] = off[:-1]
    seg["in_len"] = flen
    seg["out_off"] = 100 + np.arange(n) * stride
    seg["n"] = stride
    seg["n0"] = seg["out_off"]
    seg["gain"], seg["noise_sigma"] = 0.6, 0.6 * 10 ** (-30 / 20)
    seg["cfo"] = rng.uniform(-0.01, 0.01, n)
    seg["n_taps"] = 1
    seg["tap_re"][:, 0] = 1.0
    seg["seed"] = 5
    h.channel_dev(tx.data_ptr(), cap.data_ptr(), seg)
    res = h.rx_batch_dev(cap.data_ptr(), np.array([0, n * stride + 200], np.uint64), fetch=True)
    assert len(res.frames) == n
    sent = {p[:-4] for p in psdus}
    got = res.pdus()
    assert len(got) >= 0.99 * n and all(g in sent for g in got)     # 30 dB: a few genuine channel losses
    # the head of the same capture through the oracle: identical frame table, failures included
    m = 48
    head = cap[:2 * (100 + m * stride)].cpu().numpy().view(np.complex64)
    ref = O.rx(head, algo=1, final=False)
    sub = W.wifi_b200.RxResult(res.frames[:len(ref.frames) - 1], res.store)
    ref.frames = ref.frames[:-1]   # the last burst of the head is cut by the slice
    from util import assert_frames_equal as afe
    afe(sub, ref)
    h.close()


def test_config1_shape_bpsk_1500_byte_psdus(H, O, W):
    """BASELINE configs[0] shape: BPSK 1/2, 1500-byte PSDUs (501 symbols, 40481 samples), AWGN 20 dB."""
    rng = np.random.default_rng(61)
    y, psdus = make_capture(O, rng, [(0, 1500)] * 3, snr_db=20, seed=6)
    H.set_param(W.wifi_b200.P_CHAN_EST, 0)
    res, ref = H.rx_batch(y), O.rx(y, algo=0)
    assert_frames_equal(res, ref)
    assert res.pdus() == [p[:-4] for p in psdus]


def test_config2_shape_16qam_multipath_cfo(H, O, W):
    """BASELINE configs[1] shape at reduced length: 16-QAM 1/2, 1500-byte PSDUs, per-frame CFO,
    3-tap channel h=[1, 0.4e^{j.}, 0, 0.2e^{j.}], 25 dB."""
    rng = np.random.default_rng(62)
    parts = [np.zeros(300, np.complex64)]
    for i in range(10):
        p = make_psdu(O, rng, 1500, seq=i)
        iq = np.concatenate([O.tx_frame(p, 4, 1 + i), np.zeros(1100, np.complex64)])
        taps = np.array([1.0, 0.4 * np.exp(1j * rng.uniform(0, 6.28)), 0.2 * np.exp(1j * rng.uniform(0, 6.28))])
        taps /= np.linalg.norm(taps)
        parts.append(O.channel(iq, n0=i * 20000, gain=0.6, cfo=float(rng.uniform(-0.0157, 0.0157)), noise_sigma=0.6 * 10 ** (-25 / 20),
                               taps=((0, taps[0]), (1, taps[1]), (3, taps[2])), seed=62))
    y = np.concatenate(parts)
    for algo in (1, 2):
        H.set_param(W.wifi_b200.P_CHAN_EST, algo)
        res, ref = H.rx_batch(y), O.rx(y, algo=algo)
        assert_frames_equal(res, ref)
        assert int(ref.frames["crc_ok"].sum()) >= 8


def test_config4_shape_many_links(O, W):
    """BASELINE configs[3] shape at reduced length: 1024 independent links in one call."""
    rng = np.random.default_rng(63)
    base, _ = make_capture(O, rng, [(7, 200), (7, 120)], snr_db=30, seed=1, lead=64, gap=500, cfo=0.002)
    n_links = 1024
    links = []
    for l in range(n_links):
        links.append(O.channel(base, n0=0, gain=1.0, noise_sigma=0.02, cfo=float(rng.uniform(-0.005, 0.005)), seed=100 + l))
    x = np.concatenate(links)
    off = np.arange(n_links + 1, dtype=np.uint64) * base.size
    h = W.Handle(max_samples=x.size + 1024, max_frames=4 * n_links, chan_est=1)
    res = h.rx_batch(x, off)
    ref = O.rx_links(x, off[:-1].astype(np.int64), np.full(n_links, base.size, np.int64), n_threads=8, algo=1, want_carrier=False)
    order = np.lexsort((res.frames["trigger"], res.frames["link"]))
    res.frames = res.frames[order]
    assert_frames_equal(res, ref)
    assert int(ref.frames["crc_ok"].sum()) >= 2 * n_links - 8
    h.close()


@pytest.mark.parametrize("enc", range(8))
def test_config5_shape_per_ladder_is_identical(H, O, W, enc):
    """BASELINE configs[4] shape: 599-byte PSDUs (571-byte feature-map patches) over an SNR ladder.
    The frame tables are equal, so the PER curve is the oracle's by construction."""
    H.set_param(W.wifi_b200.P_CHAN_EST, 0)
    per = []
    for snr in (2, 8, 14, 20, 26):
        rng = np.random.default_rng(1000 * enc + snr)
        y, _ = make_capture(O, rng, [(enc, 599)] * 6, snr_db=snr, seed=enc * 31 + snr, gap=600)
        res, ref = H.rx_batch(y), O.rx(y, algo=0)
        assert_frames_equal(res, ref)
        per.append(1 - ref.frames["crc_ok"].sum() / 6)
    assert per[0] >= per[-1]


def test_setters_take_effect(O, W):
    h = W.Handle(max_samples=1 << 18, sensitivity=0.56)
    rng = np.random.default_rng(71)
    y, _ = make_capture(O, rng, [(3, 100)] * 2, snr_db=12, seed=7)
    h.set_param(W.wifi_b200.P_SENSITIVITY, 0.8)
    h.set_param(W.wifi_b200.P_BANDWIDTH, 20e6)
    h.set_param(W.wifi_b200.P_FREQUENCY, 2.412e9)
    h.set_param(W.wifi_b200.P_CHAN_EST, 3)
    assert_frames_equal(h.rx_batch(y), O.rx(y, threshold=0.8, bw=20e6, freq=2.412e9, algo=3))
    with pytest.raises(W.WifiB200Error):
        h.set_param(W.wifi_b200.P_CHAN_EST, 9)
    with pytest.raises(W.WifiB200Error):
        h.rx_batch(np.zeros((1 << 18) + 10, np.complex64))     # more samples than max_samples
    h.close()


def test_facade_loopback_like_irs_tranceiver(O, W):
    """mac -> wifi_phy_hier TX -> x0.6 -> pad -> channel -> RX -> 'Extract Pics' slice, as
    gnu_radio/IRS_tranceiver.py wires it (:271-344)."""
    import struct
    phy = W.wifi_phy_hier(bandwidth=20e6, chan_est=0, encoding=3, frequency=5.89e9, sensitivity=0.56, max_samples=1 << 19)
    m = W.mac([0x23] * 6, [0x42] * 6, [0xff] * 6)
    payloads = [struct.pack("=L", 268) + bytes(np.random.default_rng(i).integers(0, 256, 264, dtype=np.uint8)) for i in range(5)]
    parts = []
    for p in payloads:
        burst = phy.mac_in(m.app_in(p))
        parts += [np.zeros(100, np.complex64), 0.6 * burst, np.zeros(1000, np.complex64)]   # foo.packet_pad2(100, 1000)
    x = np.concatenate(parts).astype(np.complex64)
    y = O.channel(x, gain=float(10 ** (22 / 20)), noise_sigma=float(np.sqrt(2)), cfo=0.001, seed=3)   # snr slider 22, noise_voltage 1
    got = []
    phy.msg_connect_mac_out(lambda pdu: got.append(pdu))
    for i in range(0, y.size, 4096):
        phy.samp_in(y[i:i + 4096], flush=(i + 4096 >= y.size))
    assert [pdu[1][24:][4:] for pdu in got] == [p[4:] for p in payloads]
    assert all(pdu[0]["dlt"] == 105 and pdu[0]["encoding"] == 3 for pdu in got)
    phy.set_encoding(5)
    assert phy.get_encoding() == 5 and phy.mac_in(m.app_in(b"x" * 100)).size == W.wifi_b200.frame_samples(5, 128)


def test_udp_runner_speaks_the_apps_contract(O, W):
    """upload_image_udp.py datagrams in (=L length + pickle(((y,x,c), 10x10x1 uint8))), decoded patches
    out on the viewer's port, through mac -> TX -> channel -> RX on the GPU."""
    import pickle
    import socket
    import struct
    import threading
    out = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    out.bind(("127.0.0.1", 0))
    out.settimeout(20)
    t = W.loopback_runner.IrsTransceiver(in_port=0, out_addr=("127.0.0.1", out.getsockname()[1]), snr=27.0, encoding=3, idle_flush_s=0.05)
    rng = np.random.default_rng(81)
    pieces = [((int(rng.integers(0, 30)), int(rng.integers(0, 30)), int(rng.integers(0, 3))), rng.integers(0, 256, (10, 10, 1), dtype=np.uint8)) for _ in range(12)]
    th = threading.Thread(target=t.serve, kwargs={"max_datagrams": len(pieces)})
    th.start()
    s = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    for piece in pieces:
        data = pickle.dumps(piece)
        s.sendto(struct.pack("=L", len(data)) + data, ("127.0.0.1", t.in_port))      # upload_image_udp.py:29-32
    got = []
    for _ in pieces:
        got.append(pickle.loads(out.recvfrom(2048)[0]))                               # download_image_udp.py:36-44
    th.join(timeout=30)
    assert [g[0] for g in got] == [p[0] for p in pieces]
    assert all(np.array_equal(g[1], p[1]) for g, p in zip(got, pieces))
    assert t.stats["pdus_out"] == len(pieces)
    t.close()


@pytest.mark.parametrize("soft", [False, True])
def test_host_batch_link_groups_give_the_single_pass_table(O, W, soft):
    """wifi_b200_rx_batch pipelines groups of links (copy / decode / results on three streams); frame records, rows, equalised
    points and PSDU slots of the groups follow each other exactly as one pass over all links would lay them out."""
    rng = np.random.default_rng(23)
    links, offs = [], [0]
    for l in range(7):
        y, _ = make_capture(O, rng, [(int(rng.integers(0, 8)), int(rng.integers(40, 400))) for _ in range(int(rng.integers(1, 5)))],
                            snr_db=float(rng.uniform(12, 30)), cfo=float(rng.uniform(-0.01, 0.01)), seed=l, lead=int(rng.integers(20, 300)), gap=int(rng.integers(200, 900)))
        links.append(y if l != 3 else np.zeros(500, np.complex64))          # one silent link: a group without frames
        offs.append(offs[-1] + links[-1].size)
    x = np.concatenate(links)
    ref = O.rx_links(x, offs[:-1], np.diff(offs), algo=1, soft=soft)
    h = W.Handle(max_samples=1 << 19, max_frames=512, chan_est=1, want_carrier=True, soft_decision=soft)
    try:
        for group in (1, 9000, 0):                                          # a group per link, a few links per group, one group
            h.set_param(W.wifi_b200.P_HOST_GROUP_SAMPLES, group)
            res = h.rx_batch(x, np.array(offs, np.uint64))
            assert_frames_equal(res, ref)
            rows, car = h.rows(carrier=True)
            used = np.concatenate([np.arange(int(r["row_off"]), int(r["row_off"]) + int(r["n_rows"])) for r in res.frames])
            assert np.array_equal(rows[used], ref.rows) and np.array_equal(car[used], ref.carrier)
            if soft:
                assert np.array_equal(h.soft_rows()[used], ref.soft)
            i16 = np.clip(np.rint(np.stack([x.real, x.imag], axis=1) * 2048), -32768, 32767).astype(np.int16)
            xq = (i16.astype(np.float32) * np.float32(1 / 2048)).view(np.complex64).reshape(-1)
            assert_frames_equal(h.rx_batch_sc16(i16, 1 / 2048, np.array(offs, np.uint64)), O.rx_links(xq, offs[:-1], np.diff(offs), algo=1, soft=soft))
    finally:
        h.close()


def test_host_alloc_gives_page_locked_memory_the_entry_points_accept(O, W):
    rng = np.random.default_rng(71)
    y, psdus = make_capture(O, rng, [(6, 300), (2, 150)], snr_db=30, seed=4)
    h = W.Handle(max_samples=1 << 17)
    try:
        a = h.host_alloc(y.size, np.complex64)
        assert a.size == y.size and not a.any()                 # zero filled by the first touch
        a[:] = y
        res = h.rx_batch(a)
        assert res.pdus() == [p[:-4] for p in psdus]
        h.host_free(a)
        with pytest.raises(W.WifiB200Error):
            h.host_alloc(0)
    finally:
        h.close()


def test_asynchronous_pushes_equal_synchronous_ones(O, W):
    """wifi_b200_rx_push_links_async / _rx_push_wait with two page-locked buffers used in turn: the copy of push k + 1 is in
    flight while push k is decoded; the frames that come out are those of the synchronous calls, in the same order."""
    import torch
    rng = np.random.default_rng(61)
    n_links, chunk = 5, 6000
    caps = [make_capture(O, rng, [(int(rng.integers(0, 8)), int(rng.integers(60, 500))) for _ in range(9)], snr_db=28,
                         cfo=float(rng.uniform(-0.01, 0.01)), seed=l, lead=int(rng.integers(50, 400)))[0] for l in range(n_links)]
    n_push = max(-(-c.size // chunk) for c in caps)
    off = (np.arange(n_links + 1) * chunk).astype(np.uint64)

    def fill(buf, k):
        for l, c in enumerate(caps):
            seg = c[k * chunk:(k + 1) * chunk]
            buf[l * chunk:l * chunk + seg.size] = seg
            buf[l * chunk + seg.size:(l + 1) * chunk] = 0

    def run(asynchronous):
        h = W.Handle(max_samples=n_links * (1 << 17), max_frames=512)
        pins = [torch.empty(2 * n_links * chunk, dtype=torch.float32, pin_memory=True) for _ in range(2)]
        bufs = [p.numpy().view(np.complex64) for p in pins]
        out = []
        if not asynchronous:
            for k in range(n_push):
                fill(bufs[0], k)
                h.rx_push_links_blob(bufs[0], off, flush=(k == n_push - 1))
                out += h.rx_pop(cap=512)
        else:
            fill(bufs[0], 0)
            h.rx_push_links_async(bufs[0], off, flush=(n_push == 1))
            for k in range(1, n_push + 1):
                if k < n_push:
                    fill(bufs[k & 1], k)                         # the other buffer: push k - 1 may still be copying from its own
                    h.rx_push_links_async(bufs[k & 1], off, flush=(k == n_push - 1))
                assert h.rx_push_wait()                          # completes push k - 1
                out += h.rx_pop(cap=512)
            assert not h.rx_push_wait()                          # nothing pending
            with pytest.raises(W.WifiB200Error):                 # a fourth pending push is refused
                for _ in range(4):
                    h.rx_push_links_async(bufs[0], off)
        h.close()
        return [(int(f["link"]), int(f["trigger"]), d) for f, d in out]

    sync, asyn = run(False), run(True)
    assert sync == asyn and len(sync) >= 30
    want = []
    for l, c in enumerate(caps):
        pad = np.concatenate([c, np.zeros(n_push * chunk - c.size, np.complex64)])
        r = O.rx(pad, algo=0, want_carrier=False)
        want += [(l, int(f["trigger"]), r.psdu(i)[:-4]) for i, f in enumerate(r.frames) if f["crc_ok"]]
    assert sorted(sync) == sorted(want)


def test_wire_format_pushes_equal_float_pushes(O, W):
    """wifi_b200_rx_push_links_sc16_async: int16 I/Q over PCIe, converted while it is appended to the streams.  The frames are
    those of pushing x = float32(i16) * scale as complex64 (and of the oracle on that capture); the two forms mix freely."""
    import torch
    rng = np.random.default_rng(77)
    n_links, chunk, scale = 4, 5000, np.float32(1.0 / 4096)
    caps16 = []
    for l in range(n_links):
        c = make_capture(O, rng, [(int(rng.integers(0, 8)), int(rng.integers(60, 500))) for _ in range(8)], snr_db=30,
                         cfo=float(rng.uniform(-0.01, 0.01)), seed=40 + l, lead=int(rng.integers(50, 400)))[0]
        q = np.clip(np.round(c.view(np.float32) / scale), -32768, 32767).astype(np.int16)          # what an ADC + DDC would deliver
        caps16.append(q)
    n_push = max(-(-(q.size // 2) // chunk) for q in caps16)
    caps16 = [np.concatenate([q, np.zeros(2 * n_push * chunk - q.size, np.int16)]) for q in caps16]
    capsf = [(q.astype(np.float32) * scale).view(np.complex64) for q in caps16]
    off = (np.arange(n_links + 1) * chunk).astype(np.uint64)

    def run(wire):
        h = W.Handle(max_samples=n_links * (1 << 17), max_frames=512)
        pf = [torch.empty(2 * n_links * chunk, dtype=torch.float32, pin_memory=True) for _ in range(2)]
        p16 = [torch.empty(2 * n_links * chunk, dtype=torch.int16, pin_memory=True) for _ in range(2)]
        out = []

        def push(k):
            if wire(k):
                b = p16[k & 1].numpy()
                for l in range(n_links):
                    b[2 * l * chunk:2 * (l + 1) * chunk] = caps16[l][2 * k * chunk:2 * (k + 1) * chunk]
                h.rx_push_links_sc16_async(b, float(scale), off, flush=(k == n_push - 1))
            else:
                b = pf[k & 1].numpy().view(np.complex64)
                for l in range(n_links):
                    b[l * chunk:(l + 1) * chunk] = capsf[l][k * chunk:(k + 1) * chunk]
                h.rx_push_links_async(b, off, flush=(k == n_push - 1))

        push(0)
        for k in range(1, n_push + 1):
            if k < n_push:
                push(k)
            assert h.rx_push_wait()
            out += h.rx_pop(cap=512)
        with pytest.raises(W.WifiB200Error):
            h.rx_push_links_sc16_async(p16[0].numpy(), 0.0, off)           # scale 0 is refused
        h.close()
        return [(int(f["link"]), int(f["trigger"]), float(f["freq_long"]), float(f["snr"]), d) for f, d in out]

    as_float, as_wire, mixed = run(lambda k: False), run(lambda k: True), run(lambda k: k % 3 != 1)
    assert as_float == as_wire == mixed and len(as_float) >= 24
    want = []
    for l, c in enumerate(capsf):
        r = O.rx(c, algo=0, want_carrier=False)
        want += [(l, int(f["trigger"]), float(f["freq_long"]), float(f["snr"]), r.psdu(i)[:-4]) for i, f in enumerate(r.frames) if f["crc_ok"]]
    a_, b_ = sorted(as_wire), sorted(want)
    assert [x[:3] + x[4:] for x in a_] == [x[:3] + x[4:] for x in b_]                # stream, trigger, frequency offset, bytes
    assert np.allclose([x[3] for x in a_], [x[3] for x in b_], rtol=1e-9, atol=1e-9)  # snr: double log10, libm vs device


def test_loopback_epsilon_is_the_channel_models_frequency_offset(O, W):
    """channel_model(frequency_offset = epsilon * freq / 10e6) is cycles per sample (IRS_tranceiver.py:284,434): with the
    slider at its end stop (20e-6) the receiver must report 2 pi * 0.01178 = 0.074 rad/sample, not a 2e7 times smaller one."""
    import math
    t = W.loopback_runner.IrsTransceiver(in_port=0, out_addr=("127.0.0.1", 9), snr=27.0, epsilon=20e-6, encoding=3)
    try:
        want = 2 * math.pi * 20e-6 * 5.89e9 / 10e6
        burst = t.phy.mac_in(t.mac.app_in(b"x" * 300))
        y = t._through_channel(burst)
        pdus, res = t.phy.rx(y)
        assert len(pdus) == 1 and pdus[0][1][24:] == b"x" * 300
        f = res.frames[0]
        assert abs((float(f["freq_short"]) - float(f["freq_long"])) - want) < 2e-3, (f["freq_short"], f["freq_long"], want)
        assert abs(pdus[0][0]["freqofs"] - want * 20e6 / (2 * math.pi)) < 2e-3 * 20e6 / (2 * math.pi)
        t.set_epsilon(0.0)
        _, res0 = t.phy.rx(t._through_channel(burst))
        assert abs(float(res0.frames[0]["freq_short"]) - float(res0.frames[0]["freq_long"])) < 2e-3
    finally:
        t.close()


@pytest.mark.parametrize("soft", [False, True])
def test_collection_through_more_than_four_bursts(O, W, soft):
    """decode_mac keeps collecting a frame's symbols through any number of bursts whose tags it refuses (oversize
    SIGNAL fields); the library used to give up beyond four and fail the whole call."""
    y = capture_with_collection_over_many_bursts(O, np.random.default_rng(5))
    ref = O.rx(y, algo=0, soft=soft)
    assert ref.frames[0]["decoded"] == 1 and int((ref.frames["n_rows"] > 0).sum()) >= 6 and int(ref.frames["accepted"].sum()) == 1
    h = W.Handle(max_samples=1 << 16, max_frames=64, soft_decision=soft)
    try:
        assert_frames_equal(h.rx_batch(y), ref)
        # streamed: the open collection is carried from run to run with the held bursts
        want = [(int(f["trigger"]), ref.psdu(i)[:-4]) for i, f in enumerate(ref.frames) if f["crc_ok"]]
        got = []
        for pos in range(0, y.size, 3000):
            h.rx_push(y[pos:pos + 3000], flush=(pos + 3000 >= y.size))
            got += h.rx_pop()
        assert [(int(f["trigger"]), d) for f, d in got] == want
    finally:
        h.close()


def test_streaming_recovers_after_a_failed_run(O, W):
    """A run that fails (here: more triggers than max_frames) drops the buffered region instead of re-running it on
    every later push; the stream decodes what follows."""
    rng = np.random.default_rng(77)
    y, _ = make_capture(O, rng, [(3, 60)] * 12, snr_db=30, gap=700, seed=1)
    z, psdus = make_capture(O, rng, [(3, 200)] * 2, snr_db=30, seed=2)
    h = W.Handle(max_samples=1 << 18, max_frames=4)
    try:
        with pytest.raises(W.WifiB200Error) as e:
            h.rx_push(y, flush=False)
        assert e.value.code == W.wifi_b200.E_OVERFLOW
        h.rx_push(z, flush=True)
        assert [d for _, d in h.rx_pop()] == [p[:-4] for p in psdus]
    finally:
        h.close()


@pytest.mark.parametrize("algo", [0, 1, 3])
def test_soft_decision_mode_matches_oracle(O, W, algo):
    """Soft-decision extension (max-log LLR demapper + soft Viterbi, DESIGN.md 9): no reference
    counterpart, the oracle defines it.  int8 soft values and everything downstream must be equal."""
    rng = np.random.default_rng(90 + algo)
    specs = [(e, int(rng.integers(40, 500))) for e in range(8)] * 2 + [(7, 1528), (1, 919)]
    taps = ((0, 1.0), (2, 0.35 * np.exp(1j * 0.7)))
    y, psdus = make_capture(O, rng, specs, snr_db=17, cfo=0.007, taps=taps, seed=algo, gap=700)
    h = W.Handle(max_samples=1 << 21, max_frames=1024, chan_est=algo, soft_decision=True, want_carrier=True)
    res = h.rx_batch(y)
    ref = O.rx(y, algo=algo, soft=True)
    assert_frames_equal(res, ref)
    soft = h.soft_rows()
    for i in range(len(ref.frames)):
        f, g = ref.frames[i], res.frames[i]
        ncb = [48, 48, 96, 96, 192, 192, 288, 288][f["encoding"]]
        a = soft[g["row_off"]:g["row_off"] + g["n_rows"], :ncb]
        b = ref.soft[f["row_off"]:f["row_off"] + f["n_rows"], :ncb]
        assert np.array_equal(a, b), ("soft", i)
    # the soft decoder recovers frames the hard decoder loses at this SNR
    hard = O.rx(y, algo=algo)
    assert ref.frames["crc_ok"].sum() > hard.frames["crc_ok"].sum()
    # switching the parameter at run time gives the hard-decision result again
    h.set_param(W.wifi_b200.P_SOFT_DECISION, 0)
    assert_frames_equal(h.rx_batch(y), hard)
    h.close()


def test_soft_decision_truncated_and_gathered(O, W):
    rng = np.random.default_rng(95)
    y, _ = make_capture(O, rng, [(3, 120), (5, 300), (6, 500), (1, 60)], snr_db=25, gap=150, seed=5)
    y = y[:-500]
    h = W.Handle(max_samples=1 << 19, soft_decision=True, chan_est=1)
    assert_frames_equal(h.rx_batch(y), O.rx(y, algo=1, soft=True))
    h.close()


@pytest.mark.parametrize("minp", [1, 3, 5])
def test_min_plateau_variants(O, W, minp):
    rng = np.random.default_rng(110 + minp)
    y, _ = make_capture(O, rng, [(2, 90), (6, 200), (0, 40)], snr_db=9, seed=minp, gap=520)
    h = W.Handle(max_samples=1 << 18, min_plateau=minp)
    assert_frames_equal(h.rx_batch(y), O.rx(y, min_plateau=minp))
    h.close()


@pytest.mark.parametrize("scale", [1e-4, 1.0, 3e3])
def test_amplitude_extremes_and_frame_at_sample_zero(H, O, W, scale):
    """The front-end decides |a|^2 > thr^2 p^2 (DESIGN.md choice 7); very small and very large inputs, exact zeros
    (0 > 0: not over, as upstream's 0/0) and a frame that starts at sample 0 must not change decisions."""
    rng = np.random.default_rng(120)
    y, _ = make_capture(O, rng, [(3, 150), (5, 260)], snr_db=22, seed=8, lead=0, gap=600, cfo=0.019)
    y = (y * np.float32(scale)).astype(np.complex64)
    y[5000:5400] = 0                       # dead air: 0/0 in the correlation ratio
    H.set_param(W.wifi_b200.P_CHAN_EST, 0)
    assert_frames_equal(H.rx_batch(y), O.rx(y, algo=0))
    assert np.array_equal(H.flags(0, y.size), O.flags(y, 0.56))


def test_streaming_small_pushes_and_soft(O, W):
    rng = np.random.default_rng(130)
    y, _ = make_capture(O, rng, [(int(rng.integers(0, 8)), int(rng.integers(40, 300))) for _ in range(8)], snr_db=16, cfo=-0.004, seed=9)
    ref = O.rx(y, algo=0, soft=True)
    want = [(int(f["trigger"]), ref.psdu(i)[:-4]) for i, f in enumerate(ref.frames) if f["crc_ok"]]
    h = W.Handle(max_samples=1 << 18, soft_decision=True)
    got, pos = [], 0
    while pos < y.size:
        n = int(rng.integers(1, 700))
        h.rx_push(y[pos:pos + n], flush=(pos + n >= y.size))
        got += h.rx_pop()
        pos += n
    assert [(int(f["trigger"]), d) for f, d in got] == want and len(want) >= 5
    st = h.stats()
    assert st["crc_ok"] == len(want) and st["pdu_bytes"] == sum(len(d) for _, d in want)
    h.close()


@pytest.mark.parametrize("trunc", [500, 641])
def test_time_sharding_reconciles_adversarial_traffic(O, W, trunc):
    """Back-to-back traffic without one idle gap (trigger chains that never merge; a decode_mac tag pending across the
    whole zone): the ranks' check fails, the lowest rank decodes again from a known state through
    wifi_b200_rx_batch_dev_state, and the union of the owned frames equals the sequential oracle's table."""
    S = W.sharding
    y = adversarial_stream(O, trunc=trunc)
    truth = S.records(O.rx(y, algo=0, want_carrier=False).frames, 0)
    h = W.Handle(max_samples=1 << 18, max_frames=1024, chan_est=0)
    try:
        dec = gpu_segment_decoder(h, y)
        for world in (2, 4):
            owned, rounds = S.simulate_ranks(dec, S.shard_stream(y.size, world), y.size)
            assert S.same(np.concatenate(owned), truth) and rounds >= 1, (world, rounds)
    finally:
        h.close()


@pytest.mark.parametrize("seed", range(int(os.environ.get("WIFI_FUZZ_SEEDS", "3"))))
def test_fuzz_time_sharding_random_traffic(O, W, seed):
    """Random traffic (gaps from none to a long silence, frames cut short by the next one) cut across 2..6 ranks on the GPU,
    whole tables and owned tails only: always the sequential oracle's table."""
    S = W.sharding
    rng = np.random.default_rng(900 + seed)
    parts = [np.zeros(int(rng.integers(0, 400)), np.complex64)]
    for i in range(int(rng.integers(25, 60))):
        f = O.tx_frame(make_psdu(O, rng, int(rng.integers(30, 500)), seq=i), int(rng.integers(0, 8)), seed=1 + i % 127)
        if rng.random() < 0.2:
            f = f[:int(rng.integers(350, f.size))]
        parts += [f, np.zeros(int(rng.choice([0, 0, 40, 300, 900, 2500, 60000 if i % 17 == 5 else 700])), np.complex64)]
    x = np.concatenate(parts).astype(np.complex64)
    y = O.channel(x, gain=0.6, cfo=float(rng.uniform(-0.01, 0.01)), noise_sigma=0.6 * 10 ** (-float(rng.uniform(14, 30)) / 20), seed=seed)
    algo = int(rng.integers(0, 4))
    truth = S.records(O.rx(y, algo=algo, want_carrier=False).frames, 0)
    h = W.Handle(max_samples=y.size + 1024, max_frames=2048, chan_est=algo)
    try:
        dec = gpu_segment_decoder(h, y)
        for world in (2, 3, 6):
            owned, rounds = S.simulate_ranks(dec, S.shard_stream(y.size, world), y.size)
            assert S.same(np.concatenate(owned), truth), (seed, world, rounds)
            owned, rounds = S.simulate_ranks(dec, S.shard_stream(y.size, world), y.size, tail_rows=16)
            assert S.same(np.concatenate(owned), truth), (seed, world, rounds, "tails")
    finally:
        h.close()


def test_resumed_stream_state_entry_point_matches_oracle(O, W):
    """wifi_b200_rx_batch_dev_state against the oracle given the same (min_pos, fo_carry, hist), every field and PSDU."""
    S = W.sharding
    rng = np.random.default_rng(41)
    y, _ = make_capture(O, rng, [(int(e), 150 + 60 * int(e)) for e in (0, 3, 5, 7, 2, 6, 1, 4)], snr_db=27, seed=6, gap=300, cfo=0.01)
    truth = S.records(O.rx(y, algo=3, want_carrier=False).frames, 0)
    h = W.Handle(max_samples=1 << 18, max_frames=256, chan_est=3)
    try:
        dec = gpu_segment_decoder(h, y)
        for k in (2, 5):
            lo, st, _ = S.resume_point(truth, 0, int(truth[k, S.TRIG]) + 1)
            ref = O.rx(y[lo - st["hist"]:], algo=3, hist=st["hist"], min_pos=st["min_pos"], fo_carry=st["fo_carry"])
            dec(lo, y.size, st, True)
            assert_frames_equal(h.results(), ref)
            assert S.same(S.records(ref.frames, lo), truth[k:])
        with pytest.raises(W.WifiB200Error):       # history that is not there
            bad = np.zeros(1, W.wifi_b200.LINK_STATE_DTYPE)
            bad["hist"] = 64
            h.rx_batch_dev_state(dec.keepalive.data_ptr(), np.array([0, 1000], np.uint64), bad)
    finally:
        h.close()


def test_overlapping_segment_shards_dedup_to_whole_stream(O, W):
    """SURVEY 8e (ii): one capture cut into overlapping segments (as ranks would take them), each
    decoded on its own, frames owned by the segment whose core region holds the trigger.  The union
    equals the single-pass result (here both segments run on the same GPU, one after the other)."""
    S = W.sharding
    rng = np.random.default_rng(140)
    y, _ = make_capture(O, rng, [(int(rng.integers(0, 8)), int(rng.integers(100, 700))) for _ in range(40)], snr_db=24, seed=14, gap=900,
                        cfo=0.003)
    h = W.Handle(max_samples=1 << 21, max_frames=512, chan_est=0)
    whole = h.rx_batch(y)
    got = []
    for seg in S.shard_stream(y.size, 3):
        r = h.rx_batch(y[seg["start"]:seg["end"]], final=(seg["end"] == y.size))
        keep = S.owned(r.frames, seg)
        for i in np.nonzero(keep)[0]:
            f = r.frames[i]
            got.append((int(f["trigger"]) + seg["start"], int(f["crc_ok"]), int(f["encoding"]), int(f["length"]), r.psdu(i) if f["decoded"] else None))
    want = [(int(f["trigger"]), int(f["crc_ok"]), int(f["encoding"]), int(f["length"]), whole.psdu(i) if f["decoded"] else None)
            for i, f in enumerate(whole.frames)]
    assert sorted(got, key=lambda t: t[0]) == want
    assert sum(w[1] for w in want) >= 36
    h.close()


@pytest.mark.parametrize("soft", [False, True])
def test_non_finite_samples_do_not_break_parity(O, W, soft):
    """NaN / Inf samples (a saturated or corrupted capture) poison the frames they touch in the same
    way on both sides; the other frames decode."""
    rng = np.random.default_rng(150)
    y, psdus = make_capture(O, rng, [(2, 200), (5, 300), (7, 400), (0, 80)], snr_db=28, seed=15, gap=800)
    y = y.copy()
    y[1500:1503] = np.nan              # inside frame 0's data
    y[6000] = np.inf + 0j               # inside frame 1
    h = W.Handle(max_samples=1 << 18, soft_decision=soft, chan_est=1)
    res, ref = h.rx_batch(y), O.rx(y, algo=1, soft=soft)
    assert_frames_equal(res, ref)
    assert ref.frames["crc_ok"].sum() >= 2
    h.close()


@pytest.mark.gpu
def test_sc16_wire_format_ingest_equals_host_conversion(H, O, W):
    """int16 I/Q converted on the GPU (x = float32(i16) * scale, UHD's sc16 -> fc32 rule) decodes exactly like the
    same samples converted on the host and pushed through the fc32 entry point."""
    H.set_param(W.wifi_b200.P_CHAN_EST, 0)
    rng = np.random.default_rng(21)
    parts = [np.zeros(411, np.complex64)]
    psdus = []
    for i, enc in enumerate((7, 4, 0, 5, 2)):
        p = O.mac_frame(rng.integers(0, 256, 150 + 90 * i, dtype=np.uint8).tobytes(), seq=i)
        psdus.append(p)
        parts += [O.tx_frame(p, enc, seed=i + 1), np.zeros(900 + 37 * i, np.complex64)]
    x = np.concatenate(parts).astype(np.complex64)
    y = O.channel(x, gain=0.5, cfo=0.002, noise_sigma=0.5 * 10 ** (-30 / 20), seed=4)
    scale = np.float32(1.0 / 8192.0)                                    # ~13-bit ADC headroom
    i16 = np.clip(np.rint(np.stack([y.real, y.imag], axis=1) / scale), -32768, 32767).astype(np.int16)
    host = (i16.astype(np.float32) * scale).reshape(-1).view(np.complex64)
    # two links so that the odd link offset exercises the unaligned tail of the converter
    cut = 3001
    off = np.array([0, cut, host.size], np.uint64)
    a = H.rx_batch(host, off)
    b = H.rx_batch_sc16(i16, float(scale), off)
    ref = O.rx_links(host, [0, cut], [cut, host.size - cut], algo=0)
    for k in ("trigger", "link", "burst_len", "frame_start", "sig_ok", "encoding", "length", "n_rows", "decoded", "crc_ok"):
        assert np.array_equal(a.frames[k], b.frames[k]) and np.array_equal(b.frames[k], ref.frames[k]), k
    assert np.array_equal(a.frames["freq_short"], b.frames["freq_short"]) and np.array_equal(a.frames["snr"], b.frames["snr"])
    assert a.pdus() == b.pdus() == ref.pdus()
    assert len(b.pdus()) >= 3


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(int(os.environ.get("WIFI_FUZZ_SEEDS", "8"))))
def test_fuzz_random_captures(O, W, seed):
    """Random frame mixes (all MCS, lengths 1..1528, tight and wide gaps, 4-34 dB, CFO, 3-tap multipath, every
    equalizer, hard and soft decisions, several links): frame table, rows, equalised points and PSDUs equal the
    oracle's -- including the frames that fail."""
    rng = np.random.default_rng(9000 + seed)
    algo = int(rng.integers(0, 4))
    soft = bool(seed & 1)
    n_links = int(rng.integers(1, 4))
    links, offs = [], [0]
    for l in range(n_links):
        parts = [np.zeros(int(rng.integers(0, 400)), np.complex64)]
        for i in range(int(rng.integers(3, 9))):
            enc = int(rng.integers(0, 8))
            ln = int(rng.choice([int(rng.integers(1, 60)), int(rng.integers(60, 600)), int(rng.integers(600, 1529))], p=[0.2, 0.6, 0.2]))
            if enc < 2 and ln > 400:
                ln = int(rng.integers(1, 400))          # keep the BPSK frames (and the oracle's run time) short
            parts.append(O.tx_frame(make_psdu(O, rng, ln, seq=i), enc, seed=int(rng.integers(1, 128))))
            parts.append(np.zeros(int(rng.choice([int(rng.integers(0, 60)), int(rng.integers(300, 1500))], p=[0.25, 0.75])), np.complex64))
        x = np.concatenate(parts).astype(np.complex64)
        taps = ((0, 1.0),) if rng.random() < 0.5 else ((0, 1.0), (1, 0.4 * np.exp(1j * rng.uniform(0, 6.28))), (3, 0.2 * np.exp(1j * rng.uniform(0, 6.28))))
        snr = float(rng.uniform(4, 34))
        yl = O.channel(x, gain=0.6, cfo=float(rng.uniform(-0.02, 0.02)), noise_sigma=0.6 * 10 ** (-snr / 20), taps=taps, seed=100 * seed + l)
        u = rng.random()
        if u < 0.3:
            yl = yl[:int(rng.integers(1, yl.size))]             # the capture ends anywhere: mid-frame, mid-preamble, short final bursts
        elif u < 0.4:
            yl = yl[:int(rng.integers(0, 100))]                 # a (nearly) empty link
        links.append(yl)
        offs.append(offs[-1] + links[-1].size)
    y = np.concatenate(links)
    final = bool(rng.random() < 0.8)
    h = W.Handle(max_samples=y.size + 1024, max_frames=256, want_carrier=True, chan_est=algo, soft_decision=soft)
    h.set_param(W.wifi_b200.P_HOST_GROUP_SAMPLES, int(rng.choice([0, 1, 5000])))
    try:
        res = h.rx_batch(y, np.array(offs, np.uint64), final=final) if y.size else h.rx_batch(np.zeros(0, np.complex64))
        ref = O.rx_links(y, np.array(offs[:-1], np.int64), np.diff(offs).astype(np.int64), algo=algo, soft=soft, final=final)
        assert_frames_equal(res, ref)
        rows, car = h.rows(carrier=True)
        for i in range(len(ref.frames)):
            f, g = ref.frames[i], res.frames[i]
            assert np.array_equal(rows[g["row_off"]:g["row_off"] + g["n_rows"]], ref.rows[f["row_off"]:f["row_off"] + f["n_rows"]]), ("rows", i)
            assert np.array_equal(car[g["row_off"]:g["row_off"] + g["n_rows"]], ref.carrier[f["row_off"]:f["row_off"] + f["n_rows"]]), ("carrier", i)
        assert res.pdus() == ref.pdus()
    finally:
        h.close()


@pytest.mark.gpu
def test_streaming_releases_a_lone_frame_and_batches_small_pushes(O, W):
    """(1) Sparse traffic: a frame followed by noise only is published once MAX_SAMPLES (43200) of the stream have
    arrived behind its trigger -- no later frame and no flush needed.  (2) WIFI_P_STREAM_BATCH: small pushes only
    buffer; the PDUs are those of the whole-capture decode, in order."""
    rng = np.random.default_rng(77)
    y1, _ = make_capture(O, rng, [(5, 300)], snr_db=28, cfo=0.004, seed=9, gap=200)
    noise = O.channel(np.zeros(60000, np.complex64), gain=1.0, noise_sigma=0.6 * 10 ** (-28 / 20), seed=10)
    y2, _ = make_capture(O, rng, [(3, 500), (7, 900)], snr_db=28, cfo=-0.003, seed=11)
    y = np.concatenate([y1, noise, y2]).astype(np.complex64)
    ref = O.rx(y, algo=0)
    want = [(int(f["trigger"]), ref.psdu(i)[:-4]) for i, f in enumerate(ref.frames) if f["crc_ok"]]
    assert len(want) == 3
    # (1) pushes of 4096 samples, never flushed until the very end
    h = W.Handle(max_samples=1 << 18)
    got, first_seen_at = [], None
    for pos in range(0, y.size, 4096):
        h.rx_push(y[pos:pos + 4096], flush=False)
        new = h.rx_pop()
        if new and first_seen_at is None:
            first_seen_at = pos + 4096
        got += new
    t0 = want[0][0]
    assert first_seen_at is not None and first_seen_at <= t0 + 43200 + 2 * 4096, (first_seen_at, t0)     # before the next frame (y1.size + 60000) arrives
    assert first_seen_at < y1.size + 60000
    h.rx_push(np.zeros(0, np.complex64), flush=True)
    got += h.rx_pop()
    assert [(int(f["trigger"]), d) for f, d in got] == want
    h.close()
    # (2) 1000-sample pushes with a 20000-sample batch threshold
    h = W.Handle(max_samples=1 << 18)
    h.set_param(W.wifi_b200.P_STREAM_BATCH, 20000)
    assert h.get_param(W.wifi_b200.P_STREAM_BATCH) == 20000
    got, runs = [], 0
    for pos in range(0, y.size, 1000):
        before = h.stats()["samples"]
        h.rx_push(y[pos:pos + 1000], flush=(pos + 1000 >= y.size))
        runs += h.stats()["samples"] != before
        got += h.rx_pop()
    assert [(int(f["trigger"]), d) for f, d in got] == want
    assert runs <= y.size // 20000 + 2, runs          # the pipeline ran once per batch, not once per push
    # an empty push runs the pipeline on what is buffered without ending the stream
    h.rx_reset()
    h.rx_push(y[:y1.size + 50000], flush=False)       # one push above the threshold: runs, frame 1 is released (43200 behind it)
    first = h.rx_pop()
    h.rx_push(y[y1.size + 50000:y1.size + 50000 + 12000], flush=False)    # below the threshold: buffered only
    before = h.stats()["samples"]
    h.rx_push(np.zeros(0, np.complex64), flush=False)
    assert h.stats()["samples"] != before
    h.rx_push(y[y1.size + 62000:], flush=True)
    rest = h.rx_pop()
    assert [(int(f["trigger"]), d) for f, d in first + rest] == want
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(int(os.environ.get("WIFI_FUZZ_SEEDS", "6"))))
def test_fuzz_streaming_equals_whole_capture(O, W, seed):
    """Random streams (frames of every MCS, dead air from 0 to 60000 samples between them so that bursts end by a
    later trigger, by MAX_SAMPLES or by the flush), pushed in random chunk sizes with a random WIFI_P_STREAM_BATCH:
    the published PDUs and their absolute trigger positions equal the whole-capture decode."""
    rng = np.random.default_rng(4200 + seed)
    parts = [np.zeros(int(rng.integers(0, 300)), np.complex64)]
    for i in range(int(rng.integers(4, 10))):
        enc = int(rng.integers(0, 8))
        ln = int(rng.integers(20, 400 if enc < 2 else 1200))
        parts.append(0.6 * O.tx_frame(make_psdu(O, rng, ln, seq=i), enc, seed=int(rng.integers(1, 128))))
        parts.append(np.zeros(int(rng.choice([int(rng.integers(0, 200)), int(rng.integers(500, 3000)), int(rng.integers(44000, 60000))], p=[0.2, 0.5, 0.3])), np.complex64))
    x = np.concatenate(parts).astype(np.complex64)
    y = O.channel(x, gain=1.0, cfo=float(rng.uniform(-0.01, 0.01)), noise_sigma=0.6 * 10 ** (-float(rng.uniform(18, 32)) / 20), seed=seed)
    algo = int(rng.integers(0, 4))
    ref = O.rx(y, algo=algo)
    want = [(int(f["trigger"]), ref.psdu(i)[:-4]) for i, f in enumerate(ref.frames) if f["crc_ok"]]
    h = W.Handle(max_samples=1 << 20, max_frames=256, chan_est=algo)
    try:
        h.set_param(W.wifi_b200.P_STREAM_BATCH, int(rng.choice([0, 0, 5000, 40000, 200000])))
        got, pos = [], 0
        while pos < y.size:
            n = int(rng.choice([int(rng.integers(1, 500)), int(rng.integers(500, 20000)), int(rng.integers(20000, 90000))]))
            h.rx_push(y[pos:pos + n], flush=(pos + n >= y.size))
            if rng.random() < 0.1:
                h.rx_push(np.zeros(0, np.complex64))          # "run now"
            got += h.rx_pop()
            pos += n
        assert [(int(f["trigger"]), d) for f, d in got] == want
    finally:
        h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["fc32", "sc16"])
def test_ota_runners_record_and_replay(O, W, fmt, tmp_path):
    """IRS_user stand-in (UDP 52001-style datagrams -> MAC -> TX -> x0.5 -> pad -> IQ file) and IRS_AP stand-in (IQ file
    -> RX -> 'Extract Pics' -> UDP): the recording equals the oracle's TX, the replay returns every payload."""
    import io
    import socket
    rng = np.random.default_rng(55)
    payloads = [rng.integers(0, 256, int(rng.integers(20, 900)), dtype=np.uint8).tobytes() for _ in range(7)]
    rec = io.BytesIO()
    u = W.ota_runners.IrsUser(rec, in_port=0, encoding=4, multi_const=0.5, fmt=fmt)
    for p in payloads:
        u.handle_datagram(p)
    u.handle_datagram(bytes(1501))                                   # oversize: dropped like upstream's mac
    assert u.stats["bursts_out"] == 7 and u.stats["dropped_oversize"] == 1
    raw = rec.getvalue()
    want = np.concatenate([np.concatenate([np.zeros(100, np.complex64), np.complex64(0.5) * O.tx_frame(O.mac_frame(p, seq=i), 4, seed=i + 1),
                                           np.zeros(1000, np.complex64)]) for i, p in enumerate(payloads)]).astype(np.complex64)
    if fmt == "fc32":
        assert np.array_equal(np.frombuffer(raw, np.complex64), want)
    else:
        q = np.clip(np.rint(want.view(np.float32) / np.float32(1.0 / 16384.0)), -32768, 32767).astype(np.int16)
        assert np.array_equal(np.frombuffer(raw, np.int16), q)
    u.close()
    out = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    out.bind(("127.0.0.1", 0))
    out.settimeout(20)
    path = tmp_path / ("rec." + fmt)
    path.write_bytes(raw)
    a = W.ota_runners.IrsAp(("127.0.0.1", out.getsockname()[1]), chan_est=0, fmt=fmt, chunk=20000)
    st = a.run(str(path))
    # the zeros between the noise-free frames are silence (no trigger in them cuts a frame short, DESIGN.md choice 7):
    # the replay forwards exactly the oracle's PDUs, every payload once
    played = want if fmt == "fc32" else (q.astype(np.float32) * np.float32(1.0 / 16384.0)).view(np.complex64)
    ref = O.rx(played, algo=0)
    assert st["samples_in"] == want.size and st["pdus_out"] == len(ref.pdus()) == 7
    got = [out.recvfrom(4096)[0] for _ in range(st["pdus_out"])]
    assert got == [p[24:][4:] for p in ref.pdus()]                   # "Extract Pics" strips the MAC header and 4 more bytes
    assert got == [p[4:] for p in payloads]
    a.close()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(int(os.environ.get("WIFI_FUZZ_SEEDS", "6"))))
def test_fuzz_multi_link_streaming(O, W, seed):
    """wifi_b200_rx_push_links: several continuous streams in one handle, each fed its own random chunk sizes (some
    pushes bring nothing for a link): per link, the published PDUs and absolute triggers equal that link's
    whole-capture decode."""
    rng = np.random.default_rng(7700 + seed)
    n_links = int(rng.integers(2, 6))
    algo = int(rng.integers(0, 4))
    streams, want = [], []
    for l in range(n_links):
        parts = [np.zeros(int(rng.integers(0, 500)), np.complex64)]
        for i in range(int(rng.integers(2, 7))):
            enc = int(rng.integers(0, 8))
            ln = int(rng.integers(20, 300 if enc < 2 else 1000))
            parts.append(0.6 * O.tx_frame(make_psdu(O, rng, ln, seq=i), enc, seed=int(rng.integers(1, 128))))
            parts.append(np.zeros(int(rng.choice([int(rng.integers(0, 300)), int(rng.integers(600, 4000)), int(rng.integers(44000, 50000))], p=[0.2, 0.6, 0.2])), np.complex64))
        x = np.concatenate(parts).astype(np.complex64)
        y = O.channel(x, gain=1.0, cfo=float(rng.uniform(-0.01, 0.01)), noise_sigma=0.6 * 10 ** (-float(rng.uniform(20, 32)) / 20), seed=10 * seed + l)
        streams.append(y)
        ref = O.rx(y, algo=algo)
        want.append([(int(f["trigger"]), ref.psdu(i)[:-4]) for i, f in enumerate(ref.frames) if f["crc_ok"]])
    h = W.Handle(max_samples=1 << 21, max_frames=512, chan_est=algo)
    try:
        h.set_param(W.wifi_b200.P_STREAM_BATCH, int(rng.choice([0, 8000, 60000])))
        pos = [0] * n_links
        got = [[] for _ in range(n_links)]
        while any(pos[l] < streams[l].size for l in range(n_links)):
            chunks = []
            for l in range(n_links):
                n = 0 if rng.random() < 0.2 else int(rng.choice([int(rng.integers(1, 800)), int(rng.integers(800, 30000))]))
                chunks.append(streams[l][pos[l]:pos[l] + n])
                pos[l] += len(chunks[-1])
            done = all(pos[l] >= streams[l].size for l in range(n_links))
            h.rx_push_links(chunks, flush=done)
            if not done and seed % 3 == 2 and rng.random() < 0.5:
                continue                                     # results pile up over several runs before they are collected
            while True:
                if seed & 1:                                 # bulk pop: records + one blob; packed copies or views of the library's buffers
                    meta, blob = h.rx_pop_arrays(cap=int(rng.integers(1, 40)), copy=bool(seed & 2) or rng.random() < 0.3)
                    for f in meta:
                        got[int(f["link"])].append((int(f["trigger"]), blob[f["psdu_off"]:f["psdu_off"] + f["length"] - 4].tobytes()))
                    n_popped = len(meta)
                else:
                    n_popped = 0
                    for f, d in h.rx_pop(cap=int(rng.integers(1, 40))):
                        got[int(f["link"])].append((int(f["trigger"]), d))
                        n_popped += 1
                if not n_popped:
                    break
        assert got == want
        with pytest.raises(W.WifiB200Error):
            h.rx_push(np.zeros(10, np.complex64))          # a multi-link stream is not fed through the one-link call
    finally:
        h.close()


@pytest.mark.gpu
def test_library_matches_the_committed_digests(O, W):
    """The CUDA library against tests/golden/oracle_regression.json directly: TX IQ of every MCS, and for the golden
    capture the frame table, decisions, equalised points and PSDUs under every equalizer, hard and soft."""
    import hashlib
    import json
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_regression.json")))

    def sha(a):
        return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()

    rng = np.random.default_rng(2024)
    h = W.Handle(max_samples=1 << 20, max_frames=256, want_carrier=True)
    try:
        for enc in range(8):
            psdu = make_psdu(O, rng, 100 + 150 * enc, seq=enc)
            iq, _ = h.tx([psdu], enc=enc, seed=[17 + enc])
            assert sha(iq) == gold["tx"][str(enc)]["iq_sha256"], enc
        specs = [(e, 60 + 90 * e) for e in range(8)] + [(7, 1528), (3, 296)]
        taps = ((0, 1.0), (1, 0.4 * np.exp(1j * 1.0)), (3, 0.2 * np.exp(-2j)))
        y, _ = make_capture(O, np.random.default_rng(7), specs, snr_db=24, cfo=0.009, taps=taps, seed=5, gap=900)
        assert sha(y) == gold["capture_sha256"]
        for algo in range(4):
            for soft in (False, True):
                h.set_param(W.wifi_b200.P_CHAN_EST, algo)
                h.set_param(W.wifi_b200.P_SOFT_DECISION, int(soft))
                res = h.rx_batch(y)
                g = gold["rx"]["algo%d_%s" % (algo, "soft" if soft else "hard")]
                f = res.frames
                for k, name in (("trigger", "triggers"), ("frame_start", "frame_start"), ("encoding", "encoding"), ("length", "length"), ("crc_ok", "crc_ok")):
                    assert [int(v) for v in f[k]] == g[name], (algo, soft, k)
                assert sha(np.stack([f["freq_short"], f["freq_long"]])) == g["freq_sha256"]
                rows, car = h.rows(carrier=True)
                # the library reserves row ranges per frame; the oracle's rows are the used ones back to back
                used = np.concatenate([np.arange(int(r["row_off"]), int(r["row_off"]) + int(r["n_rows"])) for r in f]) if len(f) else np.zeros(0, int)
                assert sha(rows[used]) == g["rows_sha256"] and sha(car[used]) == g["carrier_sha256"], (algo, soft)
                assert hashlib.sha256(b"".join(res.pdus())).hexdigest() == g["pdus_sha256"]
    finally:
        h.close()


@pytest.mark.gpu
def test_maximum_and_minimum_frame_sizes(O, W):
    """The limits of [UPSTREAM] utils.h: MAX_PSDU_SIZE 1528 at BPSK 1/2 is MAX_SYM 511 symbols (41281 samples, the longest
    PPDU: its burst fills sync_short's 43200-sample COPY almost completely); BPSK 3/4 goes through k_pack (36 data bits
    per symbol do not fill whole trellis words); the shortest PSDUs (an FCS alone: 4 bytes, and 5 bytes).  Batch and streaming."""
    rng = np.random.default_rng(123)
    specs = [(0, 1528), (1, 1528), (0, 1), (5, 2), (7, 5), (6, 1528)]
    y, psdus = make_capture(O, rng, specs, snr_db=26, cfo=0.005, seed=2, gap=1500)
    assert O.n_sym(0, 1528) == 511
    ref = O.rx(y, algo=0)
    h = W.Handle(max_samples=1 << 18, max_frames=64, want_carrier=True)
    try:
        res = h.rx_batch(y)
        assert_frames_equal(res, ref)
        assert res.pdus() == ref.pdus()
        ok = {int(f["length"]) for f in res.frames if f["crc_ok"]}
        assert {1528, 4, 5} <= ok
        assert int(res.frames["frame_symbols"].max()) == 511 and int(res.frames["burst_len"].max()) >= 41281
        want = [(int(f["trigger"]), ref.psdu(i)[:-4]) for i, f in enumerate(ref.frames) if f["crc_ok"]]
        got = []
        for pos in range(0, y.size, 30000):
            h.rx_push(y[pos:pos + 30000], flush=(pos + 30000 >= y.size))
            got += h.rx_pop()
        assert [(int(f["trigger"]), d) for f, d in got] == want
        # one byte more than the mapper accepts
        with pytest.raises(W.WifiB200Error):
            h.tx([bytes(1529)], enc=0)
    finally:
        h.close()
