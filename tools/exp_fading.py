"""Fading channel measurements on one GPU, written as JSON to OUT/r03_fading_channel.json.

1. Generation cost at the bench's geometry (74 links x 512 frames of 64-QAM 3/4 with 1528-byte PSDUs, 229.6 Msamples):
   k_channel (one static tap) against k_channel_fading (3 taps of an exponential power-delay profile, 8 sinusoids each,
   Doppler 5e-4 cycles/sample), both on the same TX output and segment table.  Kernel times come from a torch.profiler
   trace, call times (descriptor copy + kernel + synchronise) from CUDA events; >= 20 launches each after a warm-up.
   The static SASS size of the per-sinusoid loop body is counted from cuobjdump.
2. What the equalizers buy under Doppler: PER of LS, LMS, COMB, STA (hard) and LS (soft) for QPSK 1/2 and 64-QAM 3/4 with
   1528-byte PSDUs over the same 3-tap channel, independent per frame, Doppler {0, 1e-4, 5e-4, 2e-3} x SNR {10, 20, 30} dB.

    python tools/exp_fading.py --out DIR
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PDP = ((0, 1.0), (1, np.exp(-1.0)), (2, np.exp(-2.0)))          # exponential power-delay profile, normalised below
PDP = tuple((d, p / sum(q for _, q in PDP)) for d, p in PDP)
N_SIN = 8
GAIN = 0.6


def device_record(torch):
    rec = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True, timeout=30)
        rec["nvidia_smi"] = out.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError) as e:
        rec["nvidia_smi"] = "unavailable: %s" % e
    return rec


def geometry(n_links, fpl, flen, gap, lead):
    n = n_links * fpl
    stride = flen + gap
    link_len = lead + fpl * stride
    f = np.arange(n)
    out_off = (f // fpl) * link_len + lead + (f % fpl) * stride
    return n, stride, link_len, out_off


def tables(W, n, flen, stride, out_off, snr_db, doppler, seed):
    """Segment table of the bench recipe (gain 0.6, per-frame CFO, Philox AWGN) and one fading record per frame."""
    w = W.wifi_b200
    rng = np.random.default_rng(seed)
    seg = np.zeros(n, w.CHANSEG_DTYPE)
    seg["in_off"] = np.arange(n) * flen
    seg["in_len"], seg["n"], seg["out_off"] = flen, stride, out_off
    seg["n0"] = out_off
    seg["gain"], seg["noise_sigma"], seg["seed"] = GAIN, GAIN * 10 ** (-snr_db / 20), seed
    seg["cfo"] = rng.uniform(-0.0025 * 2 * np.pi, 0.0025 * 2 * np.pi, n)
    fad = np.zeros(n, w.FADING_DTYPE)
    fad["n_taps"], fad["n_sin"], fad["doppler"] = len(PDP), N_SIN, doppler
    for t, (d, p) in enumerate(PDP):
        fad["delay"][:, t], fad["power"][:, t] = d, p
    fad["t0"], fad["seed"], fad["stream"] = out_off, seed + 1, np.arange(n)
    return seg, fad


def static_loop_size(so):
    """Static instruction count of k_channel_fading's per-sinusoid loop: the innermost backward branch whose body holds
    the NCO's int -> float conversions, divided by their number (the compiler unrolls the loop)."""
    try:
        sass = subprocess.check_output(["cuobjdump", "-sass", so], text=True, timeout=300)
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": str(e)}
    m = re.search(r"Function : (\S*k_channel_fading\S*)\n(.*?)(?=\n\s*Function :|\Z)", sass, re.S)
    if not m:
        return {"error": "k_channel_fading not found"}
    ins = [(int(a, 16), t.strip()) for a, t in re.findall(r"/\*([0-9a-f]{4,})\*/\s+([^;]*);", m.group(2))]
    best = None
    for addr, text in ins:
        b = re.search(r"BRA(?:\.U)?\s+(?:!?U?P\d,\s*)?0x([0-9a-f]+)", text)
        if not b or int(b.group(1), 16) >= addr:
            continue
        body = [t for a, t in ins if int(b.group(1), 16) <= a <= addr]
        k = sum("I2FP" in t or "I2F" in t.split()[0] for t in body)
        if k and (best is None or len(body) < best[0]):
            best = (len(body), k)
    if best is None:
        return {"error": "loop not found"}
    return {"instructions_in_loop": best[0], "sinusoids_per_iteration": best[1],
            "static_instructions_per_sinusoid": best[0] / best[1], "note": "static SASS count (cuobjdump), not a profile"}


def time_kernels(torch, h, call, names, reps, trace_dir):
    from torch.profiler import ProfilerActivity, profile
    stream = torch.cuda.ExternalStream(h.stream)
    res = {}
    for name, fn in call.items():
        fn()
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        res[name] = {"call_ms": e0.elapsed_time(e1) / reps}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for name, fn in call.items():
            for _ in range(reps):
                fn()
        torch.cuda.synchronize()
    path = os.path.join(trace_dir, "trace.json")
    prof.export_chrome_trace(path)
    ev = json.load(open(path))["traceEvents"]
    for name, kname in names.items():
        d = [e["dur"] for e in ev if e.get("cat") == "kernel" and re.search(r"\b%s\b" % kname, e.get("name", ""))]
        res[name].update(kernel_launches=len(d), kernel_ms=float(np.mean(d)) / 1e3 if d else None,
                         kernel_ms_min=float(np.min(d)) / 1e3 if d else None, kernel_ms_max=float(np.max(d)) / 1e3 if d else None)
    return res


def part1(torch, W, B, reps):
    w = W.wifi_b200
    n_links, fpl = 74, 512
    B.ENC, B.PSDU_LEN, B.N_DBPS = 7, 1528, 216
    flen = B.frame_samples()
    n, stride, link_len, out_off = geometry(n_links, fpl, flen, B.GAP, B.LEAD)
    total = n_links * link_len
    h = W.Handle(max_samples=1 << 20, max_frames=n + 1024)
    try:
        psdus = B.make_psdus(n, 1000)
        tx = torch.empty(2 * n * flen, dtype=torch.float32, device="cuda")
        tot, _ = h.tx_dev(psdus, tx.data_ptr(), n * flen, enc=7)
        assert tot == n * flen
        cap = torch.zeros(2 * total, dtype=torch.float32, device="cuda")
        seg, fad = tables(W, n, flen, stride, out_off, 30.0, 5e-4, 1000)
        stat = seg.copy()
        stat["n_taps"], stat["tap_re"][:, 0] = 1, 1.0
        calls = {"k_channel": lambda: h.channel_dev(tx.data_ptr(), cap.data_ptr(), stat),
                 "k_channel_fading": lambda: h.channel_fading_dev(tx.data_ptr(), cap.data_ptr(), seg, fad)}
        with tempfile.TemporaryDirectory() as td:
            res = time_kernels(torch, h, calls, {k: k for k in calls}, reps, td)
        out_samples = n * stride
        for k in res:
            if res[k]["kernel_ms"]:
                res[k]["gsamples_per_s"] = out_samples / (res[k]["kernel_ms"] * 1e-3) / 1e9
        return {"geometry": {"links": n_links, "frames_per_link": fpl, "encoding": "64-QAM 3/4", "psdu_bytes": 1528,
                             "segments": n, "samples_generated": out_samples, "capture_samples": total,
                             "fading": {"pdp": PDP, "n_sin": N_SIN, "doppler": 5e-4}, "launches_timed": reps},
                "timing": res, "sass": static_loop_size(W.build.SO)}
    finally:
        h.close()


def part2(torch, W, B, n_links, fpl):
    w = W.wifi_b200
    out = []
    for enc, label in ((2, "QPSK 1/2"), (7, "64-QAM 3/4")):
        B.ENC, B.PSDU_LEN = enc, 1528
        B.N_DBPS = {2: 48, 7: 216}[enc]
        flen = B.frame_samples()
        n, stride, link_len, out_off = geometry(n_links, fpl, flen, B.GAP, B.LEAD)
        h = W.Handle(max_samples=n_links * link_len + 1024, max_frames=n + n_links + 1024)
        try:
            psdus = B.make_psdus(n, 2000 + enc)
            tx = torch.empty(2 * n * flen, dtype=torch.float32, device="cuda")
            tot, _ = h.tx_dev(psdus, tx.data_ptr(), n * flen, enc=enc)
            assert tot == n * flen, (tot, n * flen)
            cap = torch.zeros(2 * n_links * link_len, dtype=torch.float32, device="cuda")
            lo = (np.arange(n_links + 1) * link_len).astype(np.uint64)
            sent = {p[:-4] for p in psdus}
            for doppler in (0.0, 1e-4, 5e-4, 2e-3):
                for snr in (10.0, 20.0, 30.0):
                    seg, fad = tables(W, n, flen, stride, out_off, snr, doppler, 3000 + enc)
                    cap.zero_()
                    h.channel_fading_dev(tx.data_ptr(), cap.data_ptr(), seg, fad)
                    row = {"mcs": label, "doppler": doppler, "snr_db": snr, "frames": n}
                    for name, algo, soft in (("LS", 0, 0), ("LMS", 1, 0), ("COMB", 2, 0), ("STA", 3, 0), ("LS_soft", 0, 1)):
                        h.set_param(w.P_CHAN_EST, algo)
                        h.set_param(w.P_SOFT_DECISION, soft)
                        r = h.rx_batch_dev(cap.data_ptr(), lo, fetch=True)
                        good = sum(1 for p in r.pdus() if p in sent)
                        row[name] = round(1.0 - good / n, 4)
                    out.append(row)
                    print(json.dumps(row), flush=True)
        finally:
            h.close()
    return {"frames_per_cell": n_links * fpl, "channel": {"pdp": PDP, "n_sin": N_SIN, "per_frame": "independent (one stream per frame)",
                                                           "cfo": "uniform +-0.0025 cycles/sample per frame", "gain": GAIN,
                                                           "snr": "noise_sigma = gain * 10^(-snr/20), as bench.py"},
            "per": out, "per_definition": "1 - (CRC-ok PSDUs that were sent) / frames sent"}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--per-links", type=int, default=8)
    ap.add_argument("--per-frames", type=int, default=256)
    a = ap.parse_args()
    if a.reps < 20:
        ap.error("--reps must be >= 20")
    import torch
    if not torch.cuda.is_available():
        sys.exit("exp_fading.py measures on a GPU; none is visible")
    import importlib
    W = importlib.import_module("gnuradio-wifi-imagetransfer_b200")
    import bench as B
    os.makedirs(a.out, exist_ok=True)
    t = time.time()
    rec = device_record(torch)
    rec["generation"] = part1(torch, W, B, a.reps)
    print(json.dumps(rec["generation"]["timing"]), flush=True)
    rec["per_sweep"] = part2(torch, W, B, a.per_links, a.per_frames)
    rec["wall_s"] = round(time.time() - t, 1)
    with open(os.path.join(a.out, "r03_fading_channel.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", os.path.join(a.out, "r03_fading_channel.json"))


if __name__ == "__main__":
    main()
