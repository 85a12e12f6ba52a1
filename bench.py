#!/usr/bin/env python
"""bench.py -- RX throughput of the 802.11a/g baseband on B200 (BASELINE.json metric:
"RX Msamples/s and decoded Mb/s per GPU, 64-QAM 3/4").

Workload (BASELINE.json configs[2], SURVEY.md 8d "C3"): synthetic 20 MHz baseband, 64-QAM 3/4,
1528-byte PSDUs (57 OFDM symbols, 4961 samples) back to back with 1100-sample idle gaps,
74 links x 512 frames per GPU (37888 frames = 148 SMs x 4 blocks x 64: whole waves of the Viterbi kernel),
AWGN at 30 dB, LMS equalizer, hard-decision Viterbi.  The capture is generated on the GPU by
the library's own TX chain and Philox channel and is far larger than L2 (no flush needed).

One "step" = one wifi_b200_rx_batch_dev pass over the whole resident capture (all links).
`value` = complex samples consumed per second, all ranks (device-resident input).
`e2e`   = the same pass through wifi_b200_rx_batch with pinned HOST input and host results.
`--impl reference` times the CPU oracle (a port of the reference algorithm; the real
gr-ieee802-11 flowgraph cannot be built here) on a bounded sample with all host threads.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENC = 7
PSDU_LEN = 1528
GAP = 1100
SNR_DB = 30.0
ALGO = 1          # LMS
LEAD = 128
TX_INFO = {}
SC16_SCALE = 1.0 / 4096.0   # int16 wire format of the e2e sc16 line: full scale +-8, quantisation noise ~78 dB below the signal


def set_workload(name):
    global ENC, PSDU_LEN, GAP, SNR_DB, N_DBPS, TAPS, WORKLOAD_DESC
    if name == "c2":
        ENC, PSDU_LEN, GAP, SNR_DB, N_DBPS = 4, 1500, 1100, 25.0, 96
        TAPS = True
        WORKLOAD_DESC = "BASELINE configs[1]: one 20 Msps stream, 16-QAM 1/2, 1500-byte PSDUs (126 symbols, 10481 samples) + 1100-sample gaps, per-frame CFO, 3-tap multipath, 25 dB"


N_DBPS = 216
TAPS = False
WORKLOAD_DESC = "BASELINE configs[2]: 54 Mb/s 64-QAM 3/4 batched RX, 1528-byte PSDUs (57 symbols, 4961 samples) + 1100-sample gaps, AWGN 30 dB"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--links", type=int, default=74, help="independent links per GPU (74 x 512 frames = 148 SMs x 4 blocks x 64 trellises: whole waves of k_viterbi)")
    ap.add_argument("--frames-per-link", type=int, default=512)
    ap.add_argument("--algo", type=int, default=ALGO)
    ap.add_argument("--workload", default="c3", choices=["c3", "c2"], help="c3 = BASELINE configs[2] (metric workload); c2 = configs[1]: one 10 s 20 Msps stream, 16-QAM 1/2, CFO + 3-tap multipath")
    ap.add_argument("--soft", action="store_true", help="soft-decision mode (extension, DESIGN.md 9)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--strict", action="store_true", help="fail the run if the time-sharded union differs from the single-GPU table (it is always reported)")
    ap.add_argument("--no-time-shard", action="store_true", help="skip the time-sharded section (one capture cut into overlapping segments across the ranks)")
    ap.add_argument("--ts-frames", type=int, default=151552, help="frames of the single-link capture the time-sharded section cuts across the ranks (the same at every N: strong scaling)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--viterbi-form", type=int, default=0, help="pin the Viterbi kernel form of the main handle (WIFI_P_VITERBI_FORM: 1 warp, 2 four lanes, 3 thread per trellis; 0 = by frame count)")
    ap.add_argument("--cpu-frames", type=int, default=8192, help="frames of the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (frame table, "
                    "decoded PSDU bytes; a fixed, seeded sample beyond %d frames / %d PSDUs) as DIR/<name>.npy in float64 / float32; "
                    "rank 0 only" % (DUMP_FRAMES, DUMP_PSDUS))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_FRAMES, DUMP_PSDUS, PSDU_MAX = 65536, 8192, 1528     # PSDU_MAX: the largest PSDU the receiver decodes
# --dump-outputs writes at most 65536 x 20 x 8 B (frame table) + 8192 x 1528 x 4 B (PSDU bytes) + 8192 x 8 B = 61 MB


def dump_outputs(path, frames, psdu):
    """--dump-outputs: the results of the last timed step as a caller receives them -- every field of the frame table and
    the decoded PSDU bytes -- so that two builds can be compared output for output on the same inputs.  Integer and float
    fields go out as float64 (exact), bytes as float32 with -1 where a frame has no decoded byte.  Beyond DUMP_FRAMES frames
    the table is a sample drawn with a fixed seed (frame_index.npy says which rows), and the PSDU bytes are those of at
    most DUMP_PSDUS of its rows (psdu_index.npy)."""
    os.makedirs(path, exist_ok=True)
    rng = np.random.default_rng(0)
    n = len(frames)
    rows = np.arange(n) if n <= DUMP_FRAMES else np.sort(rng.choice(n, DUMP_FRAMES, replace=False))
    sel = rows if len(rows) <= DUMP_PSDUS else np.sort(rng.choice(rows, DUMP_PSDUS, replace=False))
    out = {"frame_index": rows, "psdu_index": sel}
    for k in frames.dtype.names:
        out["frame_" + k] = frames[k][rows]
    b = np.full((len(sel), PSDU_MAX), -1.0, np.float32)
    for j, i in enumerate(sel):
        p = psdu(int(i))
        if p is not None:
            b[j, :len(p)] = np.frombuffer(p, np.uint8)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v.astype(np.float64))
    np.save(os.path.join(path, "psdu_bytes.npy"), b)


def frame_samples():
    n_sym = -(-(16 + 8 * PSDU_LEN + 6) // N_DBPS)
    return 80 * (5 + n_sym) + 1


def make_psdus(n, seed):
    import zlib
    rng = np.random.default_rng(seed)
    out = []
    hdr = bytes([0x08, 0, 0, 0]) + b"\x42" * 6 + b"\x23" * 6 + b"\xff" * 6
    pay = rng.integers(0, 256, (n, PSDU_LEN - 28), dtype=np.uint8)
    for i in range(n):
        body = hdr + int((i & 0xfff) << 4).to_bytes(2, "little") + pay[i].tobytes()
        out.append(body + zlib.crc32(body).to_bytes(4, "little"))
    return out


def build_capture(h, W, torch, n_links, fpl, seed):
    """TX + channel on the GPU.  Returns (capture tensor [2*N] f32, link_off, psdus)."""
    n = n_links * fpl
    flen = frame_samples()
    stride = flen + GAP
    link_len = LEAD + fpl * stride
    psdus = make_psdus(n, seed)
    tx = torch.empty(2 * n * flen, dtype=torch.float32, device="cuda")
    tot, off = h.tx_dev(psdus, tx.data_ptr(), n * flen, enc=ENC)
    assert tot == n * flen
    # the TX chain is not on the metric path; its rate is reported beside it (PSDU blob over PCIe, IQ stays on the device)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h.tx_dev(psdus, tx.data_ptr(), n * flen, enc=ENC)
    torch.cuda.synchronize()
    TX_INFO.update(value=n * flen / (time.perf_counter() - t0) / 1e6, unit="Msamples/s", frames=n,
                   how="wifi_b200_tx_dev: mapper .. cyclic prefixer for every frame of the capture, host PSDUs in, device IQ out")
    cap = torch.zeros(2 * n_links * link_len, dtype=torch.float32, device="cuda")
    rng = np.random.default_rng(seed + 1)
    seg = np.zeros(n + n_links, W.wifi_b200.CHANSEG_DTYPE)
    f = np.arange(n)
    seg["in_off"][:n] = off[:-1]
    seg["in_len"][:n] = flen
    seg["out_off"][:n] = (f // fpl) * link_len + LEAD + (f % fpl) * stride
    seg["n"][:n] = stride
    # noise-only lead-in of every link
    seg["in_len"][n:] = 0
    seg["out_off"][n:] = np.arange(n_links) * link_len
    seg["n"][n:] = LEAD
    seg["n0"] = seg["out_off"]
    seg["gain"] = 0.6
    seg["noise_sigma"] = 0.6 * 10 ** (-SNR_DB / 20)
    seg["cfo"][:n] = rng.uniform(-0.0025 * 2 * np.pi, 0.0025 * 2 * np.pi, n)   # |eps| <= 50 kHz at 20 Msps
    seg["phase0"][:n] = rng.uniform(-np.pi, np.pi, n)
    seg["n_taps"] = 1
    seg["tap_re"][:, 0] = 1.0
    if TAPS:   # h = [1, 0.4 e^{j phi1}, 0, 0.2 e^{j phi2}] / |h| per frame (SURVEY 8d C2)
        p1, p2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
        nrm = 1.0 / np.sqrt(1 + 0.16 + 0.04)
        seg["n_taps"][:n] = 3
        seg["delay"][:n, 1], seg["delay"][:n, 2] = 1, 3
        seg["tap_re"][:n, 0] = nrm
        seg["tap_re"][:n, 1], seg["tap_im"][:n, 1] = 0.4 * nrm * np.cos(p1), 0.4 * nrm * np.sin(p1)
        seg["tap_re"][:n, 2], seg["tap_im"][:n, 2] = 0.2 * nrm * np.cos(p2), 0.2 * nrm * np.sin(p2)
    seg["seed"] = seed
    seg["stream"] = 0
    h.channel_dev(tx.data_ptr(), cap.data_ptr(), seg)
    del tx
    link_off = (np.arange(n_links + 1) * link_len).astype(np.uint64)
    return cap, link_off, psdus


def run_time_sharded(W, torch, dist, args, rank, world, local):
    """SURVEY 8e (ii) on hardware: ONE long single-link capture (the same on every rank: the TX chain and the Philox channel
    are deterministic) is cut into `world` overlapping segments (sharding.shard_stream, overlap 44128 samples); every rank
    decodes its segment, the frame records are all-gathered over NCCL, every rank checks that it joined the sequential
    receiver's state (sharding.reconcile; a rank that did not decodes again from a known state), frames are owned by the
    segment whose core region holds their trigger.  Rank 0 also decodes the whole capture alone and asserts that the union
    of the owned frames IS that table.  Strong scaling: the total work is fixed."""
    S = W.sharding
    fpl = args.ts_frames
    flen = frame_samples()
    n_total = LEAD + fpl * (flen + GAP)
    h = W.Handle(device=local, chan_est=args.algo, encoding=ENC, max_samples=n_total + 1024, max_frames=fpl + 1024, soft_decision=args.soft)
    cap, link_off, _ = build_capture(h, W, torch, 1, fpl, seed=2000)          # identical on every rank
    torch.cuda.synchronize()
    segs = S.shard_stream(n_total, world)
    dev = torch.device("cuda", local)
    decode_ms = [0.0]
    last_stage = {}

    problems = []

    def decode(lo, end, st, final):
        # a rank that fails must not leave the others waiting in the all-gather: it reports an empty table and the problem
        try:
            off = np.array([lo, end], np.uint64)
            if st is None:
                h.rx_batch_dev(cap.data_ptr(), off, final=final, fetch=False)
            else:
                state = np.zeros(1, W.wifi_b200.LINK_STATE_DTYPE)
                state["min_pos"], state["fo_carry"], state["hist"] = st["min_pos"], st["fo_carry"], st["hist"]
                h.rx_batch_dev_state(cap.data_ptr(), off, state, final=final, fetch=False)
            st_ = h.stage_times()
            last_stage.clear()
            last_stage.update({k: round(v, 3) for k, v in st_.items() if v})
            decode_ms[0] += sum(st_.values())
            return h.frames(reuse=True)                                          # 96 bytes per trigger; PSDUs stay on the device
        except Exception as ex:
            problems.append(repr(ex))
            return np.zeros(0, W.wifi_b200.FRAME_DTYPE)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    reps, warm = 5, 2
    own = owned_all = None
    phases = {}
    rounds = 0
    for it in range(warm + reps):
        if it == warm:
            barrier()
            decode_ms[0] = 0.0
            phases.clear()
            t0 = time.perf_counter()
        own, _tails, rounds = S.reconcile(decode, segs, rank, n_total, device=dev if world > 1 else None, max_rounds=world + 2, tail_rows=512, trace=phases)
    barrier()
    t_sh = (time.perf_counter() - t0) / reps
    dec_sh = decode_ms[0] / reps
    # the sequential answer: the whole capture in one call on one GPU (rank 0 checks, every rank times it)
    for _ in range(warm):
        h.rx_batch_dev(cap.data_ptr(), link_off, final=True, fetch=False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        h.rx_batch_dev(cap.data_ptr(), link_off, final=True, fetch=False)
        whole = h.frames()
    t_one = (time.perf_counter() - t0) / reps
    one_stage = {k: round(v, 3) for k, v in h.stage_times().items() if v}
    # outside the timed region: every rank's owned records travel to rank 0, which compares their union with its own decode
    owned_all = S.gather_owned(own, dev if world > 1 else None)
    equal = None
    if rank == 0:
        equal = S.same(np.concatenate(owned_all), S.records(whole, 0))
    tv = torch.tensor([t_sh, dec_sh, t_one], dtype=torch.float64, device="cuda")
    cnt = S.allreduce_stats(np.array([len(own), int(own[:, S.CRC].sum())], np.int64), device=dev if world > 1 else None)
    if world > 1:
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
    h.close()
    del cap
    if equal is False or problems:          # reported, loudly, but the headline line still goes out
        print("time_sharded: union == single-GPU table: %s, problems: %s" % (equal, problems), file=sys.stderr)
    if args.strict:
        assert equal is not False and not problems, "time-sharded frame table differs from the single-GPU table"
    t_sh, dec_sh, t_one = [float(v) for v in tv.tolist()]
    return {"capture": "one link, %d frames, %d samples (%.2f GB), the same on every rank" % (fpl, n_total, n_total * 8 / 1e9),
            "ranks": world, "overlap_samples": S.OVERLAP, "sharded_ms": 1e3 * t_sh, "sharded_decode_device_ms": dec_sh,
            "sharded_stage_ms_rank0_last_decode": dict(last_stage), "sharded_wall_ms_by_phase_rank0": {k: round(1e3 * v / reps, 3) for k, v in phases.items()}, "single_gpu_ms": 1e3 * t_one, "single_gpu_stage_ms": one_stage, "speedup_over_single_gpu": t_one / t_sh if t_sh else None,
            "value_msamples_per_s": n_total / t_sh / 1e6, "frames_owned_total": int(cnt[0]), "crc_ok_total": int(cnt[1]),
            "re_decode_rounds": rounds, "union_equals_single_gpu_table": equal, "problems": problems or None, "scaling": "strong",
            "collective": "per round two NCCL all_gathers of fixed-size buffers: the last 512 owned frame records of every rank (96 bytes each), then the ranks' verdicts; + one counter all_reduce" if world > 1 else "none (one rank)",
            "timing": "wall clock around sharding.reconcile (decode, record all-gather, join check), barrier + synchronize on both sides, max over ranks, mean of %d; the union check against rank 0's whole-capture decode runs outside it" % reps}


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp"

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)        # the sampler must not outlive bench.py, even when a section fails before stop()
        except Exception:
            self.p = None

    def stop(self, t_begin=None, t_end=None):
        """t_begin / t_end (time.time()): keep the samples taken inside the timed region (nvidia-smi needs a few hundred
        milliseconds to start, so the sampler is launched well before it); all samples if none fall inside."""
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.p:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 7:
                continue
            try:
                row = (float(c[0]), float(c[1]), {nm for k, nm in enumerate(names) if c[3 + k].lower().startswith("active")})
            except ValueError:
                continue
            ts = None
            if len(c) >= 8:
                try:
                    ts = datetime.datetime.strptime(c[7], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except ValueError:
                    ts = None
            rows.append((ts,) + row)
        inside = [r for r in rows if r[0] is not None and t_begin is not None and t_begin - 0.02 <= r[0] <= t_end + 0.02]
        use = inside or rows
        if use:
            reasons = set().union(*[r[3] for r in use])
            out = {"sm_mhz": float(np.median([r[1] for r in use])), "sm_max_mhz": float(max(r[2] for r in use)), "reasons": sorted(reasons),
                   "samples": len(use), "samples_inside_timed_region": len(inside)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def config_dict(args, n_links, fpl):
    return {"workload": WORKLOAD_DESC,
            "equalizer": ["LS", "LMS", "COMB", "STA"][args.algo], "decisions": "soft" if getattr(args, "soft", False) else "hard", "links_per_gpu": n_links, "frames_per_link": fpl,
            "samples_per_gpu": int(n_links * (LEAD + fpl * (frame_samples() + GAP))),
            "l2_policy": "input (%.2f GB per GPU) larger than L2, no flush" % (n_links * (LEAD + fpl * (frame_samples() + GAP)) * 8 / 1e9),
            "parallelism": "links sharded across GPUs, no data-path collective"}


def build_capture_cpu(O, n_links, fpl, seed):
    """The b200 arm's capture recipe (build_capture) restated with the oracle's TX and Philox channel: the same frame
    layout, per-frame CFO / phase (/ taps) drawn the same way, the same noise convention."""
    n = n_links * fpl
    flen = frame_samples()
    stride = flen + GAP
    link_len = LEAD + fpl * stride
    psdus = make_psdus(n, seed)
    rng = np.random.default_rng(seed + 1)
    cfo = rng.uniform(-0.0025 * 2 * np.pi, 0.0025 * 2 * np.pi, n)
    ph0 = rng.uniform(-np.pi, np.pi, n)
    if TAPS:
        p1, p2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
        nrm = 1.0 / np.sqrt(1 + 0.16 + 0.04)
    sigma = 0.6 * 10 ** (-SNR_DB / 20)
    x = np.zeros(n_links * link_len, np.complex64)
    for l in range(n_links):
        x[l * link_len:l * link_len + LEAD] = O.channel(np.zeros(LEAD, np.complex64), n0=l * link_len, gain=0.6, noise_sigma=sigma, seed=seed)
    buf = np.zeros(stride, np.complex64)
    for f in range(n):
        buf[:flen] = O.tx_frame(psdus[f], ENC, 1 + f % 127)
        taps = ((0, 1.0),)
        if TAPS:
            taps = ((0, nrm), (1, 0.4 * nrm * np.exp(1j * p1[f])), (3, 0.2 * nrm * np.exp(1j * p2[f])))
        o = (f // fpl) * link_len + LEAD + (f % fpl) * stride
        x[o:o + stride] = O.channel(buf, n0=o, gain=0.6, cfo=float(cfo[f]), phase0=float(ph0[f]), noise_sigma=sigma, taps=taps, seed=seed)
    off = (np.arange(n_links) * link_len).astype(np.int64)
    return x, off, np.full(n_links, link_len, np.int64), psdus


def run_reference(args, out_fd):
    """CPU arm: the oracle (a port of the reference algorithm; gr-ieee802-11 itself cannot be built here) on all host
    threads.  Each step is a BOUNDED sample of the b200 arm's workload -- the same frames, gaps, SNR and per-frame CFO,
    one link per host thread, fewer frames per link -- and the line's config says what ran."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    threads = os.cpu_count() or 1
    fpl = min(args.frames_per_link, 96)
    n_links = max(threads, 1)
    x, off, ln, _ = build_capture_cpu(O, n_links, fpl, seed=1000)
    times = []
    ok = 0
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = O.rx_links(x, off, ln, n_threads=threads, algo=args.algo, want_carrier=False, soft=args.soft)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
            ok = int(r.frames["crc_ok"].sum())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r.frames, r.psdu)
    t = float(np.sum(times))
    msps = x.size * len(times) / t / 1e6
    cfg = config_dict(args, n_links, fpl)
    cfg["l2_policy"] = "CPU arm: not applicable"
    cfg["parallelism"] = "one link per host thread (%d threads)" % threads
    cfg["bounded_sample_of"] = "the b200 arm's %d links x %d frames per GPU: same frame layout, SNR, per-frame CFO and phase, %d links x %d frames here" % (
        args.links, args.frames_per_link, n_links, fpl)
    line = {"impl": "reference", "metric": "rx_msamples_per_s", "value": msps, "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / len(times), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32+u8", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": msps, "unit": "Msamples/s", "cores": threads, "kind": "port",
                             "sample": "%d links x %d frames (%d samples) per step, one link per host thread" % (n_links, fpl, x.size)},
            "e2e": {"value": msps, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "crc_ok_per_step": ok, "frames_per_step": n_links * fpl}
    line["decoded_mbps"] = ok * (PSDU_LEN - 4) * 8 / (t / len(times)) / 1e6
    _emit(out_fd, line)


def _claim_stdout():
    """Libraries write banners to file descriptor 1 (NCCL prints its version there); the contract is ONE
    JSON line on stdout.  Everything else goes to stderr, the line goes to the saved descriptor."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return real


def _emit(real_fd, line):
    sys.stdout.flush()
    os.write(real_fd, (json.dumps(line) + "\n").encode())


def main():
    args = parse()
    out_fd = _claim_stdout()
    set_workload(args.workload)
    if args.workload == "c2" and args.links == 74 and args.frames_per_link == 512:
        args.links, args.frames_per_link = 1, 17270          # 10 s at 20 Msps
    if args.impl == "reference":
        run_reference(args, out_fd)
        return
    import torch
    import torch.distributed as dist
    import wifi_b200 as pkg
    W = pkg
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # every rank keeps to its own share of the host cores: the page-locked capture of the e2e section is first touched
        # (and, where the box shows NUMA nodes, placed) from the cores that will feed this rank's GPU
        cpus = sorted(os.sched_getaffinity(0))
        per = len(cpus) // world
        if per >= 1:
            os.sched_setaffinity(0, cpus[local * per:(local + 1) * per])
    n_links, fpl = args.links, args.frames_per_link
    n = n_links * fpl
    flen = frame_samples()
    n_samples = n_links * (LEAD + fpl * (flen + GAP))
    h = W.Handle(device=local, chan_est=args.algo, encoding=ENC, max_samples=n_samples + 1024, max_frames=n + n_links + 1024,
                 soft_decision=args.soft)
    if args.viterbi_form:
        h.set_param(W.wifi_b200.P_VITERBI_FORM, args.viterbi_form)
    sampler = ClockSampler(local) if rank == 0 else None           # started early: nvidia-smi takes a while to produce its first line
    cap, link_off, psdus = build_capture(h, W, torch, n_links, fpl, seed=1000 + rank)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        h.rx_batch_dev(cap.data_ptr(), link_off, final=True, fetch=False)

    for _ in range(args.warmup):
        step()
    barrier()
    stage_acc = {}
    barrier()
    t0 = time.perf_counter()
    wall0 = time.time()
    for _ in range(args.steps):
        step()                      # synchronises its own stream before returning
        for k, v in h.stage_times().items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    # the library times every stage with CUDA events on its own stream; the step time on the device is
    # their sum, the host wall clock adds launch/sync gaps -- report the larger (honest) one
    dev_ms = sum(stage_acc.values())
    elapsed = max(wall, dev_ms / 1e3)
    clocks = sampler.stop(wall0, time.time()) if sampler else None
    res = h.results()
    st_frames = len(res.frames)
    st_ok = int(res.frames["crc_ok"].sum())
    # parity property at full size: every CRC-ok PDU is one of the PSDUs that were sent
    sent = {p[:-4] for p in psdus}
    pd = res.pdus()
    assert all(p in sent for p in pd[:2000]), "decoded PDU not among the transmitted ones"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res.frames, res.psdu)
    tvec = torch.tensor([elapsed], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([n_samples, st_frames, st_ok, st_ok * (PSDU_LEN - 4)], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(tvec, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)     # the only collective: counters over NCCL
    elapsed_max = float(tvec.item())
    tot_samples, tot_frames, tot_ok, tot_bytes = [int(v) for v in cnt.tolist()]
    value = tot_samples * args.steps / elapsed_max / 1e6
    mbps = tot_bytes * 8 * args.steps / elapsed_max / 1e6

    # ---- e2e: host buffers through the C ABI (H2D + D2H inside the timed region) ----
    e2e = None
    if not args.no_e2e:
        import threading
        # page-locked host capture from the library's own allocator: first touched on the cores next to this rank's GPU
        hn = h.host_alloc(cap.numel() // 2, np.complex64)
        torch.from_numpy(hn.view(np.float32)).copy_(cap)       # device -> page-locked host, no temporary
        torch.cuda.synchronize()
        host = hn
        parts = 4 if n_links >= 4 else 1
        bounds = [n_links * i // parts for i in range(parts + 1)]
        part_samples = max(int(link_off[bounds[i + 1]] - link_off[bounds[i]]) for i in range(parts))
        part_frames = (max(bounds[i + 1] - bounds[i] for i in range(parts))) * (fpl + 1) + 1024
        hs = [W.Handle(device=local, chan_est=args.algo, encoding=ENC, max_samples=part_samples + 1024, max_frames=part_frames, soft_decision=args.soft) for _ in range(2)]
        tot = {"frames": 0, "store": 0, "ok": 0}
        lock = threading.Lock()

        mode = {"sc16": None}

        def worker(k, count):
            for i in range(k, parts, 2):
                if mode["sc16"] is not None:
                    hs[k].rx_batch_sc16(mode["sc16"], SC16_SCALE, link_off[bounds[i]:bounds[i + 1] + 1], final=True, fetch=False)
                else:
                    hs[k].rx_batch(hn, link_off[bounds[i]:bounds[i + 1] + 1], final=True, fetch=False)   # frames + PSDU store land in pinned host memory
                if count:
                    c = hs[k].counts()
                    with lock:
                        tot["frames"] += c["n_frames"]
                        tot["store"] += c["psdu_store_bytes"]
                        tot["ok"] += c["n_pdus"]

        def e2e_step(count=False):
            th = [threading.Thread(target=worker, args=(k, count)) for k in range(2 if parts > 1 else 1)]
            for t_ in th:
                t_.start()
            for t_ in th:
                t_.join()

        # headline: ONE wifi_b200_rx_batch call per step on the pinned host capture.  The library cuts the links into
        # groups and overlaps the host->device copy of one group with the decode of the previous one and the copy of its
        # results back (three streams inside the handle); the frame table and the PSDU store land in pinned host memory.
        for _ in range(2):
            h.rx_batch(hn, link_off, final=True, fetch=False)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            h.rx_batch(hn, link_off, final=True, fetch=False)
        barrier()
        te = time.perf_counter() - t0
        c1 = h.counts()
        assert c1["n_pdus"] == st_ok, (c1, st_ok)          # same answers through the host path
        # for comparison: two handles driven from two host threads over four link groups (round 1's way to overlap)
        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(max(1, args.steps // 2)):
            e2e_step()
        barrier()
        t1 = (time.perf_counter() - t0) / max(1, args.steps // 2)
        e2e_step(count=True)
        assert tot["ok"] == st_ok, (tot, st_ok)
        tv = torch.tensor([te, t1], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        e2e = {"value": tot_samples * args.steps / float(tv[0].item()) / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": int(n_samples * 8), "d2h_bytes_per_step": int(c1["n_frames"] * 96 + c1["psdu_store_bytes"]),
               "decoded_mbps": tot_bytes * 8 * args.steps / float(tv[0].item()) / 1e6,
               "how": "one wifi_b200_rx_batch call per step on pinned host IQ (the library pipelines link groups: H2D, decode, D2H on three streams); frame table + PSDU store copied to pinned host memory",
               "single_call_value": tot_samples * args.steps / float(tv[0].item()) / 1e6,
               "two_handles_two_threads_value": tot_samples / float(tv[1].item()) / 1e6}
        # the same capture in the radio's wire format (int16 I/Q, converted on the GPU): half the PCIe bytes.
        # Reported beside the headline, not as it: the reference's samp_in port is complex float.
        try:
            h16 = torch.empty(cap.numel(), dtype=torch.int16, pin_memory=True)
            h16.copy_(torch.clamp(torch.round(cap / SC16_SCALE), -32768, 32767).to(torch.int16))
            torch.cuda.synchronize()
            a16 = h16.numpy()
            h.rx_batch_sc16(a16, SC16_SCALE, link_off, final=True, fetch=False)
            barrier()
            t0 = time.perf_counter()
            for _ in range(max(1, args.steps // 2)):
                h.rx_batch_sc16(a16, SC16_SCALE, link_off, final=True, fetch=False)
            barrier()
            t16 = (time.perf_counter() - t0) / max(1, args.steps // 2)
            tv16 = torch.tensor([t16], dtype=torch.float64, device="cuda")
            ok16 = torch.tensor([h.counts()["n_pdus"]], dtype=torch.int64, device="cuda")
            if world > 1:
                dist.all_reduce(tv16, op=dist.ReduceOp.MAX)
                dist.all_reduce(ok16, op=dist.ReduceOp.SUM)
            e2e["sc16_ingest"] = {"value": tot_samples / float(tv16.item()) / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": int(n_samples * 4),
                                  "crc_ok_per_step": int(ok16.item()),
                                  "how": "one wifi_b200_rx_batch_sc16 call per step: int16 I/Q over PCIe, x = float(i16) * scale on the GPU (extension; not the headline)"}
            del h16
        except Exception as ex:     # the headline must not depend on the extension
            e2e["sc16_ingest"] = {"error": repr(ex)}
        mode["sc16"] = None
        for x_ in hs:
            x_.close()
        # live form: one hundred continuous 20 Msps streams pushed chunk by chunk into ONE handle (what many SDR front-ends
        # feeding one GPU look like): two page-locked buffers used in turn, wifi_b200_rx_push_links_async for chunk k + 1
        # while wifi_b200_rx_push_wait decodes chunk k, bulk pop.  Stream l plays link l mod n_links of the capture.
        try:
            chunk, pushes, s_links = 262144, 6, 100
            link_len = int(link_off[1] - link_off[0])
            if link_len >= chunk * pushes:
                off = (np.arange(s_links + 1) * chunk).astype(np.uint64)
                hv = hn.reshape(n_links, link_len)
                src = np.arange(s_links) % n_links

                def live(wire):
                    """One handle, `pushes` chunks of every stream; wire = int16 I/Q (the radios' format) instead of complex64."""
                    hl = W.Handle(device=local, chan_est=args.algo, encoding=ENC, max_samples=s_links * (chunk + 131072) + 1024,
                                  max_frames=s_links * (chunk // 4096 + 16), soft_decision=args.soft)
                    # every chunk gets its own page-locked buffer, filled BEFORE the timed region (that is the radios' job): the
                    # timed loop is library calls only, back to back, so no copy hides behind untimed host work
                    if wire:
                        pins = [torch.empty(2 * s_links * chunk, dtype=torch.int16, pin_memory=True) for _ in range(pushes)]
                        blobs = [p_.numpy() for p_ in pins]
                        for k in range(pushes):
                            x = hv[src, k * chunk:(k + 1) * chunk].view(np.float32)
                            blobs[k].reshape(s_links, 2 * chunk)[:] = np.clip(np.rint(x * np.float32(1.0 / SC16_SCALE)), -32768, 32767).astype(np.int16)
                        push = lambda k, fl: hl.rx_push_links_sc16_async(blobs[k], SC16_SCALE, off, flush=fl)
                    else:
                        pins = [torch.empty(2 * s_links * chunk, dtype=torch.float32, pin_memory=True) for _ in range(pushes)]
                        blobs = [p_.numpy().view(np.complex64) for p_ in pins]
                        for k in range(pushes):
                            blobs[k].reshape(s_links, chunk)[:] = hv[src, k * chunk:(k + 1) * chunk]
                        push = lambda k, fl: hl.rx_push_links_async(blobs[k], off, flush=fl)

                    def drain():
                        n_ = 0
                        while True:
                            meta, _pd = hl.rx_pop_arrays(cap=8192, copy=False)
                            if not len(meta):
                                return n_
                            n_ += len(meta)

                    # untimed warm-up: the arena, the staging buffers and the pinned result mirrors are allocated on first use
                    for k in range(3):                     # three pending pushes: every staging slot is allocated here, not in the timed loop
                        push(k, k == 2)
                    for k in range(3):
                        hl.rx_push_wait()
                        drain()
                    hl.rx_reset()
                    n_pdu, push_ms, wait_ms, stage_last = 0, [], [], {}
                    barrier()
                    t_start = time.perf_counter()
                    push(0, False)
                    push(1, False)                         # two copies queued ahead: the copy engine never idles
                    for k in range(1, pushes + 1):
                        t0 = time.perf_counter()
                        if k + 1 < pushes:
                            push(k + 1, k + 1 == pushes - 1)
                        tw = time.perf_counter()
                        hl.rx_push_wait()
                        wait_ms.append(round(1e3 * (time.perf_counter() - tw), 2))
                        if k == pushes - 1:
                            stage_last = {kk: round(v, 3) for kk, v in hl.stage_times().items() if v}
                        n_pdu += drain()
                        push_ms.append(round(1e3 * (time.perf_counter() - t0), 2))
                    t_lib = time.perf_counter() - t_start
                    hl.close()
                    del pins
                    return {"value": s_links * chunk * pushes / t_lib / 1e6, "push_ms": push_ms, "wait_ms": wait_ms, "stage_ms_of_one_push": stage_last,
                            "unit": "Msamples/s", "links": s_links, "format": "sc16" if wire else "fc32", "h2d_bytes_per_push": int(s_links * chunk * (4 if wire else 8)),
                            "samples_per_push_per_link": chunk, "pushes": pushes, "pdus": n_pdu,
                            "realtime_factor_per_20Msps_link": chunk * pushes / t_lib / 20e6,
                            # pipeline full (the first push waits for its own copy, the last one also flushes): pushes 2 .. n-1
                            "steady_state_realtime_factor": (chunk / 20e6) / (1e-3 * float(np.mean(push_ms[1:-1]))) if len(push_ms) > 2 else None,
                            "how": "wifi_b200_rx_push_links%s_async(k+2), rx_push_wait(k), rx_pop per chunk; pre-filled pinned host buffers, one handle; wall time of the whole loop, per-rank figure" % ("_sc16" if wire else "")}

                e2e["streaming"] = live(False)
                try:
                    e2e["streaming_sc16"] = live(True)
                except Exception as ex:
                    e2e["streaming_sc16"] = {"error": repr(ex)}
        except Exception as ex:
            e2e["streaming"] = {"error": repr(ex)}
        h.host_free(hn)
        del host, hn

    tsh = None
    if not args.no_time_shard and args.workload == "c3":
        try:
            tsh = run_time_sharded(W, torch, dist, args, rank, world, local)
        except AssertionError:
            if args.strict:
                raise
            tsh = {"error": "assertion failed"}
        except Exception as ex:       # the headline must not depend on this section
            tsh = {"error": repr(ex)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    stage_ms = {k: v / args.steps for k, v in stage_acc.items()}
    n_jobs = st_ok if st_ok else n
    n_sym_w = -(-(16 + 8 * PSDU_LEN + 6) // N_DBPS)
    n_cbps = {216: 288, 96: 192}[N_DBPS]
    vit_ms = stage_ms.get("viterbi", 0.0)
    # ---- dominant kernel (k_viterbi): bound by the integer ALU pipe, not by memory (SURVEY 8d).  achieved = the
    # kernel's alu-pipe warp-instructions (ncu's dynamic count per decoded frame of this workload, committed under
    # profiles/ -- the count is a property of the code and the frame length, not of the run) x frames decoded here
    # / the kernel's CUDA-event time measured in this run; peak = the alu pipe's issue rate measured in this run by the
    # library's probe kernel (independent LOP3 chains on every SM).
    alu_peak, alu_probe_ms = h.alu_peak(8192)
    pipe = None
    try:
        pipe = json.load(open(os.path.join(ROOT, "profiles", "r02_viterbi_pipe_counts.json")))
    except Exception:
        pass
    dec_bits = n * (PSDU_LEN + 2) * 8
    vit_alg_bytes = n * (n_sym_w * n_cbps / 8 + PSDU_LEN)
    if pipe and vit_ms > 0 and pipe.get("psdu_len") == PSDU_LEN and pipe.get("n_dbps") == N_DBPS:
        alu_inst = pipe["alu_warp_inst_per_frame"] * st_frames
        achieved = alu_inst / (vit_ms * 1e-3)
        roof = {"kernel": "k_viterbi", "bound": "alu", "achieved": achieved / 1e9, "peak": alu_peak / 1e9, "unit": "Gwarp-inst/s",
                "frac": achieved / alu_peak, "traffic": pipe.get("dram_bytes_per_frame", 0) * st_frames or None,
                "peak_source": "measured in this run: wifi_b200_alu_peak (LOP3 issue probe, %.2f ms)" % alu_probe_ms,
                "instruction_count_source": "committed ncu (%s): smsp__inst_executed_pipe_alu.sum per decoded frame" % pipe.get("source", "profiles/"),
                "alu_warp_inst_per_launch": alu_inst, "ms_per_launch": vit_ms,
                "algorithmic_bytes_per_launch": vit_alg_bytes, "hbm_frac_for_reference": vit_alg_bytes / (vit_ms * 1e-3) / 1e9 / hbm_peak,
                "note": "one trellis per thread, metric and path byte of a state in one halfword, add-compare-select by VIADDMNMX.U16x2 (alu pipe 73 %%, fma pipe 32 %%, issue 72 %% in ncu); %.2f Tint-op/s algorithmic (256 int-op per decoded bit)" % (
                    dec_bits * 256 / (vit_ms * 1e-3) / 1e12)}
    else:
        roof = {"kernel": "k_viterbi", "bound": "alu", "achieved": None, "peak": alu_peak / 1e9, "unit": "Gwarp-inst/s", "frac": None, "traffic": None,
                "peak_source": "measured in this run: wifi_b200_alu_peak", "ms_per_launch": vit_ms,
                "note": "no committed instruction count for this workload shape (profiles/r02_viterbi_pipe_counts.json is for the default workload)"}
    # ---- the HBM-side stages: algorithmic bytes per launch (DESIGN.md 4) / CUDA-event time of this run, against the measured copy peak
    n_frames_w, n_rows_w = st_frames, st_frames * n_sym_w
    stage_alg = {
        "detect": ("k_detect", n_samples * (8 + 1.0 / 8 + 1.0 / 512)),
        "sync_long": ("k_sync_long", n_frames_w * ((320 + 63) * 8 + 16)),
        "demod_head": ("k_demod phase 0", n_frames_w * (3 * 64 * 8 + 624)),
        "demod_data": ("k_demod phase 1", n_rows_w * (64 * 8 + 48 + (N_DBPS // 8) * 4)),
    }
    roof_stages = {}
    for key, (kname, bytes_) in stage_alg.items():
        ms = stage_ms.get(key, 0.0)
        gbs = bytes_ / (ms * 1e-3) / 1e9 if ms else 0.0
        roof_stages[key] = {"kernel": kname, "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                            "algorithmic_bytes_per_launch": bytes_, "ms_per_launch": ms}
    roof_det = dict(roof_stages["detect"], peak_source=peak_src,
                    note="the streaming front-end reads the whole capture once (8 B per sample) and writes one flag bit per sample")
    path_alg = n_samples * 8 + n * PSDU_LEN
    step_ms = 1e3 * elapsed_max / args.steps
    line = {"metric": "rx_msamples_per_s", "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+u8", "data": "synthetic",
            "decoded_mbps": mbps, "frames_per_step": tot_frames, "crc_ok_per_step": tot_ok,
            "config": config_dict(args, n_links, fpl), "clocks": clocks, "e2e": e2e, "gpu_launches": 14 * args.steps,   # detect, select_spec, select_fix, select, reserve, frames_init, sync_long, demod x2, signal, plan_fast, plan, pack, viterbi (profiles/r02_ncu_launches.csv)
            "roofline": roof, "roofline_frontend": roof_det, "roofline_stages": roof_stages, "stage_ms": stage_ms, "tx": dict(TX_INFO), "time_sharded": tsh,
            "path_hbm": {"algorithmic_GBps": path_alg / (step_ms * 1e-3) / 1e9, "frac_of_peak": path_alg / (step_ms * 1e-3) / 1e9 / hbm_peak}}
    if not args.no_cpu and world == 1:
        from oracle import oracle as O
        nf = min(args.cpu_frames, fpl * n_links)
        nl = max(1, nf // fpl)
        sl = int(link_off[nl])
        xs = cap[:2 * sl].cpu().numpy().view(np.complex64)
        t0 = time.perf_counter()
        r = O.rx_links(xs, link_off[:nl].astype(np.int64), np.diff(link_off[:nl + 1]).astype(np.int64), n_threads=1, algo=args.algo, want_carrier=False,
                       soft=args.soft)
        dt = time.perf_counter() - t0
        # same inputs, same answers: the GPU frame table of these links equals the oracle's
        g = res.frames[np.isin(res.frames["link"], np.arange(nl))]
        g = g[np.lexsort((g["trigger"], g["link"]))]
        same = len(g) == len(r.frames) and all(np.array_equal(g[k], r.frames[k]) for k in ("trigger", "frame_start", "encoding", "length", "crc_ok"))
        line["cpu_baseline"] = {"value": sl / dt / 1e6, "unit": "Msamples/s", "cores": 1, "kind": "port",
                                "sample": "first %d links (%d frames, %d samples) of the same capture, oracle single thread, %.1f s" % (nl, nl * fpl, sl, dt),
                                "matches_gpu_frame_table": bool(same)}
    _emit(out_fd, line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the tree it runs from may be read-only: no __pycache__ beside the sources
    main()
