#!/usr/bin/env python
"""bench.py — FSK demod + center + digitize of a synthetic 1 GiSample complex64 capture per B200 (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   (CPU arm: the reference's own kernels)

One "step" (default --center detect) = ONE library call per GPU, urh_demod_center_digitize (N>1:
urh_shard_demod_center_digitize): afp_demod FSK with per-tile statistics -> capture-wide detect_center (rank window, bin
edges, histogram, peak pick: all on the device) -> grab_pulse_lens over qad -> pulse table; the host synchronises once.
--center given: the fused single-pass step for a known center (urh_demod_digitize / urh_shard_digitize), reported as
`other_variant` otherwise.
`value` = whole-job MSamples/s with the IQ already in HBM; `e2e` = the same step fed from pinned HOST memory through the
public Python API (H2D of the IQ and D2H of the pulse table inside the timed region).  The capture (8 GiB / GPU) is far
larger than the 126 MB L2, so no explicit L2 flush is needed.
After the timed loops every run checks itself against the CPU oracle (outside the timed region): `parity` in the JSON line.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SPS = 100
FS = 2e6
# +-100 kHz: detect_center's peak test needs the two levels >= 5 % of the histogram span apart, and a bursty capture's span is
# 2*pi (one random-phase sample opens every burst), so a whole-capture center needs a deviation of >= ~0.16 rad/sample
FDEV = 100e3
NOISE_MAG = 0.05
SIGMA = 0.01
TOL = 5
CENTER = 0.0
# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel: read at run time from the committed summary of this
# round's `ncu --set full` capture (tools/ncu_summary.py writes profiles/traffic.json: bytes per sample per kernel, captured at
# 2^28 samples; the kernels stream, so DRAM bytes scale with n).  null when the file is missing.
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "traffic.json")
ALG_BYTES_PER_SAMPLE = 12  # dominant kernel, SURVEY §8d: read IQ 8 B + write qad 4 B (pulse table ~0.1 B/sample ignored)
STEP_BYTES_PER_SAMPLE = {"detect": 16, "given": 12}  # SURVEY §8d per-path budgets (detect: qad re-read once)
PARITY_LOG2 = 24  # parity windows of 2^24 samples (first / middle / last of every shard)
# --dump-outputs: at most this many demodulated samples and pulse-table rows over all ranks, at fixed seeded positions when the
# output is larger (qad 12 B per sample with its index, rows 24 B: 48 MB in all)
DUMP_QAD_SAMPLES = 1 << 21
DUMP_PULSE_ROWS = 1 << 20


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def capture_gaps(n, rank):
    """Every 2^log2n-sample block of the capture has the same structure: bursts of 5 M samples every 6 M, one long gap at 40-43 % of
    the block and silence from 97 % on.  One block per GPU: the per-GPU work is the same at every N (weak scaling).  With the long
    gap and the tail defined on the WHOLE capture instead, two of eight shards hold them all and the other six do 8 % more work in
    the histogram and digitizer passes than the single-GPU run (silent tiles are skipped): measured with tools/timeline_dist.py,
    profiles/r02_timeline_n4_globalgaps_*.json - 318 of the 390 us a step lost from 1 to 8 GPUs were that imbalance, 87 us the exchanges."""
    off = n * rank
    return off + int(0.40 * n), off + int(0.43 * n), off + int(0.97 * n)


def make_symbols(nsym, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    b = (rng.integers(0, 2, nsym, dtype=np.int8) * 2 - 1).astype(np.int8)
    s = np.zeros(nsym, dtype=np.int32)
    np.cumsum(b[:-1], out=s[1:], dtype=np.int32)
    return b, s


class ClockSampler:
    """Sample nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def _reference_detect_center():
    """the reference's own detect_center (numpy code, AutoInterpretation.py:226-277) when its Python layer travelled
    with oracle/_ref (oracle/build_ref.py stages it), else the oracle's restatement of it"""
    from oracle import oracle, ref_loader
    try:
        ns = ref_loader.load_python_layer()
        return ns.AutoInterpretation.detect_center, "reference"
    except Exception:
        return oracle.detect_center, "port"


def cpu_reference_arm(n_cpu, steps, warmup, iq_slice=None, detect=True, outputs=None):
    """Time the reference's own CPU implementation (its compiled kernels under oracle/_ref when present, else the C oracle
    port) of afp_demod(FSK) [+ detect_center] + grab_pulse_lens on a bounded slice, all host threads.  `outputs` (a dict)
    receives the last step's qad, center and pulse table."""
    from oracle import oracle, ref_loader

    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)  # torchrun presets 1; the reference's prange should use every core
    try:
        C.CDLL("libgomp.so.1").omp_set_num_threads(cores)  # in case libgomp is already loaded (torch)
    except OSError:
        pass
    kind = "port"
    demod, grab = oracle.afp_demod, oracle.grab_pulse_lens
    try:
        sf, _, _ = ref_loader.load_kernels()
        demod = lambda iq, nm, mt, mo: np.asarray(sf.afp_demod(iq, nm, mt, mo))  # noqa: E731
        grab = lambda q, c, t, mt, sps: np.asarray(sf.grab_pulse_lens(q, c, t, mt, sps))  # noqa: E731
        kind = "reference"
    except Exception:
        oracle.build()
    detect_center, center_kind = _reference_detect_center()
    if iq_slice is None:
        iq_slice = host_synth(n_cpu)
    n_cpu = len(iq_slice)
    times = []
    rows = None
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        q = demod(iq_slice, NOISE_MAG, "FSK", 2)
        center = detect_center(q) if detect else CENTER
        rows = grab(q, center, TOL, "FSK", SPS)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    sec = float(np.median(times))
    if outputs is not None:
        outputs.update(qad=q, center=center, rows=rows)
    return {"value": n_cpu / sec / 1e6, "unit": "MSamples/s", "cores": cores, "kind": kind,
            "sample": "%d-sample slice of the same synthetic 2-FSK recipe (afp_demod FSK [%s]%s + grab_pulse_lens [%s]), median of %d"
                      % (n_cpu, kind, (" + detect_center [%s, numpy as in the reference]" % center_kind) if detect else "", kind, len(times)),
            "ms_per_step": sec * 1e3, "rows": int(len(rows))}


def host_synth(n, seed=0):
    """numpy version of the synthetic recipe for the CPU-only arm (no GPU needed)."""
    rng = np.random.default_rng(seed)
    nsym = n // SPS + 2
    b = rng.integers(0, 2, nsym) * 2 - 1
    m = np.repeat(b, SPS)[:n]
    phase = 2 * np.pi * (FDEV / FS) * np.cumsum(m)
    g = np.arange(n)
    on = ((g % 6_000_000) < 5_000_000) & (g < int(0.97 * n))
    x = on * np.exp(1j * phase) + SIGMA * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    iq = np.empty((n, 2), np.float32)
    iq[:, 0] = x.real
    iq[:, 1] = x.imag
    return iq


def dump_outputs(dirname, rank, world, n, get_qad, rows, center):
    """Write what the step hands its caller - the detected (or given) center, the pulse table and the demodulated signal (qad) -
    as float64 / float32 .npy files under `dirname` (suffix _rank<r> when world > 1).  Tables larger than the dump budget are
    sampled at positions drawn with a fixed seed, so two builds run with the same arguments write comparable files; the *_index
    files hold the positions.  get_qad(a, b) returns qad[a:b] on the host."""
    os.makedirs(dirname, exist_ok=True)
    sfx = "" if world == 1 else "_rank%d" % rank
    rng = np.random.default_rng(20240 + rank)

    def positions(total, cap):
        return np.arange(total) if total <= cap else np.unique(rng.integers(0, total, cap))

    qi = positions(n, DUMP_QAD_SAMPLES // world)
    qad = np.empty(len(qi), np.float32)
    chunk = 1 << 26
    for a in range(0, n, chunk):
        lo, hi = np.searchsorted(qi, [a, min(a + chunk, n)])
        if hi > lo:
            qad[lo:hi] = get_qad(a, min(a + chunk, n))[qi[lo:hi] - a]
    ri = positions(len(rows), DUMP_PULSE_ROWS // world)
    out = {"center": np.array([np.nan if center is None else center], np.float64),
           "qad": qad, "qad_index": qi.astype(np.float64),
           "pulses": rows[ri].astype(np.float64), "pulses_index": ri.astype(np.float64)}
    for name, arr in out.items():
        np.save(os.path.join(dirname, name + sfx + ".npy"), arr)


def parity_windows(n_local):
    w = min(n_local, 1 << PARITY_LOG2)
    starts = sorted({0, ((n_local // 2) // 2048) * 2048 if n_local // 2 + w <= n_local else 0, n_local - w})
    return w, starts


def parity_block(ctx, rank, world, dist, d_iq, halo_host, d_qad, rows, center, n, n_total, offset):
    """GPU result of the last timed step vs the CPU oracle (oracle/_ref = the reference's compiled kernels when they
    travelled, else the C restatement), outside the timed region, on the first / middle / last 2^24 samples of this rank's
    shard: every qad word, and every pulse boundary (position, state) of the WHOLE-capture pulse table that falls inside the
    window (minus a margin in which a digitizer started at the window edge has not yet seen two runs)."""
    from oracle import oracle, ref_loader

    kind = "port"
    demod, grab = oracle.afp_demod, oracle.grab_pulse_lens
    try:
        sfr, _, _ = ref_loader.load_kernels()
        demod = lambda iq, nm, mt, mo: np.asarray(sfr.afp_demod(iq, nm, mt, mo))  # noqa: E731
        grab = lambda q, c, t, mt, sps: np.asarray(sfr.grab_pulse_lens(q, c, t, mt, sps))  # noqa: E731
        kind = "reference"
    except Exception:
        oracle.build()
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    # absolute position of the firing that ends row j: tol - 1 + (sum of all lengths up to and including row j)
    s_local = int(rows[:, 1].sum())
    before = 0
    if dist is not None:
        import torch

        allv = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(allv, torch.tensor([s_local], dtype=torch.int64))
        before = int(sum(int(v.item()) for v in allv[:rank]))
    fire_rows = rows[:-1] if rank == world - 1 else rows   # the capture's last row is the tail row, not a firing
    pos_gpu = TOL - 1 + before + np.cumsum(fire_rows[:, 1])
    st_gpu = fire_rows[:, 0]
    w, starts = parity_windows(n)
    margin = min(w // 4, 1 << 21)
    out = {"oracle": kind, "window_samples": w, "windows": len(starts), "qad_words_compared": 0, "qad_words_differing": 0,
           "boundaries_compared": 0, "boundaries_differing": 0}
    for a in starts:
        # one predecessor sample for the FSK conjugate product (the halo for the shard's first sample)
        if a > 0:
            iq = d_iq[a - 1: a + w].get()
        elif rank > 0:
            iq = np.concatenate([halo_host, d_iq[0: w].get()])
        else:
            iq = d_iq[0: w].get()
        q_ref = demod(np.ascontiguousarray(iq), NOISE_MAG, "FSK", 2)
        if a > 0 or rank > 0:
            q_ref = q_ref[1:]
        q_gpu = d_qad[a: a + w].get()
        out["qad_words_compared"] += int(w)
        out["qad_words_differing"] += int(np.count_nonzero(q_gpu.view(np.uint32) != q_ref.view(np.uint32)))
        r_ref = grab(np.ascontiguousarray(q_ref), float(center), TOL, "FSK", SPS)
        g0 = offset + a
        pos_ref = g0 + TOL - 1 + np.cumsum(r_ref[:-1, 1])
        st_ref = r_ref[:-1, 0]
        lo, hi = g0 + margin, g0 + w
        mg = (pos_gpu > lo) & (pos_gpu < hi)
        mr = (pos_ref > lo) & (pos_ref < hi)
        pg, sg, pr, sr = pos_gpu[mg], st_gpu[mg], pos_ref[mr], st_ref[mr]
        out["boundaries_compared"] += int(len(pr))
        if len(pg) != len(pr):
            out["boundaries_differing"] += abs(len(pg) - len(pr)) + 1
        else:
            out["boundaries_differing"] += int(np.count_nonzero((pg != pr) | (sg != sr)))
    if dist is not None:
        import torch

        keys = ("qad_words_compared", "qad_words_differing", "boundaries_compared", "boundaries_differing")
        t = torch.tensor([out[k_] for k_ in keys], dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        for k_, v in zip(keys, t.tolist()):
            out[k_] = int(v)
        out["windows"] = len(starts) * world
    out["ok"] = out["qad_words_differing"] == 0 and out["boundaries_differing"] == 0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2n", type=int, default=30, help="samples per GPU = 2**log2n (default 1 GiSample)")
    ap.add_argument("--cpu-log2n", type=int, default=26)
    ap.add_argument("--center", default="detect", choices=["detect", "given"],
                    help="detect: demod + detect_center + digitize (BASELINE configs[1]); given: fused demod+digitize, center known")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the last step's center, pulse table and qad (sampled) to DIR/<name>.npy")
    ap.add_argument("--worst", action="store_true",
                    help="also time the unfavourable inputs (noise gate off / white-noise IQ / +-300 kHz deviation: every sample pair "
                         "leaves the packed-f32x2 fast path) and report them under `worst_case`")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    world = env_int("WORLD_SIZE", 1)
    n = 1 << args.log2n
    layout = ("2^%d samples on one GPU" % args.log2n if world == 1 else
              "ONE capture of %d x 2^%d samples (every 2^%d-sample block built like the single-GPU capture) sharded by contiguous range "
              "(1-sample halo, run stitching across shards)" % (world, args.log2n, args.log2n))
    workload = ("2-FSK complex64, %s @2MS/s sps=100 +-100kHz AWGN sigma=0.01 bursts+gaps; %s (tol=5, noise=0.05)"
                % (layout, "demod + detect_center (capture-wide) + digitize" if args.center == "detect"
                   else "fused demod+digitize, center=0 given"))
    base = {"metric": "MSamples/s IQ demod+digitize (complex64)", "unit": "MSamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "samples_per_gpu": n, "l2": "inputs (8 B/sample) larger than L2; no flush"}}

    if args.impl == "reference":
        if rank != 0:
            return 0
        last = {}
        r = cpu_reference_arm(1 << args.cpu_log2n, args.steps, max(1, min(args.warmup, 2)), detect=args.center == "detect", outputs=last)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, 0, 1, len(last["qad"]), lambda a, b: last["qad"][a:b], last["rows"], last["center"])
        line = dict(base)
        line.update({"impl": "reference", "value": r["value"], "ms_per_step": r["ms_per_step"],
                     "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                     "e2e": {"value": r["value"], "unit": "MSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "gpu_launches": 0})
        line["config"] = dict(base["config"], reference_sample=r["sample"])
        print(json.dumps(line))
        return 0

    dist = None
    if world > 1:
        import torch.distributed as dist  # gloo: only barrier + max-reduce of timings (no data-path collective)

        dist.init_process_group("gloo", rank=rank, world_size=world)

    from urh_b200 import _lib
    from urh_b200.device import DeviceArray, PinnedArray
    from urh_b200.cythonext import signal_functions as sf

    ctx = _lib.default_context(local_rank)
    lib = ctx.lib
    info = ctx.device_info()
    n_total = n * world
    offset = n * rank

    # ---- synthesise this rank's shard of ONE capture of world*2^log2n samples directly in HBM -------------------
    # (N > 1: contiguous shards, 1-sample halo from the left neighbour over NCCL, run stitching as in urh_b200/dist.py)
    from urh_b200 import dist as udist

    nsym = n // SPS + 2
    b, s = make_symbols(nsym, seed=1000 + rank)
    d_b = DeviceArray(ctx, (nsym,), np.int8).set(b)
    d_s = DeviceArray(ctx, (nsym,), np.int32).set(s)
    sb = udist.ShardBuffer(ctx, n, np.float32)
    d_iq = sb.shard
    d_qad = DeviceArray(ctx, (n,), np.float32)
    period, burst = 6_000_000, 5_000_000
    ctx.check(lib.urh_synth_fsk(ctx.handle, C.c_void_p(d_iq.ptr), n, offset, SPS, C.c_void_p(d_b.ptr), C.c_void_p(d_s.ptr),
                                C.c_double(FDEV / FS), 1.0, SIGMA, 12345, period, burst, *capture_gaps(n, rank)))
    ctx.sync()
    if world > 1:
        hx = udist.HostExchange()
        udist.init_nccl(ctx, hx)
        base["config"]["exchange"] = ("NVLink peer mailboxes (device-resident, stream-ordered)" if getattr(ctx, "p2p", False)
                                      else "NCCL (stream-ordered)")
        udist.exchange_halo(ctx, hx, sb)

    from urh_b200.ainterpretation import AutoInterpretation as AI

    dense_of_step = [0.0]

    def read_dense_ms():
        ms = C.c_float()
        lib.urh_last_dense_ms(ctx.handle, C.byref(ms))
        return ms.value

    def step_given():
        if world > 1:
            k = udist.demod_digitize_distributed(ctx, rank, world, sb, offset, n_total, NOISE_MAG, "FSK", CENTER, TOL, SPS,
                                                 d_qad=d_qad, fetch=False)
            dense_of_step[0] = read_dense_ms()
            return k
        k = C.c_int64(0)
        ctx.check(lib.urh_demod_digitize(ctx.handle, C.c_void_p(d_iq.ptr), _lib.DT_F32, n, NOISE_MAG, _lib.MOD_FSK,
                                         CENTER, TOL, SPS, 1, 0.1, C.c_void_p(d_qad.ptr), C.byref(k)))
        dense_of_step[0] = read_dense_ms()
        return k.value

    center_seen = [None]

    def step_detect():
        if world > 1:
            center, k = udist.demod_center_digitize_distributed(ctx, rank, world, sb, offset, n_total, NOISE_MAG, "FSK", TOL, SPS, d_qad,
                                                                fetch=False)
            dense_of_step[0] = read_dense_ms()
            center_seen[0] = center
            return k
        center, state, k = C.c_double(0.0), C.c_int(0), C.c_int64(0)
        ctx.check(lib.urh_demod_center_digitize(ctx.handle, C.c_void_p(d_iq.ptr), _lib.DT_F32, n, NOISE_MAG, _lib.MOD_FSK, TOL, SPS, -1,
                                                C.c_void_p(d_qad.ptr), C.byref(center), C.byref(state), C.byref(k)))
        assert state.value == 1, "detect_center: state %d" % state.value
        dense_of_step[0] = read_dense_ms()
        center_seen[0] = center.value
        return k.value

    step_resident = step_detect if args.center == "detect" else step_given

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()

    # ---- resident (HBM) timing -----------------------------------------------------------------------------
    lib.urh_set_profiling(ctx.handle, 1)
    for _ in range(args.warmup):
        k_rows = step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    dense_ms = []
    ctx.timer_start()
    for _ in range(args.steps):
        k_rows = step_resident()
        dense_ms.append(dense_of_step[0])
    total_ms = ctx.timer_stop()
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    barrier()
    if dist is not None:
        import torch

        t = torch.tensor([total_ms], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * n / (ms_per_step * 1e-3) / 1e6

    # ---- the last timed step's outputs, and their parity against the CPU oracle (outside the timed region) -----------
    rows_last = None
    if args.dump_outputs or not args.no_parity:
        rows_last = np.empty((k_rows, 2), dtype=np.int64)
        if k_rows:
            ctx.check(lib.urh_fetch_pulses(ctx.handle, rows_last.ctypes.data_as(C.c_void_p), k_rows))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, world, n, lambda a, b: d_qad[a:b].get(), rows_last,
                     center_seen[0] if args.center == "detect" else CENTER)
    parity = None
    if not args.no_parity:
        lens = int(rows_last[:, 1].sum())
        if dist is not None:
            import torch

            t = torch.tensor([lens], dtype=torch.int64)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            lens = int(t.item())
        c_used = center_seen[0] if args.center == "detect" else CENTER
        parity = parity_block(ctx, rank, world, dist, d_iq, sb.halo.get() if world > 1 else None, d_qad, rows_last, c_used, n, n_total,
                              offset)
        parity["sum_of_pulse_lengths_is_n_minus_tol"] = lens == n_total - TOL
        parity["ok"] = bool(parity["ok"] and parity["sum_of_pulse_lengths_is_n_minus_tol"])
        del rows_last
        barrier()

    # ---- the other variant, for the record (not the headline): same capture, same timing rules, fewer steps ------
    other = step_given if args.center == "detect" else step_detect
    other_steps = max(3, min(args.steps, 20))
    for _ in range(3):
        other()
    barrier()
    other_dense = []
    ctx.timer_start()
    for _ in range(other_steps):
        other()
        other_dense.append(dense_of_step[0])
    other_ms = ctx.timer_stop()
    barrier()
    if dist is not None:
        import torch

        t = torch.tensor([other_ms], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        other_ms = float(t.item())
    other_ms /= other_steps
    other_line = {"variant": "fused demod+digitize, center=0 given" if args.center == "detect" else "demod + detect_center + digitize",
                  "value": world * n / (other_ms * 1e-3) / 1e6, "unit": "MSamples/s", "ms_per_step": other_ms, "steps": other_steps,
                  "dense_kernel_ms": float(np.mean(other_dense))}

    # stage breakdown of the detect variant at N=1 (device timers around each public call; diagnostic)
    stages = None
    if world == 1:
        stages = {}
        kept = C.c_int64(0)
        w5 = np.zeros(5)
        reps = 3
        acc = {"demod+tile_stats": 0.0, "window_stats": 0.0, "histogram+peaks": 0.0, "digitize(qad)": 0.0}
        for _ in range(reps):
            ctx.timer_start()
            ctx.check(lib.urh_afp_demod_tiles(ctx.handle, C.c_void_p(d_iq.ptr), _lib.DT_F32, n, NOISE_MAG, _lib.MOD_FSK,
                                              C.c_void_p(d_qad.ptr), 0, C.byref(kept)))
            acc["demod+tile_stats"] += ctx.timer_stop()
            r0, r1 = AI.center_rank_window(kept.value)
            ctx.timer_start()
            ctx.check(lib.urh_center_window_stats(ctx.handle, C.c_void_p(d_qad.ptr), n, r0, r1, w5.ctypes.data_as(C.c_void_p)))
            acc["window_stats"] += ctx.timer_stop()
            st = AI.center_stats_from_window(kept.value, r0, r1, w5)
            t0 = time.perf_counter()
            c = AI._center_from_stats(ctx, d_qad, n, st, lib.urh_center_histogram_tiles)
            ctx.sync()
            acc["histogram+peaks"] += (time.perf_counter() - t0) * 1e3
            k = C.c_int64(0)
            ctx.timer_start()
            ctx.check(lib.urh_grab_pulse_lens(ctx.handle, C.c_void_p(d_qad.ptr), n, float(c), TOL, _lib.MOD_FSK, SPS, 1, 0.1, C.byref(k)))
            acc["digitize(qad)"] += ctx.timer_stop()
        stages = {k_: v / reps for k_, v in acc.items()}

    # ---- end-to-end through the public API with HOST buffers ----------------------------------------------
    e2e = None
    if not args.no_e2e:
        host = PinnedArray((n, 2), np.float32, ctx)
        d_iq.get(out=host.array)  # this rank's shard now lives in pinned host memory
        e2e_steps = max(1, min(args.steps, 3))
        if world > 1:
            sb2 = udist.ShardBuffer(ctx, n, np.float32)
            halo = sb.halo.get()
            rows_pinned = PinnedArray((n // 64 + 1024, 2), np.int64, ctx)

            def step_e2e():
                sb2.halo.set(halo)
                if args.center == "detect":
                    # this rank's shard streamed from pinned host memory (chunked upload overlapped with the demodulation)
                    return udist.demod_center_digitize_distributed(ctx, rank, world, sb2, offset, n_total, NOISE_MAG, "FSK", TOL, SPS, d_qad,
                                                                   host_iq=host.array, rows_out=rows_pinned.array)[1]
                sb2.shard.set_async(host.array)
                return udist.demod_digitize_distributed(ctx, rank, world, sb2, offset, n_total, NOISE_MAG, "FSK", CENTER, TOL, SPS)
        else:
            d_e2e = DeviceArray(ctx, (n, 2), np.float32)
            rows_pinned = PinnedArray((n // 64 + 1024, 2), np.int64, ctx)   # pinned: the pulse table comes back as one DMA

            def step_e2e():
                if args.center == "detect":
                    # host IQ in, host pulse table out: the upload is chunked on the copy stream and every chunk is demodulated as
                    # soon as it has landed (urh_demod_center_digitize_host)
                    return sf.demod_center_digitize(host.array, NOISE_MAG, "FSK", TOL, SPS, scratch=d_e2e, out=d_qad, rows_out=rows_pinned.array)[1]
                d_e2e.set_async(host.array)
                qad, rows = sf.demod_digitize(d_e2e, NOISE_MAG, "FSK", CENTER, TOL, SPS, return_qad=False)
                return rows

        rows = step_e2e()
        barrier()
        t0 = time.perf_counter()
        ctx.timer_start()
        for _ in range(e2e_steps):
            rows = step_e2e()
        e2e_ms = ctx.timer_stop()
        wall_ms = (time.perf_counter() - t0) * 1e3
        e2e_ms = max(e2e_ms, wall_ms)  # host-side work (D2H of the rows) is part of the step
        if dist is not None:
            import torch

            t = torch.tensor([e2e_ms], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
        e2e = {"value": world * n / (e2e_ms / e2e_steps * 1e-3) / 1e6, "unit": "MSamples/s",
               "h2d_bytes_per_step": int(n * 8), "d2h_bytes_per_step": int(rows.nbytes), "steps": e2e_steps,
               "api": "urh_b200.cythonext.signal_functions.%s(pinned host IQ) -> pulse table on host"
                      % ("demod_center_digitize" if args.center == "detect" else "demod_digitize")}
        assert len(rows) == k_rows
        # size-independent property of the digitizer: the pulse lengths of the whole capture sum to n_total - tolerance
        lens = int(rows[:, 1].sum())
        if dist is not None:
            import torch

            t = torch.tensor([lens], dtype=torch.int64)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            lens = int(t.item())
        assert lens == n_total - TOL, (lens, n_total - TOL)
        host.free()

    # ---- the unfavourable inputs (same kernel entry points, same timing rules, fewer steps) -----------------------------------
    worst = None
    if args.worst and world == 1:
        worst = []
        cases = [("noise gate off (noise_mag = 0): no sample is skipped", FDEV / FS, 1.0, SIGMA, 0.0),
                 ("+-300 kHz deviation (0.94 rad/sample): |im/re| >= 0.4375 for every pair -> scalar bit-exact atan2f path", 0.15, 1.0, SIGMA, NOISE_MAG),
                 ("white-noise IQ (sigma = 1, no carrier), noise gate off: random angles, ~70 % of the pairs on the scalar path", 0.0, 0.0, 1.0, 0.0)]
        for name, dev, amp, sigma, noise in cases:
            ctx.check(lib.urh_synth_fsk(ctx.handle, C.c_void_p(d_iq.ptr), n, offset, SPS, C.c_void_p(d_b.ptr), C.c_void_p(d_s.ptr),
                                        C.c_double(dev), amp, sigma, 777, period, burst, *capture_gaps(n, rank)))
            ctx.sync()
            k = C.c_int64(0)

            def run():
                ctx.check(lib.urh_demod_digitize(ctx.handle, C.c_void_p(d_iq.ptr), _lib.DT_F32, n, noise, _lib.MOD_FSK, CENTER, TOL, SPS, 1, 0.1,
                                                 C.c_void_p(d_qad.ptr), C.byref(k)))
                return read_dense_ms()
            for _ in range(3):
                run()
            ctx.sync()
            dms = []
            ctx.timer_start()
            for _ in range(10):
                dms.append(run())
            ms = ctx.timer_stop() / 10
            worst.append({"input": name, "step": "fused demod+digitize, center=0 given", "ms_per_step": ms, "value": n / (ms * 1e-3) / 1e6,
                          "unit": "MSamples/s", "dense_kernel_ms": float(np.mean(dms)), "pulse_rows": int(k.value),
                          "dense_kernel_GBps": ALG_BYTES_PER_SAMPLE * n / (float(np.mean(dms)) * 1e-3) / 1e9})

    if rank != 0:
        return 0

    # ---- roofline of the dominant kernel (fused dense demod+classify+run kernel) ---------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    dense = float(np.mean(dense_ms))
    achieved = ALG_BYTES_PER_SAMPLE * n / (dense * 1e-3) / 1e9
    kernel_key = "k_fsk_fifo<WRITE,STATS>" if args.center == "detect" else "k_fsk_fifo<DIGITIZE,WRITE>"
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(TRAFFIC_FILE))
        ent = tj.get(args.center)
        if ent:
            traffic = float(ent["dram_bytes_per_sample"]) * n
            traffic_src = "%s (%s, ncu --set full, scaled by n)" % (os.path.relpath(TRAFFIC_FILE, ROOT), ent.get("capture", ""))
    except Exception:
        pass
    step_bytes = STEP_BYTES_PER_SAMPLE[args.center]
    step_gbs = step_bytes * n * world / (ms_per_step * 1e-3) / 1e9 / world   # per GPU
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "kernel": kernel_key + (" (demod + tile statistics)" if args.center == "detect" else " (fused demod + classify + runs)"),
                "kernel_ms": dense, "algorithmic_bytes_per_launch": ALG_BYTES_PER_SAMPLE * n, "peak_source": peak_src,
                "kernel_share_of_step": dense / ms_per_step,
                # the whole step against the same peak: SURVEY 8d's per-path byte budget / ms_per_step (per GPU)
                "step_bytes_per_sample": step_bytes, "step_achieved": step_gbs, "step_frac": step_gbs / peak}

    cpu = None
    if not args.no_cpu and world == 1:
        # bounded CPU sample of the same capture (first 2^cpu_log2n samples)
        ncpu = min(n, 1 << args.cpu_log2n)
        sl = d_iq[:ncpu].get()
        r = cpu_reference_arm(ncpu, 3, 1, iq_slice=sl, detect=args.center == "detect")
        cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}

    line = dict(base)
    line.update({"value": value, "ms_per_step": ms_per_step, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "parity": parity,
                 "gpu_launches": int(launches), "clocks": clocks, "pulse_rows_per_step": int(k_rows),
                 "detected_center": center_seen[0], "other_variant": other_line, "worst_case": worst, "stage_ms": stages,
                 "device": info["name"], "sm_count": info["sm_count"]})
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
