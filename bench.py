#!/usr/bin/env python
"""bench.py -- the measurement contract.

Metric (BASELINE.json): POA consensus windows/sec on synthetic 10 kb x 32-read windows (config C3: adaptive band 256, int32
scores; adaptive_storage_factor 3.0 -- the reference's default 2.0 yields exceeded_adaptive_banded_matrix_size for every window
of this workload on both this engine and the reference (SURVEY.md fact 3 / DESIGN.md), 3.0 is the smallest integer factor at
which all windows succeed; the factor only sizes the per-window score slab, results are identical). One "step" = one pass of the
hot path over one batch of 1600 windows: close to the 1623 that the free HBM of an otherwise idle B200 holds at this size, with
room left for memory that other processes or NCCL hold (1619 per GPU in a 2-GPU run). The count is fixed so that the inputs of
a run do not depend on free memory, and it is not rounded to a wave (the kernel runs a persistent grid). Windows shard
embarrassingly: every rank owns a Batch and its own windows (weak scaling), NCCL is used only for the barrier and the
max-over-ranks timing. (A fixed window list scattered from rank 0 and gathered back in input order over NCCL is
genomeworks_b200/sharding.py: sharded_consensus, proven against the single-GPU output by tests/test_gpu_sharded.py; it is not
a bench mode.)

  value : windows/s, inputs packed and resident in HBM before the timed region (K x launch, CUDA events on the batch stream,
          max over ranks)
  e2e   : windows/s through the drop-in API with HOST buffers every step: one add_poa_group call per window (packing), H2D,
          kernel, D2H of consensus + coverage (wall clock around barrier + synchronize, max over ranks)
  roofline: algorithmic bytes = executed DP cells x sizeof(ScoreT) (SURVEY.md 8d) / kernel time, vs MEASURED_PEAKS hbm_gbs;
          traffic = dram bytes per window of the shipped kernel from the committed ncu capture (profiles/r02_traffic.json)
  extra : the other driver-visible workloads on the same line: C3 with MSA output, C2 (1 kb x 16, static band, int16), C4
          (cudaaligner 10k x 10k, band 1024), each with value / e2e / roofline fraction
  cpu_baseline / --impl reference: 3rdparty/spoa (oracle/_ref/libspoa_ref.so, unmodified) on the host cores. The reference arm
          runs FULL 32-read windows: every host thread keeps one window in progress and fuses 2 reads per step, so that after 16
          steps every read position of a window has been timed against the true graph (oracle/spoa_capi.cpp, streaming interface).

Other workloads as the main line for development: --workload c2 | c4.

--dump-outputs DIR writes what the timed path returned in its last timed step (rank 0) as DIR/<name>.npy in float64, so that two
builds can be compared output for output on identical inputs (every input is generated from fixed seeds).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload):
    """dram bytes (read + write) per unit of the dominant kernel from the committed ncu --set full capture of the shipped build
    (profiles/r02_traffic.json, written from gpurun_out/ncu by tools/ncu_traffic.py). None when no capture is committed."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        return json.load(open(p)).get(workload)
    except Exception:
        return None


class ClockSampler:
    """Samples nvidia-smi SM clocks + throttle reasons during the timed region."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split("\n")[0]
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


DUMP_BYTES = 60_000_000  # all dumped arrays together, under 64 MB with the .npy headers


def sample_rows(n, row_bytes, budget):
    """A fixed, seeded sample (sorted indices) of as many of n rows as fit `budget` bytes at `row_bytes` each, all rows when they fit."""
    k = min(n, max(1, budget // max(row_bytes, 1)))
    return np.sort(np.random.RandomState(0).permutation(n)[:k])


def padded(flat, offsets, idx, width):
    """Rows idx of a ragged array (row i = flat[offsets[i]:offsets[i + 1]]) as an (len(idx), width) array, zero past each row."""
    out = np.zeros((len(idx), width), dtype=np.float64)
    for j, i in enumerate(idx):
        row = flat[offsets[i]:offsets[i + 1]]
        out[j, :len(row)] = row
    return out


def poa_outputs(r):
    """get_consensus() after the last timed launch: status and consensus length of every window; consensus (ASCII codes) and
    per-base coverage of a seeded sample of windows, zero past each window's length."""
    lens = r["lens"].astype(np.int64)
    width = int(lens.max(initial=0))
    idx = sample_rows(len(lens), 2 * 8 * width, DUMP_BYTES - 24 * len(lens))
    mask = np.arange(width)[None, :] < lens[idx, None]
    return {"status": r["status"], "consensus_length": lens, "sample_window": idx,
            "consensus": np.where(mask, r["consensus"][idx, :width], 0), "coverage": np.where(mask, r["coverage"][idx, :width], 0)}


def aligner_outputs(r):
    """sync_alignments_flat() of the last timed step: status, is_optimal and run count of every pair; the run-length encoded
    alignment (action codes, run lengths) of a seeded sample of pairs, zero past each pair's run count."""
    st, opt, offs, act, runs = r["last"]
    counts = np.diff(offs)
    width = int(counts.max(initial=0))
    idx = sample_rows(len(counts), 2 * 8 * width, DUMP_BYTES - 32 * len(counts))
    return {"status": st, "is_optimal": opt, "run_count": counts, "sample_pair": idx, "actions": padded(act, offs, idx, width),
            "runs": padded(runs, offs, idx, width)}


def dump_outputs(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def workload_params(name, windows=0):
    if name == "c3":
        return dict(kind="poa", key="c3", name="C3: cudapoa long-read consensus, 10 kb x 32 reads/window, adaptive band 256, int32 scores, "
                    "adaptive_storage_factor 3.0", backbone=10000, reads=32, mut=200, ins=100, dele=100, max_seq=10240, band=256,
                    band_mode="adaptive_band", factor=3.0, windows=windows or 1600)
    if name == "c2":
        return dict(kind="poa", key="c2", name="C2: cudapoa short-read consensus, 1 kb x 16 reads/window, static band 256, int16 scores",
                    backbone=1000, reads=16, mut=20, ins=10, dele=10, max_seq=1024, band=256, band_mode="static_band", factor=2.0,
                    windows=windows or 1024)
    if name == "c4":
        return dict(kind="aligner", key="c4", name="C4: cudaaligner global, 10000 x 10000 bp, Myers banded (max_bandwidth 1024)", genome=10000,
                    max_bw=1024, windows=windows or 512)
    raise SystemExit("unknown workload " + name)


# ------------------------------------------------------------------------------------------------------------------------------
# CPU legs (the only places bench.py executes anything under oracle/)
# ------------------------------------------------------------------------------------------------------------------------------
def spoa_sample(wp, n_windows, seed0, threads=0, reads=None):
    """Times unmodified spoa on n_windows windows of the workload (bounded sample for `cpu_baseline`). For long-read workloads a
    full window costs spoa minutes per core, so the sample uses the first `reads` reads of each window and the windows/s figure
    is extrapolated with spoa's own DP-cell count (graph nodes grow linearly with the number of reads fused). The reference arm
    (--impl reference) measures full windows instead."""
    import ref_lib
    from genomeworks_b200 import synth
    full_reads = wp["reads"]
    reads = full_reads if reads is None else min(reads, full_reads)
    win_nseq, seq_len, data = synth.poa_windows(n_windows, wp["backbone"], full_reads, wp["mut"], wp["ins"], wp["dele"], seed0=seed0,
                                                max_read_len=wp["max_seq"])
    if reads < full_reads:
        sl = seq_len.reshape(n_windows, full_reads)
        offs = np.concatenate([[0], np.cumsum(seq_len)]).astype(np.int64)
        keep = []
        for w in range(n_windows):
            keep.append(data[int(offs[w * full_reads]):int(offs[w * full_reads + reads])])
        data = np.concatenate(keep + [np.zeros(1, np.uint8)])
        seq_len = np.ascontiguousarray(sl[:, :reads]).reshape(-1)
        win_nseq = np.full(n_windows, reads, dtype=np.int32)
    r = ref_lib.spoa_consensus(win_nseq, seq_len, data, n_threads=threads, want_strings=False)
    r["windows"] = n_windows
    r["reads_used"] = reads
    L = float(wp["backbone"])
    if reads < full_reads:
        a = reads - 1
        cells_pw = r["cells"] / n_windows
        g = max(0.0, (cells_pw / (L * L) - a) / max(a * (a - 1) / 2.0, 1e-9))
        A = full_reads - 1
        full_cells = L * L * (A + g * A * (A - 1) / 2.0)
        r["scale"] = cells_pw / full_cells
    else:
        r["scale"] = 1.0
    r["windows_per_s"] = (n_windows / r["seconds"]) * r["scale"]
    return r


def spoa_full_window_stream(wp, steps, warmup, reads_per_step=2):
    """Reference arm for long-read workloads: full windows through the streaming interface. Returns (value windows/s, info dict)."""
    import ref_lib
    from genomeworks_b200 import synth
    cores = os.cpu_count() or 1
    lib = ref_lib.spoa()
    lib.spoa_stream_create.restype = C.c_void_p
    lib.spoa_stream_step.restype = C.c_double
    n_threads = max(1, min(cores, 256))
    n_windows = 3 * n_threads
    win_nseq, seq_len, data = synth.poa_windows(n_windows, wp["backbone"], wp["reads"], wp["mut"], wp["ins"], wp["dele"], seed0=1000,
                                                max_read_len=wp["max_seq"])
    h = C.c_void_p(lib.spoa_stream_create(C.c_int32(n_windows), win_nseq.ctypes.data_as(C.c_void_p), seq_len.ctypes.data_as(C.c_void_p),
                                          data.ctypes.data_as(C.c_void_p), C.c_int32(8), C.c_int32(-6), C.c_int32(-8), C.c_int32(n_threads)))
    P = wp["reads"]
    sec = np.zeros(P, dtype=np.float64)
    cel = np.zeros(P, dtype=np.float64)
    cnt = np.zeros(P, dtype=np.int64)
    done = C.c_int64(0)
    step_s = []
    for it in range(warmup + steps):
        if it == warmup:
            sec[:], cel[:], cnt[:] = 0, 0, 0
        s = lib.spoa_stream_step(h, C.c_int32(reads_per_step), C.c_int32(P), sec.ctypes.data_as(C.c_void_p), cel.ctypes.data_as(C.c_void_p),
                                 cnt.ctypes.data_as(C.c_void_p), C.byref(done))
        if it >= warmup:
            step_s.append(float(s))
    lib.spoa_stream_destroy(h)
    # Wall clock per read position: all threads walk the positions of their window in lock step (same reads per step), so a timed
    # step of `reads_per_step` reads costs step_seconds / reads_per_step per position on the fully loaded machine. (The per-thread
    # times the stream also reports are NOT used for the value: on an over-subscribed box their mean is far below the step's wall
    # time, which is what a real multi-threaded run pays.)
    wall_pos = np.zeros(P, dtype=np.float64)
    wall_cnt = np.zeros(P, dtype=np.int64)
    for k, s_wall in enumerate(step_s):
        for j in range(reads_per_step):
            pidx = ((warmup + k) * reads_per_step + j) % P
            wall_pos[pidx] += s_wall / reads_per_step
            wall_cnt[pidx] += 1
    measured = wall_cnt > 0
    per_pos = np.zeros(P)
    per_pos[measured] = wall_pos[measured] / wall_cnt[measured]
    per_pos[0] = 0.0 if not measured[0] else per_pos[0]  # position 0 is the backbone: no alignment
    todo = [p for p in range(1, P) if not measured[p]]
    if todo:
        # positions the timed steps did not reach: cost grows with the graph, i.e. linearly in the position; the line goes through
        # the measured positions (spoa's own DP-cell counts of the measured positions grow the same way)
        xs = np.array([p for p in range(1, P) if measured[p]])
        if len(xs) >= 2:
            b, a = np.polyfit(xs, per_pos[xs], 1)
            b = max(b, 0.0)
            a = float(np.mean(per_pos[xs]) - b * np.mean(xs))
        else:
            a, b = (float(per_pos[xs[0]]) if len(xs) else 0.0), 0.0
        for p_ in todo:
            per_pos[p_] = max(0.0, a + b * p_)
    t_window = float(per_pos[1:].sum() + per_pos[0])
    value = n_threads / t_window if t_window > 0 else 0.0
    info = {"threads": n_threads, "reads_per_step": reads_per_step, "positions_measured": int(measured[1:].sum()), "positions": int(P - 1),
            "seconds_per_window_per_thread": t_window, "spoa_dp_cells_per_s": float(cel.sum() / max(sum(step_s), 1e-9)),
            "windows_completed": int(done.value), "step_seconds": step_s, "time_base": "wall clock of the timed steps"}
    return value, info


def gpu_reference_leg(wp, n_windows):
    """The UNMODIFIED reference GPU kernels (oracle/_ref/libgwref.so, rebuilt for sm_100a) on a bounded sample of the same
    workload, next to this engine on the same inputs with an identical-output check (BASELINE.md B2/B3). Part of the reference
    arm's line only."""
    import ref_lib
    import torch
    from genomeworks_b200 import cudapoa, synth
    if not (ref_lib.have_gwref() and torch.cuda.is_available()):
        return {"unavailable": "oracle/_ref/libgwref.so not built or no CUDA device"}
    win_nseq, seq_len, data = synth.poa_windows(n_windows, wp["backbone"], wp["reads"], wp["mut"], wp["ins"], wp["dele"], seed0=1000,
                                                max_read_len=wp["max_seq"])
    bm = {"full_band": 0, "static_band": 1, "adaptive_band": 2}[wp["band_mode"]]
    best = None
    for _ in range(2):  # first call warms the reference's context up
        r = ref_lib.ref_poa_run(win_nseq, seq_len, data, wp["max_seq"], wp["reads"], wp["band"], bm, adaptive_storage_factor=wp["factor"],
                                mem_fraction=0.45, max_windows_per_batch=n_windows)
        ms = float(r["timings"][1])
        best = ms if best is None else min(best, ms)
    cfg = cudapoa.make_config(wp["max_seq"], wp["reads"], wp["band"], wp["band_mode"], adaptive_storage_factor=wp["factor"])
    free_b, _ = torch.cuda.mem_get_info()
    b = cudapoa.CudaPoaBatch(wp["reads"], wp["max_seq"], int(free_b * 0.45), config=cfg)
    ours_ms = None
    for _ in range(2):
        b.reset()
        b.add_poa_groups_flat(win_nseq, seq_len, data)
        t0 = time.perf_counter()
        b.generate_poa()
        c, cov, lens, st = b.get_consensus_arrays()
        ours_ms = (time.perf_counter() - t0) * 1e3
    ours = [bytes(c[i, :lens[i]]).decode() for i in range(n_windows)]
    b.close()
    same = ours == r["consensus"] and list(st) == list(r["status"]) and all(
        (cov[i, :lens[i]] == r["coverage"][i]).all() for i in range(n_windows))
    return {"engine": "unmodified cudapoa kernels (oracle/_ref/libgwref.so, sm_100a), generate_poa + get_consensus, host buffers",
            "windows": n_windows, "value": n_windows / (best / 1e3), "unit": "windows/s", "this_engine_same_call": n_windows / (ours_ms / 1e3),
            "identical_outputs": bool(same)}


def run_reference_arm(args, wp, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (3rdparty/spoa, unmodified, oracle/_ref) on the box's
    host cores. Rank 0 only."""
    if rank != 0:
        return
    import ref_lib
    if wp["kind"] != "poa":
        print(json.dumps({"impl": "reference", "unavailable": "no CPU reference implementation is named for the aligner path"}))
        return
    if not ref_lib.have_spoa():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libspoa_ref.so is not built"}))
        return
    cores = os.cpu_count() or 1
    long_reads = wp["backbone"] >= 5000
    if long_reads:
        value, info = spoa_full_window_stream(wp, args.steps, args.warmup)
        step_ms = 1e3 * float(np.mean(info["step_seconds"]))
        full = info["positions_measured"] == info["positions"]
        sample = ("full %d-read windows, one in progress per host thread (%d threads), %d reads fused per step; %d of %d read positions "
                  "timed in the %d timed steps%s; value = threads / sum of per-position seconds; spoa DP cells/s %.3e"
                  % (wp["reads"], info["threads"], info["reads_per_step"], info["positions_measured"], info["positions"], args.steps,
                     "" if full else " (the others by a straight-line fit)", info["spoa_dp_cells_per_s"]))
        per_step = info["threads"]
        extra = {"full_window_stream": {k: v for k, v in info.items() if k != "step_seconds"}, "same_config": bool(full)}
    else:
        per_step = max(8, 8 * cores)
        times, cells, wps = [], 0.0, []
        for it in range(args.warmup + args.steps):
            r = spoa_sample(wp, per_step, 1000 + it * per_step, threads=cores)
            if it >= args.warmup:
                times.append(r["seconds"])
                cells += r["cells"]
                wps.append(r["windows_per_s"])
        value = float(np.mean(wps))
        step_ms = 1e3 * sum(times) / max(len(times), 1)
        sample = "%d full windows per step x %d steps, spoa DP cells/s %.3e" % (per_step, len(times), cells / max(sum(times), 1e-9))
        extra = {"same_config": True}
    line = {
        "impl": "reference", "metric": "poa_consensus_windows_per_s", "value": value, "unit": "windows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int16 (spoa AVX2 SIMD)", "data": "synthetic",
        "config": {"workload": wp["name"], "windows_in_progress_per_step": per_step, "engine": "3rdparty/spoa kNW linear gaps, full DP, all host threads"},
        "cpu_baseline": {"value": value, "unit": "windows/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    line.update(extra)
    if not args.no_extras:
        try:
            line["gpu_reference"] = gpu_reference_leg(wp, 148 if long_reads else 1024)
        except Exception as e:  # pragma: no cover
            line["gpu_reference"] = {"unavailable": "failed: %r" % (e,)}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self, rank, world, local_rank):
        import torch
        self.torch = torch
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _red(self, x, op):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._red(x, self.dist.ReduceOp.MAX) if self.dist is not None else x

    def sum(self, x):
        return self._red(x, self.dist.ReduceOp.SUM) if self.dist is not None else x

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def window_groups(win_nseq, seq_len, data):
    """Per-window ctypes argument arrays for the drop-in add_poa_group entry (pointers into `data`, built once)."""
    base = data.ctypes.data
    groups, off, si = [], 0, 0
    for ns in win_nseq:
        ns = int(ns)
        ptrs = (C.c_char_p * ns)()
        lens = (C.c_int32 * ns)()
        for k in range(ns):
            ptrs[k] = C.cast(base + off, C.c_char_p)
            lens[k] = int(seq_len[si + k])
            off += int(seq_len[si + k])
        si += ns
        groups.append((ns, ptrs, lens))
    return groups


def poa_leg(D, wp, steps, warmup, msa=False, n_windows=0, sample_clocks=False, mem_fraction=0.95):
    """One POA workload on every rank: device-resident `value`, API-shaped `e2e`, roofline numbers."""
    import torch
    from genomeworks_b200 import _lib, cudapoa, synth
    L = _lib.lib()
    cfg = cudapoa.make_config(wp["max_seq"], wp["reads"], wp["band"], wp["band_mode"], adaptive_storage_factor=wp["factor"])
    stream = torch.cuda.Stream()
    free_b, _ = torch.cuda.mem_get_info()
    batch = cudapoa.CudaPoaBatch(wp["reads"], wp["max_seq"], int(free_b * mem_fraction), output_type="msa" if msa else "consensus", config=cfg,
                                 device_id=D.local_rank, stream=stream)
    want = n_windows or wp["windows"]
    n_win = want or min(batch.max_poas, max(batch.resident_windows, 1))
    if want and want > batch.max_poas:
        raise RuntimeError("%s: the batch holds %d windows in the free device memory, the workload has %d" % (wp["key"], batch.max_poas, want))
    win_nseq, seq_len, data = synth.poa_windows(n_win, wp["backbone"], wp["reads"], wp["mut"], wp["ins"], wp["dele"],
                                                seed0=1000 + D.rank * n_win, max_read_len=wp["max_seq"])
    # ---- device-resident timing
    rc, added = batch.add_poa_groups_flat(win_nseq, seq_len, data)
    assert rc == 0 and added == n_win, (rc, added, n_win)
    batch.upload()
    batch.sync()
    for _ in range(warmup):
        batch.launch()
        batch.sync()
    D.barrier()
    sampler = ClockSampler(D.local_rank) if (sample_clocks and D.rank == 0) else None
    if sampler:
        sampler.start()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    l0 = L.gwb200_kernel_launch_count()
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(steps):
            batch.launch()
        ev1.record(stream)
    stream.synchronize()
    D.barrier()
    timed_launches = L.gwb200_kernel_launch_count() - l0
    dev_ms = D.max(ev0.elapsed_time(ev1))
    clocks = sampler.stop() if sampler else None
    cells = batch.last_cells()
    if msa:
        _, st = batch.get_msa()
        st = np.asarray(st)
        lens = None
    else:
        c, cov, lens, st = batch.get_consensus_arrays()
    n_ok = int((st == 0).sum())
    total_windows = D.sum(float(n_win))
    value = total_windows * steps / (dev_ms / 1e3)

    # ---- end to end through the drop-in API: one add_poa_group per window, host buffers, every step
    groups = window_groups(win_nseq, seq_len, data)
    add_group = L.gwb200_poa_batch_add_group
    handle = batch._h

    def e2e_step():
        batch.reset()
        for ns, ptrs, lns in groups:
            rc = add_group(handle, C.c_int32(ns), ptrs, None, lns, None, None)
            assert rc == 0, rc
        batch.generate_poa()
        return batch.get_msa() if msa else batch.get_consensus_arrays()

    for _ in range(max(1, min(warmup, 2))):
        e2e_step()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = e2e_step()
    torch.cuda.synchronize()
    e2e_s = D.max(time.perf_counter() - t0)
    D.barrier()
    if not msa:
        assert (out[2] == lens).all() and (out[3] == st).all()
    e2e_value = total_windows * steps / e2e_s
    h2d = int(((seq_len + 3) // 4 * 4).sum()) + 24 * n_win + 4 * len(seq_len)
    if msa:
        d2h = n_win * cfg.max_sequences_per_poa * cfg.max_consensus_size + n_win * 20
    else:
        d2h = n_win * cfg.max_consensus_size * 3 + n_win * 20
    sb = batch.score_bytes
    res = dict(value=value, e2e=e2e_value, dev_ms=dev_ms, k_ms=dev_ms / steps, cells=cells, score_bytes=sb, n_win=n_win, n_ok=n_ok,
               total_windows=total_windows, h2d=h2d, d2h=d2h, timed_launches=int(timed_launches), clocks=clocks,
               max_poas=batch.max_poas, resident=batch.resident_windows, status=st, lens=lens)
    if not msa:
        res.update(consensus=c, coverage=cov)
    batch.close()
    del batch
    torch.cuda.empty_cache()
    return res


def aligner_leg(D, wp, steps, warmup, sample_clocks=False):
    import torch
    from genomeworks_b200 import _lib, cudaaligner, synth
    L = _lib.lib()
    n = wp["windows"]
    ql, qd, tl, td = synth.aligner_pairs(n, wp["genome"], seed=1 + D.rank)
    qb, tb = bytes(qd), bytes(td)
    pairs, qo, to = [], 0, 0
    for i in range(n):
        pairs.append((qb[qo:qo + ql[i]], tb[to:to + tl[i]]))
        qo += int(ql[i])
        to += int(tl[i])
    stream = torch.cuda.Stream()
    al = cudaaligner.FixedBandAligner(wp["max_bw"], stream=stream, device_id=D.local_rank)

    def step():
        # one call into the engine per batch: the per-pair add_alignment loop and the per-pair result decoding run inside the
        # library, as they do for a C++ caller (a Python loop of 3 x 512 ctypes calls costs as much as the kernel)
        rc, added = al.add_alignments(pairs)
        assert rc == 0 and added == n, (rc, added)
        al.align_all()
        return al.sync_alignments_flat()

    for _ in range(warmup):
        step()
    D.barrier()
    sampler = ClockSampler(D.local_rank) if (sample_clocks and D.rank == 0) else None
    if sampler:
        sampler.start()
    kms, t0 = 0.0, time.perf_counter()
    l0 = L.gwb200_kernel_launch_count()
    last = None
    for _ in range(steps):
        last = step()
        kms += al.last_kernel_ms()
    torch.cuda.synchronize()
    wall = D.max(time.perf_counter() - t0)
    kms = D.max(kms)
    D.barrier()
    clocks = sampler.stop() if sampler else None
    timed_launches = L.gwb200_kernel_launch_count() - l0
    cells = al.last_cells()
    st, opt, offs, act, runs = last
    total = D.sum(float(n))
    out = dict(value=total * steps / (kms / 1e3), e2e=total * steps / wall, k_ms=kms / steps, cells=cells, n=n, total=total,
               n_ok=int((st == 0).sum()), n_opt=int((opt != 0).sum()), timed_launches=int(timed_launches),
               clocks=clocks, h2d=int(ql.sum() + tl.sum()) + 20 * n, d2h=int(len(act)) * 5 + 8 * n, last=last)
    al.close()
    return out


def roofline_obj(key, kernel, cells, bytes_per_cell, k_ms, units):
    peak, peak_src = measured_peaks()
    achieved = cells * bytes_per_cell / (k_ms / 1e3) / 1e9
    tr = ncu_traffic(key)
    traffic = tr["dram_bytes_per_unit"] * units if tr else None
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "traffic_source": (tr or {}).get("source"), "algorithmic_bytes": cells * bytes_per_cell, "peak_source": peak_src, "kernel": kernel,
            "algorithmic_bytes_per_cell": bytes_per_cell, "kernel_ms_per_launch": k_ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "c2", "c4"])
    ap.add_argument("--windows", type=int, default=0, help="windows (or pairs) per GPU per step (default: C3 1600, C2 1024, C4 512)")
    ap.add_argument("--factor", type=float, default=0.0, help="override adaptive_storage_factor of the workload (C3 default 3.0)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C3-MSA / C2 / C4 legs (and gpu_reference in the reference arm)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wp = workload_params(args.workload, args.windows)
    if args.factor > 0 and wp["kind"] == "poa":
        wp["factor"] = args.factor
        wp["name"] = wp["name"].replace("adaptive_storage_factor 3.0", "adaptive_storage_factor %g" % args.factor)

    if args.impl == "reference":
        run_reference_arm(args, wp, rank, world)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    D = Dist(rank, world, local_rank)
    from genomeworks_b200 import _lib
    L = _lib.lib()
    launches0 = L.gwb200_kernel_launch_count()
    warm = max(args.warmup, 3)
    xsteps = max(2, min(args.steps, 3))  # the extra legs are short

    if wp["kind"] == "aligner":
        r = aligner_leg(D, wp, args.steps, warm, sample_clocks=True)
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, aligner_outputs(r))
        if rank == 0:
            line = {
                "metric": "cudaaligner_pairs_per_s", "value": r["value"], "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": r["k_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32 bit-vectors + int32 scores", "data": "synthetic",
                "config": {"workload": wp["name"], "pairs_per_gpu_per_step": r["n"], "max_bandwidth": wp["max_bw"],
                           "l2": "band matrices written per step (%.2f GB) exceed the 126 MB L2" % (r["cells"] * 0.375 / 1e9),
                           "pairs_ok_last_step": r["n_ok"], "pairs_optimal_last_step": r["n_opt"]},
                "dp_cells_per_step_per_gpu": r["cells"], "dp_cells_per_s": r["cells"] * world / (r["k_ms"] / 1e3),
                "roofline": roofline_obj("c4", "myers_banded_kernel", r["cells"], 0.375, r["k_ms"], r["n"]),
                "e2e": {"value": r["e2e"], "unit": "pairs/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"]},
                "gpu_launches": r["timed_launches"], "gpu_launches_total": int(L.gwb200_kernel_launch_count() - launches0), "clocks": r["clocks"],
                "cpu_baseline": {"value": None, "unit": "pairs/s", "cores": 0, "kind": "reference",
                                 "sample": "no CPU implementation of this path is named by the reference (SURVEY.md 8d)"},
            }
            print(json.dumps(line))
        D.close()
        return

    r = poa_leg(D, wp, args.steps, warm, n_windows=args.windows, sample_clocks=True)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, poa_outputs(r))
    extras = {}
    if not args.no_extras and args.workload == "c3":
        try:
            m = poa_leg(D, dict(wp, windows=0), xsteps, 3, msa=True)
            extras["c3_msa"] = {"metric": "poa_msa_windows_per_s", "value": m["value"], "e2e": m["e2e"], "unit": "windows/s",
                                "windows_per_gpu_per_step": m["n_win"], "windows_ok": m["n_ok"], "ms_per_step": m["k_ms"],
                                "roofline_frac": roofline_obj("c3_msa", "poa_window_kernel_v3", m["cells"], m["score_bytes"], m["k_ms"], m["n_win"])["frac"]}
        except Exception as e:  # pragma: no cover
            extras["c3_msa"] = {"failed": repr(e)}
        try:
            w2 = workload_params("c2")
            c2 = poa_leg(D, w2, xsteps, 3, mem_fraction=0.3)
            extras["c2"] = {"metric": "poa_consensus_windows_per_s", "workload": w2["name"], "value": c2["value"], "e2e": c2["e2e"], "unit": "windows/s",
                            "windows_per_gpu_per_step": c2["n_win"], "windows_ok": c2["n_ok"], "ms_per_step": c2["k_ms"],
                            "roofline_frac": roofline_obj("c2", "poa_window_kernel_v3", c2["cells"], c2["score_bytes"], c2["k_ms"], c2["n_win"])["frac"]}
            c2b = poa_leg(D, w2, xsteps, 3, n_windows=16 * 1024, mem_fraction=0.3)
            extras["c2_full_machine"] = {"workload": w2["name"] + " (16384 windows per step: the 1024-window BASELINE batch is 0.43 of one residency)",
                                         "value": c2b["value"], "e2e": c2b["e2e"], "unit": "windows/s", "windows_per_gpu_per_step": c2b["n_win"],
                                         "roofline_frac": roofline_obj("c2", "poa_window_kernel_v3", c2b["cells"], c2b["score_bytes"], c2b["k_ms"], c2b["n_win"])["frac"]}
        except Exception as e:  # pragma: no cover
            extras["c2"] = {"failed": repr(e)}
        try:
            w4 = workload_params("c4")
            a = aligner_leg(D, w4, max(xsteps, 5), 3)
            extras["c4"] = {"metric": "cudaaligner_pairs_per_s", "workload": w4["name"], "value": a["value"], "e2e": a["e2e"], "unit": "pairs/s",
                            "pairs_per_gpu_per_step": a["n"], "pairs_ok": a["n_ok"], "pairs_optimal": a["n_opt"], "ms_per_step": a["k_ms"],
                            "roofline_frac": roofline_obj("c4", "myers_banded_kernel", a["cells"], 0.375, a["k_ms"], a["n"])["frac"]}
        except Exception as e:  # pragma: no cover
            extras["c4"] = {"failed": repr(e)}

    # result gather over NCCL (outside the timed regions): per-window status + consensus length to rank 0
    n_ok = r["n_ok"]
    if world > 1:
        mine = torch.from_numpy(np.stack([r["status"].astype(np.int32), r["lens"].astype(np.int32)], 1)).cuda()
        gathered = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
        D.dist.gather(mine, gathered, dst=0)
        if rank == 0:
            n_ok = int(sum(int((g[:, 0] == 0).sum().item()) for g in gathered))

    if rank == 0:
        sb = r["score_bytes"]
        line = {
            "metric": "poa_consensus_windows_per_s", "value": r["value"], "unit": "windows/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": r["k_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32" if sb == 4 else "int16", "data": "synthetic",
            "config": {"workload": wp["name"], "windows_per_gpu_per_step": r["n_win"], "reads_per_window": wp["reads"],
                       "band_mode": wp["band_mode"], "band_width": wp["band"], "scores": "gap -8 mismatch -6 match 8",
                       "batch_capacity_windows": r["max_poas"], "resident_windows_per_gpu": r["resident"],
                       "parallelism": "windows sharded over %d GPU(s), one Batch per rank, persistent grid (one warp per window)" % world,
                       "l2": "score matrices written per step (%.1f GB) exceed the 126 MB L2; no explicit flush" % (r["cells"] * sb / 1e9),
                       "windows_ok_last_step": n_ok},
            "dp_cells_per_step_per_gpu": r["cells"], "dp_cells_per_s": r["cells"] * world / (r["k_ms"] / 1e3),
            "roofline": roofline_obj(wp["key"], "poa_window_kernel_v3", r["cells"], sb, r["k_ms"], r["n_win"]),
            "e2e": {"value": r["e2e"], "unit": "windows/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "api": "Batch::add_poa_group once per window + generate_poa + get_consensus (host buffers)"},
            "gpu_launches": r["timed_launches"], "gpu_launches_total": int(L.gwb200_kernel_launch_count() - launches0), "clocks": r["clocks"],
        }
        if extras:
            line["extra"] = extras
        if not args.no_cpu_baseline and world >= 1:
            try:
                import ref_lib
                if ref_lib.have_spoa():
                    cores = os.cpu_count() or 1
                    long_reads = wp["backbone"] >= 5000
                    if long_reads:
                        # bounded sample: full-size windows in progress on every host thread, one warm-up step and two timed steps of
                        # two reads each (wall clock); --impl reference runs the same stream over the driver's K steps
                        v, info = spoa_full_window_stream(wp, 2, 1)
                        line["cpu_baseline"] = {"value": v, "unit": "windows/s", "cores": cores, "kind": "reference",
                                                "sample": "unmodified 3rdparty/spoa (AVX2): one full-size window in progress per host thread (%d threads), "
                                                          "%d of %d read positions timed by wall clock (%.1f s), the other positions by a straight line "
                                                          "through them; %.3e spoa DP cells/s; --impl reference times more positions"
                                                          % (info["threads"], info["positions_measured"], info["positions"], sum(info["step_seconds"]),
                                                             info["spoa_dp_cells_per_s"])}
                    else:
                        ns = 8 * cores
                        s = spoa_sample(wp, ns, 1000, threads=cores)
                        line["cpu_baseline"] = {"value": s["windows_per_s"], "unit": "windows/s", "cores": cores, "kind": "reference",
                                                "sample": "%d full windows of the same workload, unmodified 3rdparty/spoa (AVX2), %.1f s, %.3e spoa DP cells/s"
                                                          % (ns, s["seconds"], s["cells"] / s["seconds"])}
                else:
                    line["cpu_baseline"] = {"value": None, "unit": "windows/s", "cores": 0, "kind": "reference",
                                            "sample": "oracle/_ref/libspoa_ref.so not built"}
            except Exception as e:  # pragma: no cover
                line["cpu_baseline"] = {"value": None, "unit": "windows/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (e,)}
        print(json.dumps(line))
    D.close()


if __name__ == "__main__":
    main()
