"""Throughput of the ungapped X-drop extender (genomeworks_b200.cudaextender) against the unmodified reference cudaextender
(oracle/_ref/libgwref_ext.so, built by `build()` where the reference sources are present) on two seeded workloads larger than L2:

  related  a 50 Mb target (10 000 random 5 kb backbones of the genomeutils generators, concatenated) and a query made of the same
           windows' mutated reads (generate_random_sequence, about 1/60 each of substitutions, insertions and deletions); the
           seeds are exact 12-mer matches between them (query positions drawn at random, all their target hits), capped at 16 M
  noise    the same sequences and the same number of seeds at uniformly random positions (they drop within a few positions)

For each workload and each implementation: seeds/s of the device-pointer call (CUDA events around extend_async: extension,
sort and deduplication), seeds/s through the host-pointer API (wall clock around extend_async + sync + fetching the results,
inputs in host memory), evaluated positions/s (this engine only: 2 bytes of sequence per position), and whether the two
outputs are identical. Prints one JSON line per workload and a header line with the GPU and its power limit.

    python tools/bench_extender.py [--seeds 16000000] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

K = 12


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return name, power


def workload(n_windows, window, seed):
    from genomeworks_b200 import cudaextender as ce, synth
    _, seq_len, data = synth.poa_windows(n_windows, window, 2, window // 30, window // 30, window // 30, seed0=seed)
    lens = seq_len.reshape(-1, 2)
    starts = np.concatenate([[0], np.cumsum(seq_len)[:-1]]).reshape(-1, 2)
    buf = data[:-1]
    t = np.concatenate([buf[s:s + l] for s, l in zip(starts[:, 0], lens[:, 0])])
    q = np.concatenate([buf[s:s + l] for s, l in zip(starts[:, 1], lens[:, 1])])
    return ce.encode_sequence(t.tobytes()), ce.encode_sequence(q.tobytes())


def kmer_codes(enc):
    x = enc.astype(np.int64) & 3
    n = len(x) - K + 1
    code = np.zeros(n, dtype=np.int64)
    for i in range(K):
        code = (code << 2) | x[i:i + n]
    return code


def kmer_seeds(t, q, cap, rng):
    """Exact 12-mer matches: query positions in random order, every target position with the same 12-mer, until cap seeds."""
    tc, qc = kmer_codes(t), kmer_codes(q)
    order = np.argsort(tc, kind="stable")
    sorted_codes = tc[order]
    qpos = rng.permutation(len(qc))
    out_t, out_q, total = [], [], 0
    for chunk in np.array_split(qpos, 64):
        c = qc[chunk]
        lo = np.searchsorted(sorted_codes, c, "left")
        hi = np.searchsorted(sorted_codes, c, "right")
        cnt = hi - lo
        rep = np.repeat(np.arange(len(chunk)), cnt)
        offs = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        out_t.append(order[lo[rep] + offs])
        out_q.append(chunk[rep])
        total += len(rep)
        if total >= cap:
            break
    tt = np.concatenate(out_t)[:cap]
    qq = np.concatenate(out_q)[:cap]
    return np.stack([qq.astype(np.uint32), tt.astype(np.uint32)], 1)  # rows of {query, target}


def run_engine(t, q, seeds, reps):
    import torch
    import extender_cases as ec
    from genomeworks_b200 import cudaextender as ce
    dev = torch.device("cuda:0")
    ext = ce.create_extender(ec.SAMPLE_SCORE_MATRIX, ec.SAMPLE_XDROP, False)
    d_q = torch.from_numpy(q).to(dev)
    d_t = torch.from_numpy(t).to(dev)
    d_s = torch.from_numpy(seeds.view(np.int32)).to(dev)
    d_out = torch.empty((len(seeds), 4), dtype=torch.int32, device=dev)
    d_num = torch.zeros(1, dtype=torch.int32, device=dev)
    kernel_ms = []
    for r in range(reps + 1):
        torch.cuda.synchronize()
        ext.extend_async_device(d_q, d_t, ec.SAMPLE_THRESHOLD, d_s, d_out, d_num)
        torch.cuda.synchronize()
        if r:
            kernel_ms.append(ext.last_kernel_ms())
    positions = ext.last_positions()
    k = int(d_num.item())
    dev_out = d_out[:k].cpu().numpy()
    host_ms = []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        ext.extend_async(q, t, ec.SAMPLE_THRESHOLD, seeds)
        ext.sync()
        res = ext.get_scored_segment_pairs()
        t1 = time.perf_counter()
        if r:
            host_ms.append((t1 - t0) * 1e3)
    ext.close()
    rec = ec.records(res)
    dv = dev_out.astype(np.int64)
    dv[:, :2] &= 0xFFFFFFFF
    assert dv.shape == rec.shape and (dv == rec).all(), "device and host pointer API disagree"
    return dict(kernel_ms=float(np.median(kernel_ms)), host_ms=float(np.median(host_ms)), positions=positions, records=rec)


def run_reference(t, q, seeds, reps):
    import extender_cases as ec
    import extender_lib
    dev_ms, host_ms = [], []
    rec = None
    for r in range(reps + 1):
        d = extender_lib.reference_run(q, t, ec.SAMPLE_SCORE_MATRIX, ec.SAMPLE_XDROP, False, ec.SAMPLE_THRESHOLD, seeds, device_api=True)
        h = extender_lib.reference_run(q, t, ec.SAMPLE_SCORE_MATRIX, ec.SAMPLE_XDROP, False, ec.SAMPLE_THRESHOLD, seeds, device_api=False)
        if r:
            dev_ms.append(d["timings"][0])
            host_ms.append(h["timings"][1])
        rec = h["records"]
        assert len(d["records"]) == len(rec) and (d["records"] == rec).all()
    return dict(kernel_ms=float(np.median(dev_ms)), host_ms=float(np.median(host_ms)), records=rec)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=16_000_000)
    ap.add_argument("--windows", type=int, default=10_000)
    ap.add_argument("--window", type=int, default=5_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_extender.py measures on a CUDA device; none is present")
    import extender_lib
    name, power = gpu_info()
    lines = [dict(gpu=name, power_limit=power, target_bp=a.windows * a.window, seeds_cap=a.seeds, reps=a.reps,
                  timing="median over reps after one warm-up call")]
    rng = np.random.default_rng(12)
    t, q = workload(a.windows, a.window, 777)
    related = kmer_seeds(t, q, a.seeds, rng)
    n = len(related)
    noise = np.stack([rng.integers(0, len(q), n).astype(np.uint32), rng.integers(0, len(t), n).astype(np.uint32)], 1)
    for wname, seeds in (("related", related), ("noise", noise)):
        seeds = np.ascontiguousarray(seeds)
        e = run_engine(t, q, seeds, a.reps)
        row = dict(workload=wname, target_bp=len(t), query_bp=len(q), seeds=len(seeds), segments=len(e["records"]),
                   engine_kernel_ms=e["kernel_ms"], engine_seeds_per_s_kernel=len(seeds) / e["kernel_ms"] * 1e3,
                   engine_host_ms=e["host_ms"], engine_seeds_per_s_host=len(seeds) / e["host_ms"] * 1e3,
                   engine_positions=e["positions"], engine_positions_per_s=e["positions"] / e["kernel_ms"] * 1e3,
                   engine_seq_bytes_per_s=2 * e["positions"] / e["kernel_ms"] * 1e3)
        if extender_lib.have_reference():
            r = run_reference(t, q, seeds, a.reps)
            row.update(reference_kernel_ms=r["kernel_ms"], reference_seeds_per_s_kernel=len(seeds) / r["kernel_ms"] * 1e3,
                       reference_host_ms=r["host_ms"], reference_seeds_per_s_host=len(seeds) / r["host_ms"] * 1e3,
                       identical_output=bool(len(r["records"]) == len(e["records"]) and (r["records"] == e["records"]).all()),
                       speedup_kernel=r["kernel_ms"] / e["kernel_ms"], speedup_host=r["host_ms"] / e["host_ms"])
        lines.append(row)
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
