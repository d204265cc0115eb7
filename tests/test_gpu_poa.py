"""GPU parity tests for the POA path: the CUDA engine (through the C ABI) against
  (1) the CPU oracle with the device's own fast-math division injected,
  (2) the unmodified reference kernels on the same inputs (their outputs stored by reference_outputs.py),
  (3) the reference's end-to-end golden assembly (Test_CudapoaBatchEnd2End.cu:39-91).
Bit-exact: consensus strings, coverage, MSA rows, status codes."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
import reference_outputs as ref_out
from test_oracle_poa import GOLDEN, assembly, load_sample_windows  # noqa: F401

pytestmark = pytest.mark.gpu


def _cfg8(cfg):
    return np.array([cfg.max_sequence_size, cfg.max_consensus_size, cfg.max_nodes_per_graph, cfg.matrix_sequence_dimension,
                     cfg.alignment_band_width, cfg.max_sequences_per_poa, cfg.band_mode, cfg.max_banded_pred_distance], dtype=np.int32)


def run_ours(win_nseq, seq_len, data, cfg, msa=False, mem=8 << 30, weights=None, gap=-8, mismatch=-6, match=8):
    from genomeworks_b200 import cudapoa
    batch = cudapoa.CudaPoaBatch(cfg.max_sequences_per_poa, cfg.max_sequence_size, mem, output_type="msa" if msa else "consensus", config=cfg,
                                 gap_score=gap, mismatch_score=mismatch, match_score=match)
    rc, added = batch.add_poa_groups_flat(win_nseq, seq_len, data, weights=weights)
    assert rc == 0 and added == len(win_nseq), (rc, added)
    batch.generate_poa()
    if msa:
        rows, st = batch.get_msa()
        out = dict(msa=[[r.decode() for r in w] for w in rows], status=np.array(st))
    else:
        cons, cov, st = batch.get_consensus()
        out = dict(consensus=cons, coverage=cov, status=np.array(st))
    out["cells"] = batch.last_cells()
    out["kernel_ms"] = batch.last_kernel_ms()
    batch.close()
    return out


def assert_same_consensus(a, b, what):
    assert list(a["status"]) == list(b["status"]), what + ": status differs"
    for w, (x, y) in enumerate(zip(a["consensus"], b["consensus"])):
        assert x == y, "%s: consensus of window %d differs" % (what, w)
    for w, (x, y) in enumerate(zip(a["coverage"], b["coverage"])):
        assert list(x) == list(y), "%s: coverage of window %d differs" % (what, w)


def assert_same_as_reference(a, ref, what):
    """`ref`: stored outputs of the reference kernels, consensus and coverage as per-window digests."""
    assert list(a["status"]) == list(ref["status"]), what + ": status differs"
    for w, (x, y) in enumerate(zip(a["consensus"], ref["consensus"])):
        assert ref_out.digest(x) == y, "%s: consensus of window %d differs" % (what, w)
    for w, (x, y) in enumerate(zip(a["coverage"], ref["coverage"])):
        assert ref_out.digest(x) == y, "%s: coverage of window %d differs" % (what, w)


def assert_same_msa_as_reference(a, ref):
    assert list(a["status"]) == list(ref["status"])
    assert [ref_out.digest(rows) for rows in a["msa"]] == ref["msa"]


@pytest.mark.parametrize("band_mode", ["static_band", "adaptive_band", "full_band"])
def test_small_windows_vs_oracle_and_reference(band_mode, device_fdiv):
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(48, 400, 12, 10, 5, 5, seed0=11)
    cfg = cudapoa.make_config(1024, 16, 256, band_mode)
    ours = run_ours(win_nseq, seq_len, data, cfg)
    orc = ol.poa_run(synth.split_windows(win_nseq, seq_len, data), _cfg8(cfg))
    assert_same_consensus(ours, orc, "oracle")
    assert ours["cells"] == int(orc["cells"].sum())
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 1024, 16, 256, cfg.band_mode)
    assert_same_as_reference(ours, ref, "reference")


def test_c2_config_subset_vs_oracle_and_reference(device_fdiv):
    """BASELINE config C2 (1 kb x 16 reads, static band 256, int16 scores) on 96 windows."""
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(96, 1000, 16, 20, 10, 10, seed0=1000, max_read_len=1024)
    cfg = cudapoa.make_config(1024, 16, 256, "static_band")
    ours = run_ours(win_nseq, seq_len, data, cfg)
    assert (ours["status"] == 0).all()
    orc = ol.poa_run(synth.split_windows(win_nseq, seq_len, data), _cfg8(cfg))
    assert_same_consensus(ours, orc, "oracle")
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 1024, 16, 256, 1)
    assert_same_as_reference(ours, ref, "reference")


def test_c2_full_size_vs_reference():
    """All 1024 windows of config C2 against the reference kernels (size-independent check: every output identical)."""
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(1024, 1000, 16, 20, 10, 10, seed0=1000, max_read_len=1024)
    cfg = cudapoa.make_config(1024, 16, 256, "static_band")
    ours = run_ours(win_nseq, seq_len, data, cfg, mem=16 << 30)
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 1024, 16, 256, 1)
    assert_same_as_reference(ours, ref, "reference")
    assert (ours["status"] == 0).all()


@pytest.mark.parametrize("factor", [2.0, 6.0])
def test_c3_long_reads_adaptive_int32(factor, device_fdiv):
    """BASELINE config C3 shape (10 kb x 32 reads would take the CPU oracle minutes; 10 kb x 6 reads, 3 windows):
    adaptive band, int32 scores. factor 2.0 also pins exceeded_adaptive_banded_matrix_size statuses (SURVEY.md fact 3)."""
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(3, 10000, 6, 200, 100, 100, seed0=1000, max_read_len=10240)
    cfg = cudapoa.make_config(10240, 32, 256, "adaptive_band", adaptive_storage_factor=factor)
    ours = run_ours(win_nseq, seq_len, data, cfg, mem=24 << 30)
    orc = ol.poa_run(synth.split_windows(win_nseq, seq_len, data), _cfg8(cfg))
    assert_same_consensus(ours, orc, "oracle")
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 10240, 32, 256, 2, adaptive_storage_factor=factor)
    assert_same_as_reference(ours, ref, "reference")


@pytest.mark.parametrize("band_mode", ["static_band", "adaptive_band"])
def test_msa_vs_oracle_and_reference(band_mode, device_fdiv):
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(24, 300, 10, 10, 5, 5, seed0=77)
    cfg = cudapoa.make_config(1024, 16, 256, band_mode)
    ours = run_ours(win_nseq, seq_len, data, cfg, msa=True)
    windows = synth.split_windows(win_nseq, seq_len, data)
    orc = ol.poa_run(windows, _cfg8(cfg), msa=True)
    assert list(ours["status"]) == list(orc["status"])
    assert ours["msa"] == orc["msa"]
    for rows, reads in zip(ours["msa"], windows):
        for row, rd in zip(rows, reads):
            assert row.replace("-", "") == rd
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 1024, 16, 256, cfg.band_mode, msa=True)
    assert_same_msa_as_reference(ours, ref)


def test_end2end_golden_through_gpu():
    """Test_CudapoaBatchEnd2End.cu:39-91 replayed through the CUDA engine: BatchConfig(1024, 200) = full_band."""
    from genomeworks_b200 import cudapoa
    windows = load_sample_windows()
    win_nseq, seq_len, data = ol.flatten_windows(windows)
    cfg = cudapoa.make_config(1024, 200)
    ours = run_ours(win_nseq, seq_len, data, cfg, mem=8 << 30)
    assert (ours["status"] == 0).all()
    golden = open(GOLDEN + "/sample-golden-value.txt").read().strip()
    assert assembly(ours["consensus"], ours["coverage"]) == golden


def test_batch_api_contracts():
    """Test_CudapoaBatch.cu:70-203 + pygenomeworks/test/test_cudapoa_bindings.py."""
    from genomeworks_b200 import cudapoa
    # zero memory => runtime_error
    with pytest.raises(RuntimeError):
        cudapoa.CudaPoaBatch(10, 1024, 0, config=cudapoa.make_config(1024, 10))
    with pytest.raises(ValueError):
        cudapoa.CudaPoaBatch(10, 1024, -2, config=cudapoa.make_config(1024, 10))
    b = cudapoa.CudaPoaBatch(10, 1024, 1 << 30, config=cudapoa.make_config(1024, 10, 256, "static_band"))
    # 11th read => exceeded_maximum_sequences_per_poa on that entry only
    st, per = b.add_poa_group(["ACGT" * 10] * 11)
    assert st == cudapoa.success
    assert per == [0] * 10 + [cudapoa.exceeded_maximum_sequences_per_poa]
    # 1025-base read => exceeded_maximum_sequence_size on that entry
    st, per = b.add_poa_group(["A" * 1025, "ACGT"])
    assert st == cudapoa.success and per == [cudapoa.exceeded_maximum_sequence_size, 0]
    st, per = b.add_poa_group(["A" * 1025])
    assert st == cudapoa.empty_poa_group
    assert b.total_poas == 3
    b.reset()
    assert b.total_poas == 0
    seq = "A" * 1023
    b.add_poa_group([seq, seq, seq])
    b.generate_poa()
    cons, cov, st = b.get_consensus()
    assert st == [0] and cons == [seq] and cov[0] == [3] * 1023
    with pytest.raises(RuntimeError):
        b.get_msa()
    # graph of 3 reads: 10 nodes / 11 edges (test_cudapoa_bindings.py)
    b.reset()
    b.add_poa_group(["ACTGACTG", "ACTTACTG", "ACTCACTG"])
    b.generate_poa()
    graphs, st = b.get_graphs()
    assert st == [0]
    assert graphs[0].number_of_nodes() == 10 and graphs[0].number_of_edges() == 11
    b.close()


def test_weighted_reads_and_other_scores(device_fdiv):
    """Base weights (Entry::weights) and a non-default scoring scheme, against the oracle and the reference kernels."""
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(20, 350, 9, 10, 5, 5, seed0=4242)
    rng = np.random.RandomState(3)
    weights = rng.randint(1, 40, size=int(seq_len.sum()) + 1).astype(np.int8)
    cfg = cudapoa.make_config(1024, 16, 128, "static_band")
    for (gap, mismatch, match) in [(-8, -6, 8), (-4, -3, 5)]:
        ours = run_ours(win_nseq, seq_len, data, cfg, weights=weights, gap=gap, mismatch=mismatch, match=match)
        windows = synth.split_windows(win_nseq, seq_len, data)
        wl, off = [], 0
        for w in windows:
            ww = []
            for r in w:
                ww.append(weights[off:off + len(r)])
                off += len(r)
            wl.append(ww)
        orc = ol.poa_run(windows, _cfg8(cfg), gap=gap, mismatch=mismatch, match=match, weights=wl)
        assert_same_consensus(ours, orc, "oracle")
        ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 1024, 16, 128, 1, gap=gap, mismatch=mismatch, match=match, weights=weights)
        assert_same_as_reference(ours, ref, "reference")


def test_int32_sizes_long_window_vs_reference():
    """max_sequence_size 12288 => max_nodes 36864 > INT16_MAX: the <int32 score, int32 size> instantiation (cudapoa_limits.hpp:46-53)."""
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(2, 11000, 5, 220, 110, 110, seed0=77, max_read_len=12288)
    cfg = cudapoa.make_config(12288, 8, 256, "adaptive_band", adaptive_storage_factor=6.0)
    ours = run_ours(win_nseq, seq_len, data, cfg, mem=24 << 30)
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 12288, 8, 256, 2, adaptive_storage_factor=6.0, mem_fraction=0.3, max_windows_per_batch=2)
    assert_same_as_reference(ours, ref, "reference")
    assert (ours["status"] == 0).all()


def test_static_band_512_and_128_vs_reference():
    """Other kernel configurations: 1 chunk (band 128, one warp), 3 chunks (band 384: three of four warps take part in the rows)
    and 4 chunks (band 512, four warps x one chunk)."""
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(40, 900, 10, 20, 12, 12, seed0=555, max_read_len=1024)
    for bw in (128, 384, 512):
        cfg = cudapoa.make_config(1024, 16, bw, "static_band")
        ours = run_ours(win_nseq, seq_len, data, cfg)
        ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 1024, 16, bw, 1)
        assert_same_as_reference(ours, ref, "reference bw=%d" % bw)


# ---- traceback band modes (cudapoa_nw_tb_banded.cuh): static / adaptive band with a trace matrix and a score ring ----
@pytest.mark.parametrize("band_mode,max_pred", [("static_band_traceback", 0), ("adaptive_band_traceback", 0), ("static_band_traceback", 100),
                                                ("adaptive_band_traceback", 60)])
def test_traceback_band_modes_vs_oracle_and_reference(band_mode, max_pred, device_fdiv):
    # max_pred 0 -> BatchConfig default 2 x band (int16 traces); 100 / 60 -> int8 traces and a short score ring
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(40, 700, 12, 14, 7, 7, seed0=77)
    cfg = cudapoa.make_config(1024, 16, 128, band_mode, max_pred_dist=max_pred)
    ours = run_ours(win_nseq, seq_len, data, cfg)
    orc = ol.poa_run(synth.split_windows(win_nseq, seq_len, data), _cfg8(cfg))
    assert_same_consensus(ours, orc, "oracle")
    assert ours["cells"] == int(orc["cells"].sum())
    assert (ours["status"] == 0).sum() >= 30
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 1024, 16, 128, cfg.band_mode, max_pred_dist=max_pred)
    assert_same_as_reference(ours, ref, "reference")


def test_traceback_band_mode_msa_and_long_reads_vs_reference(device_fdiv):
    from genomeworks_b200 import cudapoa, synth
    # MSA output through the traceback alignment
    win_nseq, seq_len, data = synth.poa_windows(12, 500, 10, 10, 5, 5, seed0=5)
    cfg = cudapoa.make_config(1024, 16, 256, "adaptive_band_traceback")
    ours = run_ours(win_nseq, seq_len, data, cfg, msa=True)
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 1024, 16, 256, cfg.band_mode, msa=True)
    assert_same_msa_as_reference(ours, ref)
    # 6 kb reads: int32 scores, band starts beyond one row stride (the stray boundary write of set_score_tb lands in other ring slots)
    win_nseq, seq_len, data = synth.poa_windows(6, 6000, 8, 120, 60, 60, seed0=9, max_read_len=6144)
    cfg = cudapoa.make_config(6144, 8, 256, "static_band_traceback")
    ours = run_ours(win_nseq, seq_len, data, cfg, mem=16 << 30)
    orc = ol.poa_run(synth.split_windows(win_nseq, seq_len, data), _cfg8(cfg))
    assert_same_consensus(ours, orc, "oracle")
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 6144, 8, 256, cfg.band_mode)
    assert_same_as_reference(ours, ref, "reference")


def test_c3_shape_storage_factor_status_parity_vs_reference():
    """SURVEY 8d: 10 kb x 32-read windows with the default adaptive_storage_factor 2.0 fail with
    exceeded_adaptive_banded_matrix_size in the reference; the status must be the same here, and at factor 3.0 (bench.py's C3
    configuration) every window succeeds with identical consensus and coverage."""
    from genomeworks_b200 import cudapoa, synth
    win_nseq, seq_len, data = synth.poa_windows(4, 10000, 32, 200, 100, 100, seed0=1000, max_read_len=10240)
    for factor in (2.0, 3.0):
        cfg = cudapoa.make_config(10240, 32, 256, "adaptive_band", adaptive_storage_factor=factor)
        ours = run_ours(win_nseq, seq_len, data, cfg, mem=4 << 30)
        ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 10240, 32, 256, 2, adaptive_storage_factor=factor, mem_fraction=0.05,
                                  max_windows_per_batch=4)
        assert_same_as_reference(ours, ref, "reference, factor %g" % factor)
        if factor == 2.0:
            assert set(ours["status"]) == {cudapoa.exceeded_adaptive_banded_matrix_size}
        else:
            assert (ours["status"] == 0).all()


def test_c3_full_shape_msa_vs_reference():
    """BASELINE config 3 as it is stated: long-read MSA, 10 kb windows x 32 reads, adaptive band, OutputType::msa -- rows and
    statuses bit-exact against the unmodified reference kernels (cudapoa_generate_msa.cuh:127-227 keeps 98 MB/window of per-edge
    read lists; this engine derives the rows from per-read node paths). Also the consensus of the same windows."""
    from genomeworks_b200 import cudapoa, synth
    n = 6
    win_nseq, seq_len, data = synth.poa_windows(n, 10000, 32, 200, 100, 100, seed0=1000, max_read_len=10240)
    cfg = cudapoa.make_config(10240, 32, 256, "adaptive_band", adaptive_storage_factor=3.0)
    ours = run_ours(win_nseq, seq_len, data, cfg, msa=True, mem=12 << 30)
    ref = ref_out.ref_poa_run(win_nseq, seq_len, data, 10240, 32, 256, 2, adaptive_storage_factor=3.0, msa=True, mem_fraction=0.4,
                              max_windows_per_batch=n)
    assert list(ours["status"]) == list(ref["status"]) and (ours["status"] == 0).all()
    windows = synth.split_windows(win_nseq, seq_len, data)
    for w in range(n):
        assert len(ours["msa"][w]) == 32
        assert ref_out.digest(ours["msa"][w]) == ref["msa"][w], "MSA rows of window %d differ" % w
        for row, rd in zip(ours["msa"][w], windows[w]):
            assert row.replace("-", "") == rd
    ours_c = run_ours(win_nseq, seq_len, data, cfg, mem=12 << 30)
    ref_c = ref_out.ref_poa_run(win_nseq, seq_len, data, 10240, 32, 256, 2, adaptive_storage_factor=3.0, mem_fraction=0.4, max_windows_per_batch=n)
    assert_same_as_reference(ours_c, ref_c, "reference")


def test_empty_group_stays_in_the_batch_without_touching_other_windows():
    """A group whose reads are all rejected returns empty_poa_group but still occupies a slot (cudapoa_batch.cuh:139-148); the
    kernels must not read a read length for it (it would be the next window's). Its status is empty_poa_group, the windows
    around it are unaffected."""
    from genomeworks_b200 import cudapoa
    cfg = cudapoa.make_config(1024, 10, 256, "static_band")
    good = ["ACGTTGCAAGCTTGCATGCA" * 10, "ACGTTGCAAGCTAGCATGCA" * 10, "ACGTTGCAAGCTTGCATGCA" * 10]
    for kernel_env in (None,):
        b = cudapoa.CudaPoaBatch(10, 1024, 1 << 30, config=cfg)
        assert b.add_poa_group(good)[0] == cudapoa.success
        assert b.add_poa_group(["A" * 1025])[0] == cudapoa.empty_poa_group
        assert b.add_poa_group(good)[0] == cudapoa.success
        assert b.add_poa_group(["C" * 2000, "G" * 1500])[0] == cudapoa.empty_poa_group
        assert b.total_poas == 4
        b.generate_poa()
        cons, cov, st = b.get_consensus()
        assert st == [0, cudapoa.empty_poa_group, 0, cudapoa.empty_poa_group], st
        assert cons[0] == good[0] and cons[2] == good[0] and cons[1] == "" and cons[3] == ""
        # the flat entry consumes the empty window and goes on: the window <-> result mapping of the caller stays intact
        b.reset()
        groups = [good, ["A" * 1025], good]
        win_nseq = np.array([len(g) for g in groups], dtype=np.int32)
        seq_len = np.array([len(x) for g in groups for x in g], dtype=np.int32)
        data = np.frombuffer(("".join(x for g in groups for x in g) + "\0").encode(), dtype=np.uint8)
        rc, added = b.add_poa_groups_flat(win_nseq, seq_len, data)
        assert rc == cudapoa.empty_poa_group and added == 3 and b.total_poas == 3
        b.generate_poa()
        cons, cov, st = b.get_consensus()
        assert st == [0, cudapoa.empty_poa_group, 0] and cons[0] == good[0] and cons[2] == good[0]
        b.close()
