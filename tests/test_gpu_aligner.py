"""GPU parity tests for the banded Myers aligner: CUDA engine (C ABI) vs the CPU oracle and vs the unmodified reference
AlignerGlobalMyersBanded on the same inputs (its outputs stored by reference_outputs.py). Bit-exact: status, is_optimal, basic +
extended CIGAR, edit distance."""
import random

import numpy as np
import pytest

import oracle_lib as ol
import reference_outputs as ref_out
from test_oracle_aligner import KAT

pytestmark = pytest.mark.gpu


def run_ours(pairs, max_bw, mem=-1):
    from genomeworks_b200 import cudaaligner
    al = cudaaligner.FixedBandAligner(max_bw, max_device_memory=mem)
    for q, t in pairs:
        assert al.add_alignment(q, t) == cudaaligner.success
    al.align_all()
    al.sync_alignments()
    res = al.get_alignments()
    cells = al.last_cells()
    al.close()
    return res, cells


def flat(pairs):
    ql = np.array([len(q) for q, _ in pairs], dtype=np.int32)
    tl = np.array([len(t) for _, t in pairs], dtype=np.int32)
    qd = np.frombuffer("".join(q for q, _ in pairs).encode() + b"\0", dtype=np.uint8).copy()
    td = np.frombuffer("".join(t for _, t in pairs).encode() + b"\0", dtype=np.uint8).copy()
    return ql, qd, tl, td


def check_against_oracle(pairs, max_bw):
    res, cells = run_ours(pairs, max_bw)
    tot = 0
    for (q, t), r in zip(pairs, res):
        o = ol.myers_align(q, t, max_bw)
        assert r.status == o["status"]
        assert int(r.is_optimal) == o["is_optimal"]
        assert r.convert_to_cigar() == o["cigar"]
        assert r.convert_to_cigar(extended=True) == o["cigar_extended"]
        assert r.get_edit_distance() == o["edit_distance"]
        tot += o["cells"]
    assert cells == tot
    return res


def check_against_reference(pairs, max_bw, res):
    ql, qd, tl, td = flat(pairs)
    ref = ref_out.ref_aligner_run(ql, qd, tl, td, max_bw)
    assert len(ref["status"]) == len(res)
    for i, r in enumerate(res):
        assert r.status == ref["status"][i], i
        if r.status == 0:
            assert int(r.is_optimal) == ref["is_optimal"][i], i
            assert ref_out.digest(r.convert_to_cigar()) == ref["cigar_basic"][i], i
            assert ref_out.digest(r.convert_to_cigar(extended=True)) == ref["cigar_extended"][i], i
            assert r.get_edit_distance() == ref["edit_distance"][i], i


def mutate(rng, q, n):
    t = list(q)
    for _ in range(n):
        p = rng.randrange(len(t))
        op = rng.randrange(3)
        if op == 0:
            t[p] = rng.choice("ACGT")
        elif op == 1:
            t.insert(p, rng.choice("ACGT"))
        elif len(t) > 1:
            del t[p]
    return "".join(t)


def test_kat_table_on_gpu():
    pairs = [(q, t) for q, t, _, _ in KAT]
    res = check_against_oracle(pairs, 1024)
    for (q, t, cigar, ed), r in zip(KAT, res):
        assert r.convert_to_cigar() == cigar
        if ed is not None:
            assert r.get_edit_distance() == ed
    check_against_reference(pairs, 1024, res)


def test_bw7_corner_cases_on_gpu():
    pairs = [("AACCGGTTAACCGGTTAACCGGTTTT", "AACCGGTTAAAACCCCGGGGGTTAAACGGTT"), ("AACCGGTTAACCGGTTAACCGGTTT", "AACCGGTTAAAACCCCGGGGGTTAACCGGTT")]
    res = check_against_oracle(pairs, 7)
    assert [r.convert_to_cigar() for r in res] == ["10M2I2M2I7M3I5M2D", "10M2I2M2I3M2I3M1I6M1D"]
    assert all(not r.is_optimal for r in res)
    check_against_reference(pairs, 7, res)


@pytest.mark.parametrize("max_bw", [2, 4, 16, 31, 32, 34, 63, 64, 66, 255, 256, 258, 1023, 1024, 1026, 2048])
def test_bandwidth_sweep(max_bw):
    q = "AGGGCGAATATCGCCTCCCGCATTAAGCTGTACCTTCCAGCCCCGCCGGTAATTCCAGCCGGTTGAAGCCACGTCTGCCACGGCACAATGTTTTCGCTTTGCCCGGTGACGGATTTAATCCACCACAG"
    t = "AGGGCGAATATCGCCTCCGCATTAAACTGTACTTCCCAGCCCCGCCAGTATTCCAGCGGGTTGAAGCCGCGTCTGCCACAGCGCAATGTTTTCTTTGCCCACGGTGACCGGTTTAGTCACTACAGTTGC"
    rng = random.Random(max_bw)
    pairs = [(q, t)]
    for L in (200, 900, 1500, 2600):
        a = "".join(rng.choice("ACGT") for _ in range(L))
        pairs.append((a, mutate(rng, a, L // 15)))
        pairs.append((mutate(rng, a, L // 15), a))
    res = check_against_oracle(pairs, max_bw)
    check_against_reference(pairs, max_bw, res)


def test_mixed_batch_random_lengths():
    rng = random.Random(5)
    pairs = []
    for _ in range(120):
        L = rng.choice([1, 2, 31, 32, 33, 64, 65, 100, 333, 1000, 1025, 2048, 3000])
        a = "".join(rng.choice("ACGT") for _ in range(L))
        pairs.append((a, mutate(rng, a, max(0, L // rng.choice([8, 20, 50])))))
    res = check_against_oracle(pairs, 512)
    check_against_reference(pairs, 512, res)


def test_c4_config_subset():
    """BASELINE config C4 shape: 10 000 x <=10 000 bp pairs (cudaaligner/benchmarks/main.cpp:116-129), max_bandwidth 1024."""
    from genomeworks_b200 import synth
    ql, qd, tl, td = synth.aligner_pairs(24, 10000, seed=1)
    qb, tb = bytes(qd), bytes(td)
    pairs, qo, to = [], 0, 0
    for i in range(24):
        pairs.append((qb[qo:qo + ql[i]].decode(), tb[to:to + tl[i]].decode()))
        qo += int(ql[i])
        to += int(tl[i])
    res = check_against_oracle(pairs, 1024)
    assert all(r.status == 0 for r in res)
    check_against_reference(pairs, 1024, res)


def test_c4_full_size_vs_reference():
    """All 512 pairs of config C4 against the reference kernels."""
    from genomeworks_b200 import synth
    ql, qd, tl, td = synth.aligner_pairs(512, 10000, seed=1)
    qb, tb = bytes(qd), bytes(td)
    pairs, qo, to = [], 0, 0
    for i in range(512):
        pairs.append((qb[qo:qo + ql[i]].decode(), tb[to:to + tl[i]].decode()))
        qo += int(ql[i])
        to += int(tl[i])
    res, _ = run_ours(pairs, 1024)
    check_against_reference(pairs, 1024, res)


def test_aligner_api_contracts():
    from genomeworks_b200 import cudaaligner
    with pytest.raises(ValueError):
        cudaaligner.FixedBandAligner(33)  # max_bandwidth % 32 == 1
    with pytest.raises(ValueError):
        cudaaligner.FixedBandAligner(64, max_device_memory=-2)
    # skip case: |target - query| >= max_bandwidth -> status stays uninitialized (myers_gpu.cu:903-912)
    al = cudaaligner.FixedBandAligner(4)
    al.add_alignment("ACGTACGTACGT", "AC")
    al.add_alignment("ACGT", "ACGT")
    al.align_all()
    al.sync_alignments()
    r = al.get_alignments()
    assert r[0].status == cudaaligner.uninitialized and r[1].status == cudaaligner.success and r[1].convert_to_cigar() == "4M"
    al.close()
    # an explicit bandwidth of 0 is honoured, not replaced by the aligner's own (aligner_global_myers_banded.cpp:160-178): the device
    # skips such a pair (max_bandwidth - 1 < |t - q| for every non-empty pair, myers_gpu.cu:903-912); negative -> generic_error
    al = cudaaligner.FixedBandAligner(64)
    assert al.add_alignment("ACGTACGT", "ACGTACGT", max_bandwidth=0) == cudaaligner.success
    assert al.add_alignment("ACGTACGT", "ACGTACGT") == cudaaligner.success
    assert al.add_alignment("ACGT", "ACGT", max_bandwidth=-5) == cudaaligner.generic_error
    al.align_all()
    al.sync_alignments()
    r = al.get_alignments()
    assert r[0].status == cudaaligner.uninitialized and r[1].status == cudaaligner.success and r[1].convert_to_cigar() == "8M"
    al.close()
    # pygenomeworks shim surface
    b = cudaaligner.CudaAlignerBatch(10, 10, 2)
    assert b.add_alignment("AAATC", "TACGTTTT") == 0
    assert b.add_alignment("A" * 11, "A") == cudaaligner.exceeded_max_length
    assert b.add_alignment("TGCA", "ATACGCT") == 0
    assert b.add_alignment("TGCA", "ATACGCT") == cudaaligner.exceeded_max_alignments
    b.align_all()
    out = b.get_alignments()
    assert [a.cigar for a in out] == ["3M1I2M2I", "1I1M2I3M"]


def test_reverse_complement_flags_travel_with_the_alignment():
    """add_alignment(..., reverse_complement_query/target): the Alignment's sequences and format_alignment() are those that
    were aligned (aligner_global_myers_banded.cpp:226-227,413-418), so they agree with the CIGAR."""
    from genomeworks_b200 import cudaaligner
    q, t = "AAACCGTTTTGCA", "TGCAAAACGGATT"
    al = cudaaligner.FixedBandAligner(32)
    assert al.add_alignment(q, t, reverse_complement_query=True) == cudaaligner.success
    assert al.add_alignment(q, t, reverse_complement_target=True) == cudaaligner.success
    al.align_all()
    al.sync_alignments()
    r = al.get_alignments()
    rc = {"A": "T", "C": "G", "G": "C", "T": "A"}
    q_rc = "".join(rc[c] for c in reversed(q))
    t_rc = "".join(rc[c] for c in reversed(t))
    assert r[0].get_query_sequence() == q_rc and r[0].get_target_sequence() == t
    assert r[1].get_query_sequence() == q and r[1].get_target_sequence() == t_rc
    # same result as aligning the reverse-complemented strings directly
    al2 = cudaaligner.FixedBandAligner(32)
    al2.add_alignment(q_rc, t)
    al2.add_alignment(q, t_rc)
    al2.align_all()
    al2.sync_alignments()
    r2 = al2.get_alignments()
    for a, b in zip(r, r2):
        assert a.convert_to_cigar() == b.convert_to_cigar()
        assert a.format_alignment() == b.format_alignment()
        fa = a.format_alignment()
        assert fa[0].replace("-", "") == a.get_query_sequence() and fa[2].replace("-", "") == a.get_target_sequence()
    al.close()
    al2.close()


def test_skewed_and_classic_score_passes_give_the_same_alignments(monkeypatch):
    """The skewed score pass (myers_skew.cuh, bands of >= 128 rows) and the classic one (GWB200_MYERS_SKEW=0) must produce the
    same alignments as the oracle: query longer / shorter than the target, unrelated sequences (every band up to the clamp),
    a long insertion, clamped asymmetric bands, the unbanded case, lengths around block and word boundaries."""
    rng = random.Random(77)

    def seq(n):
        return "".join(rng.choice("ACGT") for _ in range(n))

    pairs = []
    for L in (127, 128, 129, 191, 192, 640, 1000, 2047, 2048, 2049, 4097):
        a = seq(L)
        pairs.append((a, mutate(rng, a, max(1, L // 12))))
        pairs.append((mutate(rng, a, max(1, L // 30)), a))
    a = seq(3000)
    pairs.append((a, a[:1200] + seq(700) + a[1200:]))   # long insertion: query shorter than the target
    pairs.append((a[:900] + seq(500) + a[900:], a))      # long deletion: query longer than the target
    pairs.append((seq(1500), seq(1400)))                 # unrelated: all passes up to the largest band, not optimal
    pairs.append((a, a))                                 # identical
    for max_bw in (130, 256, 800, 1024, 2000):
        got = {}
        for skew in ("1", "0"):
            monkeypatch.setenv("GWB200_MYERS_SKEW", skew)
            res, cells = run_ours(pairs, max_bw)
            got[skew] = [(r.status, int(r.is_optimal), r.convert_to_cigar(extended=True)) for r in res], cells
        assert got["1"] == got["0"], max_bw
        monkeypatch.setenv("GWB200_MYERS_SKEW", "1")
        check_against_oracle(pairs, max_bw)
