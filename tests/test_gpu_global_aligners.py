"""GPU: the fixed-size global aligners (Hirschberg-Myers = the deprecated create_aligner factory, and unbanded Myers) through the
C ABI against (a) the reference's known answers, (b) the CPU oracle, (c) the unmodified reference classes on the same inputs (their
outputs stored by reference_outputs.py)."""
import random

import numpy as np
import pytest

import oracle_lib as ol
import reference_outputs as ref_out
from genomeworks_b200 import cudaaligner

pytestmark = pytest.mark.gpu

KAT = [("AAAA", "TTAT", "4M", 3), ("ATAAAAAAAA", "AAAAAAAAA", "1M1D8M", 1), ("AAAAAAAAA", "ATAAAAAAAA", "1M1I8M", 1),
       ("ACTGA", "GCTAG", "3M1D1M1I", 3), ("ACTG", "ACTG", "4M", 0), ("A", "T", "1M", 1),
       ("", "GACTCTCCCCCTCCCCTTTAAATATATAAAAATGGGGTGTAGCTAG", "46I", 46), ("GACTCTCCCCCTCCCCTTTAAATATATAAAAATGGGGTGTAGCTAG", "", "46D", 46),
       ("", "", "", 0)]


def random_pairs(rng, sizes, sub=0.04, indel=0.03):
    out = []
    for n in sizes:
        ref = "".join(rng.choice("ACGT") for _ in range(n))
        q = "".join(c for c in ref if rng.random() > indel)
        t = "".join((c if rng.random() > sub else rng.choice("ACGT")) + (rng.choice("ACGT") if rng.random() < indel else "") for c in ref)
        out.append((q, t))
    return out


def run_ours(pairs, algorithm, max_q=None, max_t=None):
    max_q = max_q if max_q is not None else max(max(len(q) for q, _ in pairs), 1)
    max_t = max_t if max_t is not None else max(max(len(t) for _, t in pairs), 1)
    al = cudaaligner.GlobalAligner(max_q, max_t, len(pairs), algorithm)
    for q, t in pairs:
        assert al.add_alignment(q, t) == cudaaligner.success
    al.align_all()
    al.sync_alignments()
    res = al.get_alignments()
    al.close()
    return res


@pytest.mark.parametrize("algorithm", ["hirschberg_myers", "myers", "ukkonen"])
def test_reference_kat_table(algorithm):
    # Ukkonen cannot handle empty sequences (Test_AlignerGlobal.cpp:151-152)
    kat = [k for k in KAT if (k[0] and k[1]) or algorithm != "ukkonen"]
    res = run_ours([(q, t) for q, t, _, _ in kat], algorithm, max_q=64, max_t=64)
    for a, (q, t, cigar, dist) in zip(res, kat):
        assert a.status == cudaaligner.success and a.is_optimal
        assert a.convert_to_cigar() == cigar and a.get_edit_distance() == dist, (q, t, a.convert_to_cigar())


@pytest.mark.parametrize("algorithm", ["hirschberg_myers", "myers"])
def test_random_pairs_vs_oracle(algorithm):
    rng = random.Random(11)
    pairs = random_pairs(rng, [1, 2, 3, 31, 32, 33, 62, 63, 64, 65, 100, 127, 128, 129, 500, 1000, 1023, 1025, 2500])
    for max_q in (None, 20000):
        res = run_ours(pairs, algorithm, max_q=max_q)
        for a, (q, t) in zip(res, pairs):
            if algorithm == "hirschberg_myers":
                st, failed = ol.hirschberg_myers_align(q, t, max_query_length=max_q if max_q else max(len(x) for x, _ in pairs))
                assert not failed
            else:
                st = ol.myers_full_align(q, t)
            assert a.status == cudaaligner.success
            assert a.convert_to_cigar(extended=True) == ol.states_to_cigar(st, extended=True), (len(q), len(t), max_q)


def test_python_binding_cases_through_cuda_aligner_batch():
    # test_cudaaligner_bindings.py:27-45
    for query, target, cigar in [("AAAAAAA", "TTTTTTT", "7M"), ("AAATC", "TACGTTTT", "3M1I2M2I"), ("TACGTA", "ACATAC", "1D5M1I"),
                                 ("TGCA", "ATACGCT", "1I1M2I3M")]:
        ab = cudaaligner.CudaAlignerBatch(len(query), len(target), 1)
        assert ab.add_alignment(query, target) == cudaaligner.success
        assert ab.add_alignment(query, target) == cudaaligner.exceeded_max_alignments
        ab.align_all()
        als = ab.get_alignments()
        assert len(als) == 1 and als[0].cigar == cigar


def test_admission_and_reset():
    al = cudaaligner.GlobalAligner(10, 12, 2)
    assert al.add_alignment("A" * 11, "A") == cudaaligner.exceeded_max_length
    assert al.add_alignment("A", "A" * 13) == cudaaligner.exceeded_max_length
    assert al.add_alignment("ACGT", "ACGT") == cudaaligner.success
    assert al.get_alignments()[0].status == cudaaligner.uninitialized   # exists before align_all / sync (aligner_global.cpp:131-138)
    assert al.add_alignment("ACGT", "AGT", reverse_complement_query=True) == cudaaligner.success
    assert al.add_alignment("A", "A") == cudaaligner.exceeded_max_alignments
    al.align_all()
    al.sync_alignments()
    a0, a1 = al.get_alignments()
    assert a0.convert_to_cigar() == "4M" and a1.get_query_sequence() == "ACGT" and a1.status == cudaaligner.success
    al.reset()
    assert al.num_alignments() == 0
    with pytest.raises(Exception):
        cudaaligner.GlobalAligner(-1, 5, 1)
    with pytest.raises(Exception):
        cudaaligner.GlobalAligner(5, 5, 0)


@pytest.mark.parametrize("algorithm,ref_alg", [("hirschberg_myers", 0), ("myers", 1), ("ukkonen", 2)])
def test_vs_unmodified_reference_classes(algorithm, ref_alg):
    rng = random.Random(5)
    sizes = [10, 40, 62, 63, 64, 200, 333, 1000, 2000, 4000] if algorithm == "hirschberg_myers" else [10, 40, 63, 64, 200, 333, 1000, 1500]
    pairs = random_pairs(rng, sizes)
    if algorithm != "ukkonen":
        pairs += [("", "ACGT"), ("ACGT", ""), ("A", "CCCCCA"), ("G", "CCCC")]
    else:
        pairs += [(t, q) for q, t in random_pairs(rng, [50, 700])]  # query longer than target: swapped orientation
    max_q = max(len(q) for q, _ in pairs)
    max_t = max(len(t) for _, t in pairs)
    res = run_ours(pairs, algorithm, max_q=max_q, max_t=max_t)
    q_len = np.array([len(q) for q, _ in pairs], dtype=np.int32)
    t_len = np.array([len(t) for _, t in pairs], dtype=np.int32)
    q_data = np.frombuffer(("".join(q for q, _ in pairs) + "\0").encode(), dtype=np.uint8)
    t_data = np.frombuffer(("".join(t for _, t in pairs) + "\0").encode(), dtype=np.uint8)
    ref = ref_out.ref_global_aligner_run(q_len, q_data, t_len, t_data, ref_alg, max_q, max_t)
    assert len(ref["status"]) == len(res)
    for i, a in enumerate(res):
        assert a.status == int(ref["status"][i])
        assert ref_out.digest(a.convert_to_cigar(extended=True)) == ref["cigar_extended"][i], (i, len(pairs[i][0]), len(pairs[i][1]))
        assert a.get_edit_distance() == int(ref["edit_distance"][i])


def test_long_pair_hirschberg_vs_reference_and_banded_distance():
    # 10 k x 10 k, the pygenomeworks long-alignment shape (test_cudaaligner_bindings.py:48-74)
    rng = random.Random(9)
    pairs = random_pairs(rng, [10000, 7000], sub=0.03, indel=0.02)
    max_q = max(len(q) for q, _ in pairs)
    max_t = max(len(t) for _, t in pairs)
    res = run_ours(pairs, "hirschberg_myers", max_q=max_q, max_t=max_t)
    q_len = np.array([len(q) for q, _ in pairs], dtype=np.int32)
    t_len = np.array([len(t) for _, t in pairs], dtype=np.int32)
    q_data = np.frombuffer(("".join(q for q, _ in pairs) + "\0").encode(), dtype=np.uint8)
    t_data = np.frombuffer(("".join(t for _, t in pairs) + "\0").encode(), dtype=np.uint8)
    ref = ref_out.ref_global_aligner_run(q_len, q_data, t_len, t_data, 0, max_q, max_t)
    assert len(ref["status"]) == len(res)
    for i, a in enumerate(res):
        assert ref_out.digest(a.convert_to_cigar(extended=True)) == ref["cigar_extended"][i]


def test_ukkonen_vs_oracle_and_length_difference_status():
    rng = random.Random(21)
    pairs = random_pairs(rng, [3, 30, 64, 100, 257, 900, 2000])
    pairs += [(t, q) for q, t in pairs[:4]]
    res = run_ours(pairs, "ukkonen", max_q=2200, max_t=2200)
    for a, (q, t) in zip(res, pairs):
        st = ol.ukkonen_align(q, t)
        assert a.status == cudaaligner.success and a.is_optimal
        assert a.convert_to_cigar(extended=True) == ol.states_to_cigar(st, extended=True), (len(q), len(t))
    al = cudaaligner.GlobalAligner(100, 100, 2, "ukkonen")
    # more than 10 % of max_target_length apart (aligner_global_ukkonen.cpp:52-60)
    assert al.add_alignment("A" * 50, "A" * 61) == cudaaligner.exceeded_max_alignment_difference
    assert al.add_alignment("A" * 50, "A" * 60) == cudaaligner.success
    al.close()
