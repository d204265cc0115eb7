"""cudaextender without a GPU: the CPU oracle reproduces the reference's golden end-to-end data and hand-computed cases of each
extension rule; the C++ headers compile; the engine refuses to run without a device; the reference's sample program compiles
and links against this engine."""
import ctypes as C
import gzip
import os
import subprocess

import numpy as np
import pytest

import extender_cases as ec
import extender_lib as el

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SAMPLE = "/root/reference/cudaextender/samples/sample_cudaextender.cpp"


def run(target, query, mat, seeds, xdrop=1000, thr=1, no_entropy=True):
    t = np.asarray(target, dtype=np.int8)
    q = np.asarray(query, dtype=np.int8)
    s = ec.seed_array([x[0] for x in seeds], [x[1] for x in seeds])  # seeds given as (target, query)
    return el.oracle_run(q, t, mat, xdrop, no_entropy, thr, s)[0].tolist()


def mat_with(entries, default=-50):
    m = np.full(64, default, dtype=np.int32)
    for (a, b), v in entries.items():
        m[a * 8 + b] = v
    return m


def test_oracle_reproduces_golden_sample():
    seq, seeds, gold = ec.golden_sample()
    assert len(seeds) == 143670
    got, kept = el.oracle_run(seq, seq, ec.SAMPLE_SCORE_MATRIX, ec.SAMPLE_XDROP, False, ec.SAMPLE_THRESHOLD,
                                np.asarray(seeds).view(np.uint32).reshape(-1, 2))
    assert got.shape == (1337, 4) and (got == gold).all()
    assert kept > 1337  # many seeds extend to the same segment and are deduplicated


def test_earliest_maximum_wins_ties():
    m = mat_with({(0, 0): 5, (1, 2): -5})
    # S = 5, 0, 5: the best stays at p = 0
    assert run([0, 1, 0], [0, 2, 0], m, [(0, 0)]) == [[0, 0, 0, 5]]


def test_drop_position_is_excluded():
    m = mat_with({(0, 0): 10, (1, 2): -20, (3, 3): 100})
    # S = 10, -10, 90: max - S = 20 at p = 1
    assert run([0, 1, 3], [0, 2, 3], m, [(0, 0)], xdrop=19) == [[0, 0, 0, 10]]
    assert run([0, 1, 3], [0, 2, 3], m, [(0, 0)], xdrop=20) == [[0, 0, 2, 90]]


def test_both_edges():
    m = mat_with({(0, 0): 1})
    # right stops at the end of the sequences, left at position 0
    assert run([0, 0, 0, 0], [0, 0, 0, 0], m, [(2, 2)]) == [[0, 0, 3, 4]]
    # |Q| < |T|: the right side ends with the query
    assert run([0] * 8, [0] * 3, m, [(1, 1)]) == [[0, 0, 2, 3]]


def test_empty_segment_has_length_minus_one():
    m = mat_with({(0, 0): 1})
    assert run([1, 0], [2, 0], m, [(0, 0)], thr=0) == [[0, 0, -1, 0]]


def test_entropy_window_and_count_cut():
    m = mat_with({(0, 0): 10})
    # 20 matching A: total 200 inside [thr, 3 thr] = [100, 300]; counts sum to 20, entropy 0 -> score 0, dropped
    assert run([0] * 20, [0] * 20, m, [(0, 0)], thr=100, no_entropy=False) == []
    assert run([0] * 20, [0] * 20, m, [(0, 0)], thr=100, no_entropy=True) == [[0, 0, 19, 200]]
    # 19 matching A: the counts sum to less than 20 -> entropy 1
    assert run([0] * 19, [0] * 19, m, [(0, 0)], thr=100, no_entropy=False) == [[0, 0, 18, 190]]
    # total above 3 thr: no entropy correction
    assert run([0] * 20, [0] * 20, m, [(0, 0)], thr=60, no_entropy=False) == [[0, 0, 19, 200]]


def test_entropy_score_is_truncated():
    m = mat_with({(0, 0): 10, (1, 1): 10})
    seq = [0, 1] * 10
    # p_A = p_C = 1/2: H = ln 2 / ln4_f32, a little under 1/2 because the f32 ln 4 (0x3FB17218) is above ln 4;
    # 200 H = 99.99999... -> 99
    assert run(seq, seq, m, [(0, 0)], thr=99, no_entropy=False) == [[0, 0, 19, 99]]
    assert run(seq, seq, m, [(0, 0)], thr=100, no_entropy=False) == []


def test_diagonals_sort_as_uint32():
    m = mat_with({(0, 0): 1})
    # diagonal t - q = -5 (0xFFFFFFFB as uint32) sorts after diagonal +5, whatever the seed order
    want = [[0, 5, 4, 5], [5, 0, 4, 5]]
    assert run([0] * 10, [0] * 10, m, [(0, 5), (5, 0)]) == want
    assert run([0] * 10, [0] * 10, m, [(5, 0), (0, 5)]) == want


def test_dedup_compares_with_the_sorted_predecessor():
    case, expected = ec.abc_dedup_case()
    got, kept = el.oracle_run(case["query"], case["target"], case["score_mat"], case["xdrop"], case["no_entropy"],
                                case["score_threshold"], case["seeds"])
    assert kept == 3  # A = [60, 169], B = [60, 109], C = [120, 169]
    # B lies inside its predecessor A and goes; C is not inside B and stays (a comparison with the last kept A would drop it)
    assert got.tolist() == expected.tolist()


def test_synthetic_cases_are_deterministic():
    a = ec.synthetic_cases()
    b = ec.synthetic_cases()
    assert sorted(a) == sorted(b) and len(a) >= 10
    for k in a:
        assert (a[k]["seeds"] == b[k]["seeds"]).all() and (a[k]["query"] == b[k]["query"]).all()


def test_encode_and_parse_helpers():
    from genomeworks_b200 import cudaextender as ce
    assert ce.encode_sequence("ACGTacgtNn&X-").tolist() == [0, 1, 2, 3, 4, 4, 4, 4, 5, 5, 7, 6, 6]
    seeds = ce.parse_seed_pairs(os.path.join(ec.GOLDEN_DIR, "sample_seed_pairs.csv.gz"))
    assert seeds.dtype.itemsize == 8 and seeds[0]["target_position_in_read"] == 18 and seeds[0]["query_position_in_read"] == 18
    assert ce.SCORED_SEGMENT_PAIR_DTYPE.itemsize == 16


def test_create_without_device_is_a_cuda_error():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from genomeworks_b200 import _lib, cudaextender as ce
    h = C.c_void_p()
    m = np.ascontiguousarray(ec.SAMPLE_SCORE_MATRIX)
    rc = _lib.lib().gwb200_extender_create(C.byref(h), m.ctypes.data_as(C.POINTER(C.c_int32)), 64, 910, 0, None, 0, 0, None, None, None)
    assert rc == _lib.E_CUDA and not h.value
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ce.create_extender(ec.SAMPLE_SCORE_MATRIX, 910)


def test_extender_headers_compile_cxx14_clean(tmp_path):
    tu = tmp_path / "tu.cpp"
    tu.write_text("#include <claraparabricks/genomeworks/cudaextender/cudaextender.hpp>\n"
                  "#include <claraparabricks/genomeworks/cudaextender/extender.hpp>\n"
                  "#include <claraparabricks/genomeworks/cudaextender/utils.hpp>\n"
                  "#include <claraparabricks/genomeworks/io/fasta_parser.hpp>\n"
                  "#include <claraparabricks/genomeworks/utils/cudautils.hpp>\n"
                  "#include <claraparabricks/genomeworks/utils/device_buffer.hpp>\n"
                  "#include <claraparabricks/genomeworks/utils/pinned_host_vector.hpp>\n"
                  "using namespace claraparabricks::genomeworks;\n"
                  "static_assert(sizeof(cudaextender::SeedPair) == 8 && sizeof(cudaextender::ScoredSegmentPair) == 16, \"ABI\");\n"
                  "int main() { std::vector<cudaextender::SeedPair> s; cudaextender::parse_seed_pairs(\"/dev/null\", s);\n"
                  "  int8_t e[3]; cudaextender::encode_sequence(e, \"AcN\", 3); return e[0] + e[1] + e[2] == 9 ? 0 : 1; }\n")
    for std in ("-std=c++14", "-std=c++17"):
        r = subprocess.run(["g++", std, "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-I",
                            "/usr/local/cuda/include", str(tu)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr


def test_fasta_parser_reads_the_sample(tmp_path):
    tu = tmp_path / "fa.cpp"
    tu.write_text("#include <claraparabricks/genomeworks/io/fasta_parser.hpp>\n#include <iostream>\n"
                  "int main(int, char** argv) { auto p = claraparabricks::genomeworks::io::create_kseq_fasta_parser(argv[1], 0, false);\n"
                  "  std::cout << p->get_num_seqences() << ' ' << p->get_sequence_by_id(0).name << ' ' << p->get_sequence_by_id(0).seq.size();\n"
                  "  return 0; }\n")
    exe = str(tmp_path / "fa")
    subprocess.check_call(["g++", "-std=c++14", "-I", os.path.join(ROOT, "include"), str(tu), "-o", exe])
    fa = tmp_path / "sample.fa"
    with gzip.open(os.path.join(ec.GOLDEN_DIR, "sample.fa.gz"), "rb") as f:
        fa.write_bytes(f.read())
    out = subprocess.run([exe, str(fa)], capture_output=True, text=True).stdout.split()
    seq = ec.read_fasta_sequence(os.path.join(ec.GOLDEN_DIR, "sample.fa.gz"))
    assert out == ["1", "chr1", str(len(seq))]


@pytest.mark.skipif(not os.path.exists(REF_SAMPLE), reason="reference sources absent")
def test_reference_sample_links_against_this_engine_only(tmp_path):
    import __graft_entry__ as g
    g.build()
    (tmp_path / "cudaextender_file_location.hpp").write_text('#define CUDAEXTENDER_DATA_DIR "cudaextender_data"\n')
    out = str(tmp_path / "sample_cudaextender")
    r = subprocess.run(["g++", "-std=c++14", "-O1", "-I", os.path.join(ROOT, "include"), "-I", str(tmp_path), "-I", "/usr/local/cuda/include",
                        REF_SAMPLE, "-o", out, "-L", os.path.join(ROOT, "genomeworks_b200"), "-lgwb200", "-L", "/usr/local/cuda/lib64",
                        "-lcudart", "-Wl,-rpath," + os.path.join(ROOT, "genomeworks_b200")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    ldd = subprocess.run(["ldd", out], capture_output=True, text=True).stdout
    assert "libgwb200.so" in ldd and "cudaextender" not in ldd and "gwref" not in ldd
