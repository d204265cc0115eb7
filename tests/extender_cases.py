"""Seeded inputs of the cudaextender tests: the reference's sample data (tests/golden/cudaextender/, the reference's
cudaextender/data/ gzipped) and small synthetic cases, each covering one rule of the ungapped X-drop extension."""
import gzip
import os

import numpy as np

from genomeworks_b200 import cudaextender as ce

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cudaextender")

# the scoring matrix of cudaextender/samples/sample_cudaextender.cpp and tests/Test_CudaextenderEnd2End.cu (row = target code)
SAMPLE_SCORE_MATRIX = np.array([
    91, -114, -31, -123, -1000, -1000, -100, -9100,
    -114, 100, -125, -31, -1000, -1000, -100, -9100,
    -31, -125, 100, -114, -1000, -1000, -100, -9100,
    -123, -31, -114, 91, -1000, -1000, -100, -9100,
    -1000, -1000, -1000, -1000, -1000, -1000, -1000, -9100,
    -1000, -1000, -1000, -1000, -1000, -1000, -1000, -9100,
    -100, -100, -100, -100, -1000, -1000, -100, -9100,
    -9100, -9100, -9100, -9100, -9100, -9100, -9100, -9100], dtype=np.int32)
SAMPLE_XDROP = 910
SAMPLE_THRESHOLD = 3000


def read_fasta_sequence(path):
    with (gzip.open(path, "rt") if path.endswith(".gz") else open(path)) as f:
        return "".join(line.strip() for line in f if not line.startswith(">"))


def golden_sample():
    """(encoded sequence, seeds as SEED_PAIR_DTYPE, expected records as an (m, 4) array of query, target, length, score)."""
    seq = ce.encode_sequence(read_fasta_sequence(os.path.join(GOLDEN_DIR, "sample.fa.gz")))
    seeds = ce.parse_seed_pairs(os.path.join(GOLDEN_DIR, "sample_seed_pairs.csv.gz"))
    gold = ce.parse_scored_segment_pairs(os.path.join(GOLDEN_DIR, "sample_scored_segment_pairs.csv.gz"))
    return seq, seeds, records(gold)


def records(ssp):
    """SCORED_SEGMENT_PAIR_DTYPE array -> (m, 4) int64 array of query, target, length, score."""
    return np.stack([ssp["query_position_in_read"].astype(np.int64), ssp["target_position_in_read"].astype(np.int64),
                     ssp["length"].astype(np.int64), ssp["score"].astype(np.int64)], 1).reshape(-1, 4)


def seed_array(target_positions, query_positions):
    """(n, 2) uint32 array of {query, target} rows, the SeedPair layout."""
    return np.stack([np.asarray(query_positions, dtype=np.uint32), np.asarray(target_positions, dtype=np.uint32)], 1).reshape(-1, 2)


def uniform_matrix(match, mismatch):
    m = np.full(64, mismatch, dtype=np.int32)
    for i in range(4):
        m[i * 8 + i] = match
    return m


def abc_dedup_case():
    """Three segments on diagonal 0 with A containing B and C, B not containing C, sorted A, B, C: the reference's
    thrust::unique_copy compares each with its predecessor, so B goes (inside A) and C stays (not inside B).
    Layout (target == query except at the 10-base mismatch runs X1, X2): R1 [0,50) X1 [50,60) R2 [60,110) X2 [110,120) R3 [120,170).
    Match +100, mismatch -100, xdrop 910: ten mismatches stop an extension, five do not."""
    rng = np.random.default_rng(7)
    t = rng.integers(0, 4, 170).astype(np.int8)
    q = t.copy()
    for a, b in ((50, 60), (110, 120)):
        q[a:b] = (t[a:b] + 1) % 4
    seeds = seed_array([60, 115, 120], [60, 115, 120])
    expected = np.array([[60, 60, 109, 9000], [120, 120, 49, 5000]], dtype=np.int64)
    return dict(query=q, target=t, score_mat=uniform_matrix(100, -100), xdrop=910, no_entropy=True, score_threshold=1000, seeds=seeds), expected


def _mutate(rng, seq, rate, alphabet=4):
    out = seq.copy()
    hit = rng.random(len(seq)) < rate
    out[hit] = (out[hit] + rng.integers(1, alphabet, hit.sum())) % alphabet
    return out


def synthetic_cases():
    """name -> dict(query, target, score_mat, xdrop, no_entropy, score_threshold, seeds)."""
    cases = {}
    rng = np.random.default_rng(2024)
    # related sequences of different lengths, query offset so that most seeds lie on a negative diagonal (t - q < 0)
    t = rng.integers(0, 4, 4099).astype(np.int8)
    q = np.concatenate([rng.integers(0, 4, 700).astype(np.int8), _mutate(rng, t[:2301], 0.04)])
    n = 3000
    tp = rng.integers(0, 2301, n)
    seeds = seed_array(np.concatenate([tp, [0, 4098, 2300, 0]]), np.concatenate([tp + 700, [700, 3000, 3000, 0]]))
    for ne in (False, True):
        cases["related_negative_diagonal_entropy%d" % (not ne)] = dict(query=q, target=t, score_mat=SAMPLE_SCORE_MATRIX, xdrop=910,
                                                                      no_entropy=ne, score_threshold=1000, seeds=seeds)
    # related, same length, positive diagonals, low-complexity stretches (entropy < 1) and codes 4-7 sprinkled in
    t = rng.integers(0, 4, 6007).astype(np.int8)
    t[1000:1300] = 0
    t[2000:2400] = np.tile(np.array([0, 1], dtype=np.int8), 200)
    t[3000:3100] = rng.integers(0, 2, 100)
    q = _mutate(rng, t, 0.03)
    odd = rng.random(len(t)) < 0.01
    q[odd] = rng.integers(4, 8, odd.sum())
    odd = rng.random(len(t)) < 0.005
    t[odd] = rng.integers(4, 8, odd.sum())
    tp = rng.integers(0, 6007, 4000)
    seeds = seed_array(np.concatenate([tp, [0, 6006, 6006]]), np.concatenate([tp, [0, 6006, 0]]))
    for ne in (False, True):
        cases["related_low_complexity_codes_entropy%d" % (not ne)] = dict(query=q, target=t, score_mat=SAMPLE_SCORE_MATRIX, xdrop=910,
                                                                         no_entropy=ne, score_threshold=600, seeds=seeds)
    # unrelated sequences: noise seeds that drop within a few positions
    t = rng.integers(0, 4, 5003).astype(np.int8)
    q = rng.integers(0, 4, 3001).astype(np.int8)
    seeds = seed_array(rng.integers(0, 5003, 5000), rng.integers(0, 3001, 5000))
    cases["unrelated"] = dict(query=q, target=t, score_mat=SAMPLE_SCORE_MATRIX, xdrop=910, no_entropy=False, score_threshold=150,
                              seeds=seeds)
    # xdrop 0, 1 and larger than any score; a matrix with zero entries (ties everywhere); duplicate seeds
    t = rng.integers(0, 4, 1031).astype(np.int8)
    q = _mutate(rng, t, 0.1)
    tp = rng.integers(0, 1031, 300)
    dup = seed_array(np.concatenate([tp, tp[:50]]), np.concatenate([tp, tp[:50]]))
    zero_mat = uniform_matrix(2, 0)
    zero_mat[1 * 8 + 1] = 0
    zero_mat[0 * 8 + 3] = -3
    for xd in (0, 1, 1 << 30):
        cases["xdrop_%d" % xd] = dict(query=q, target=t, score_mat=uniform_matrix(5, -4), xdrop=xd, no_entropy=False, score_threshold=20,
                                      seeds=dup)
        cases["zero_entries_xdrop_%d" % xd] = dict(query=q, target=t, score_mat=zero_mat, xdrop=xd, no_entropy=False, score_threshold=30,
                                                   seeds=dup)
    abc, _ = abc_dedup_case()
    cases["abc_dedup"] = abc
    return cases


def empty_case():
    t = np.zeros(100, dtype=np.int8)
    return dict(query=t, target=t, score_mat=SAMPLE_SCORE_MATRIX, xdrop=910, no_entropy=False, score_threshold=100,
                seeds=np.zeros((0, 2), dtype=np.uint32))
