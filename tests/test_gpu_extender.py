"""cudaextender on the GPU: the reference's end-to-end golden data through the host and the device pointer API, the engine
against the CPU oracle and against the stored outputs of the unmodified reference kernels on seeded cases, the status and
exception behaviour of the reference API, and the reference's own sample program built against this engine."""
import gzip
import os
import subprocess

import numpy as np
import pytest

import extender_cases as ec
import extender_lib as el
from reference_outputs import digest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ce():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from genomeworks_b200 import cudaextender
    return cudaextender


def _engine_host(ce, case):
    ext = ce.create_extender(case["score_mat"], case["xdrop"], case["no_entropy"])
    assert ext.extend_async(case["query"], case["target"], case["score_threshold"], case["seeds"]) == ce.success
    assert ext.sync() == ce.success
    out = ec.records(ext.get_scored_segment_pairs())
    ext.close()
    return out


def _engine_device(ce, case):
    import torch
    dev = torch.device("cuda:0")
    n = len(case["seeds"])
    d_q = torch.from_numpy(np.ascontiguousarray(case["query"], dtype=np.int8)).to(dev)
    d_t = torch.from_numpy(np.ascontiguousarray(case["target"], dtype=np.int8)).to(dev)
    seeds = np.ascontiguousarray(np.asarray(case["seeds"]).view(np.uint32).reshape(-1, 2)).view(np.int32)
    d_s = torch.from_numpy(seeds).to(dev)
    d_out = torch.full((max(n, 1), 4), -7, dtype=torch.int32, device=dev)
    d_num = torch.full((1,), -7, dtype=torch.int32, device=dev)
    ext = ce.create_extender(case["score_mat"], case["xdrop"], case["no_entropy"])
    torch.cuda.synchronize()
    assert ext.extend_async_device(d_q, d_t, case["score_threshold"], d_s, d_out, d_num) == ce.success
    torch.cuda.synchronize()
    k = int(d_num.item())
    out = d_out[:k].cpu().numpy().astype(np.int64)
    out[:, :2] &= 0xFFFFFFFF
    ext.close()
    return out


def _oracle(case):
    return el.oracle_run(case["query"], case["target"], case["score_mat"], case["xdrop"], case["no_entropy"], case["score_threshold"],
                           np.asarray(case["seeds"]).view(np.uint32).reshape(-1, 2))[0]


def _reference(case, device_api=False):
    return el.stored_reference_run(np.ascontiguousarray(case["query"], dtype=np.int8), np.ascontiguousarray(case["target"], dtype=np.int8),
                               np.ascontiguousarray(case["score_mat"], dtype=np.int32),
                               case["xdrop"], bool(case["no_entropy"]), case["score_threshold"],
                               np.ascontiguousarray(np.asarray(case["seeds"]).view(np.uint32).reshape(-1, 2)), device_api=device_api)


def _golden_case():
    seq, seeds, gold = ec.golden_sample()
    return dict(query=seq, target=seq, score_mat=ec.SAMPLE_SCORE_MATRIX, xdrop=ec.SAMPLE_XDROP, no_entropy=False,
                score_threshold=ec.SAMPLE_THRESHOLD, seeds=seeds), gold


def test_golden_end_to_end_host_api(ce):
    case, gold = _golden_case()
    got = _engine_host(ce, case)
    assert got.shape == gold.shape == (1337, 4)
    assert (got == gold).all()


def test_golden_end_to_end_device_api_with_torch_tensors(ce):
    case, gold = _golden_case()
    got = _engine_device(ce, case)
    assert got.shape == gold.shape and (got == gold).all()


def test_golden_matches_stored_reference_kernels(ce):
    case, gold = _golden_case()
    ref = _reference(case)
    assert ref["count"] == 1337 and ref["records"] == digest(gold.reshape(-1))


@pytest.mark.parametrize("name", sorted(ec.synthetic_cases()))
def test_engine_matches_oracle_and_reference(ce, name):
    case = ec.synthetic_cases()[name]
    want = _oracle(case)
    host = _engine_host(ce, case)
    dev = _engine_device(ce, case)
    assert host.shape == want.shape and (host == want).all(), name
    assert dev.shape == want.shape and (dev == want).all(), name
    ref = _reference(case)
    assert ref["count"] == len(want) and ref["records"] == digest(want.reshape(-1)), name


def test_abc_dedup_keeps_what_the_reference_keeps(ce):
    case, expected = ec.abc_dedup_case()
    assert (_engine_host(ce, case) == expected).all()


def test_empty_and_duplicate_seed_lists(ce):
    import torch
    case = ec.empty_case()
    assert _engine_host(ce, case).shape == (0, 4)
    # an empty tensor has no device pointer: invalid_input, as for the reference's empty device_buffer
    ext = ce.create_extender(case["score_mat"], case["xdrop"], case["no_entropy"])
    d = torch.zeros(100, dtype=torch.int8, device="cuda")
    o = torch.zeros((1, 4), dtype=torch.int32, device="cuda")
    k = torch.full((1,), -7, dtype=torch.int32, device="cuda")
    assert ext.extend_async_device(d, d, 100, torch.zeros((0, 2), dtype=torch.int32, device="cuda"), o, k) == ce.invalid_input
    ext.close()
    case = ec.synthetic_cases()["xdrop_1"]
    once = dict(case, seeds=case["seeds"][:300])
    assert (_engine_host(ce, once) == _engine_host(ce, case)).all()  # duplicates collapse in the deduplication


def test_status_and_exception_behaviour(ce):
    import torch
    from genomeworks_b200 import _lib
    ext = ce.create_extender(ec.SAMPLE_SCORE_MATRIX, 910, False)
    # sync / results without a preceding host-API call
    assert ext.sync() == ce.invalid_operation
    with pytest.raises(RuntimeError, match="Invalid API call"):
        ext.get_scored_segment_pairs()
    # null device pointers -> invalid_input
    d = torch.zeros(16, dtype=torch.int8, device="cuda")
    s = torch.zeros((1, 2), dtype=torch.int32, device="cuda")
    o = torch.zeros((1, 4), dtype=torch.int32, device="cuda")
    k = torch.zeros(1, dtype=torch.int32, device="cuda")
    assert ext.extend_async_device(None, d, 10, s, o, k) == ce.invalid_input
    assert ext.extend_async_device(d, None, 10, s, o, k) == ce.invalid_input
    assert ext.extend_async_device(d, d, 10, None, o, k) == ce.invalid_input
    assert ext.extend_async_device(d, d, 10, s, None, k) == ce.invalid_input
    assert ext.extend_async_device(d, d, 10, s, o, None) == ce.invalid_input
    # a new host call resets the previous results; reset() forgets them
    case, gold = _golden_case()
    assert ext.extend_async(case["query"], case["target"], 3000, case["seeds"]) == ce.success
    ext.sync()
    assert len(ext.get_scored_segment_pairs()) == 1337
    assert ext.extend_async(case["query"], case["target"], 3000, case["seeds"][:0]) == ce.success
    ext.sync()
    assert len(ext.get_scored_segment_pairs()) == 0
    ext.reset()
    with pytest.raises(RuntimeError):
        ext.get_scored_segment_pairs()
    assert ext.sync() == ce.invalid_operation
    ext.close()
    # another extension type, a short score matrix
    with pytest.raises(RuntimeError, match="not implemented"):
        ce.create_extender(ec.SAMPLE_SCORE_MATRIX, 910, False, extension_type=1)
    with pytest.raises(ValueError):
        ce.create_extender(ec.SAMPLE_SCORE_MATRIX[:63], 910, False)
    assert _lib.E_BAD_ALLOC == -4


def test_pool_too_small_for_the_call(ce):
    case, _ = _golden_case()
    ext = ce.create_extender(ec.SAMPLE_SCORE_MATRIX, 910, False, max_device_memory=1 << 20)
    with pytest.raises(ce.DeviceMemoryAllocationError):
        ext.extend_async(case["query"], case["target"], 3000, case["seeds"])
    ext.close()
    ext = ce.create_extender(ec.SAMPLE_SCORE_MATRIX, 910, False, max_device_memory=64 << 20)
    assert ext.extend_async(case["query"], case["target"], 3000, case["seeds"]) == ce.success
    ext.sync()
    assert len(ext.get_scored_segment_pairs()) == 1337
    ext.close()


def test_measurement_getters(ce):
    case, _ = _golden_case()
    ext = ce.create_extender(ec.SAMPLE_SCORE_MATRIX, 910, False)
    ext.extend_async(case["query"], case["target"], 3000, case["seeds"])
    ext.sync()
    assert ext.last_kernel_ms() > 0
    assert len(case["seeds"]) <= ext.last_positions() < 400 * len(case["seeds"])
    ext.close()


SAMPLE = os.path.join(ROOT, "oracle", "_ref", "sample_cudaextender")


@pytest.mark.skipif(not os.path.exists(SAMPLE), reason="the reference's sample program was not built (reference sources absent)")
@pytest.mark.parametrize("flags", [["-p"], ["-p", "-d"]])
def test_reference_sample_prints_golden_csv(flags):
    r = subprocess.run([SAMPLE] + flags, capture_output=True, text=True, cwd=os.path.join(ROOT, "oracle", "_ref"), timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert lines[0] == "Target Position, Query Position, Length, Score"
    with gzip.open(os.path.join(ec.GOLDEN_DIR, "sample_scored_segment_pairs.csv.gz"), "rt") as f:
        gold = f.read().strip().splitlines()
    assert lines[1:] == gold
