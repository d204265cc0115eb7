"""BASELINE config C1 (plumbing / correctness reference, no GPU): consensus of the reference's sample windows
(cudapoa/data/sample-windows.txt, 67 windows, first 8 reads of each) through the bundled 3rdparty/spoa on the CPU -- the usage
pattern of cudapoa/tests/Test_CudapoaGenerateMSA2.cu:60-79 (createAlignmentEngine(kNW, 8, -6, -8), createGraph, align,
add_alignment, generate_consensus), via oracle/_ref/libspoa_ref.so (unmodified spoa, oracle/spoa_capi.cpp; its outputs are stored by
reference_outputs.py, the streaming test needs the library itself). Checks the plumbing
(67 consensus strings, SURVEY.md 8c: 33 280 bases in total), that every consensus is close to its window's backbone read, and
that the CPU oracle's cudapoa restatement agrees with spoa on almost every base (spoa is not bit-exact with cudapoa: fact 6)."""
import difflib

import numpy as np
import pytest

import oracle_lib as ol
import ref_lib
import reference_outputs as ref_out
from test_oracle_poa import load_sample_windows


def _first8():
    return [w[:8] for w in load_sample_windows()]


def test_c1_sample_windows_through_spoa():
    windows = _first8()
    assert len(windows) == 67
    win_nseq, seq_len, data = ol.flatten_windows(windows)
    r = ref_out.spoa_consensus(win_nseq, seq_len, data, n_threads=4)
    cons = r["consensus"]
    assert len(cons) == 67 and all(len(c) > 0 for c in cons)
    assert sum(len(c) for c in cons) == 33280  # probe run of the survey session (SURVEY.md 8c)
    assert r["cells"] > 0
    # a consensus is never longer than the longest read of its window by more than the insertions the other reads carry
    for w, c in zip(windows, cons):
        assert len(c) <= max(len(r) for r in w) + sum(len(r) for r in w) // 20


def test_c1_oracle_restatement_is_close_to_spoa():
    windows = _first8()
    win_nseq, seq_len, data = ol.flatten_windows(windows)
    spoa = ref_out.spoa_consensus(win_nseq, seq_len, data, n_threads=4)["consensus"]
    cfg8 = ol.batch_config(1024, 8, 256, 0)  # full_band, as the reference's end-to-end test (Test_CudapoaBatchEnd2End.cu:43-51)
    orc = ol.poa_run(windows, cfg8)
    assert (orc["status"] == 0).all()
    same = sum(1 for a, b in zip(spoa, orc["consensus"]) if a == b)
    close = [difflib.SequenceMatcher(None, a, b, autojunk=False).ratio() for a, b in zip(spoa, orc["consensus"])]
    assert same >= 40, same            # most windows agree to the base
    assert min(close) > 0.9, min(close)  # and the others differ in a few positions only


@pytest.mark.skipif(not ref_lib.have_spoa(), reason="oracle/_ref/libspoa_ref.so is built only where the reference sources are")
def test_spoa_stream_interface_matches_whole_window_run():
    """The streaming interface of the reference arm (one window in progress per thread, a few reads per step) fuses the same
    reads as the whole-window call: same DP cell count after the windows complete."""
    import ctypes as C
    windows = _first8()[:8]
    win_nseq, seq_len, data = ol.flatten_windows(windows)
    whole = ref_lib.spoa_consensus(win_nseq, seq_len, data, n_threads=2)
    lib = ref_lib.spoa()
    lib.spoa_stream_create.restype = C.c_void_p
    lib.spoa_stream_step.restype = C.c_double
    h = C.c_void_p(lib.spoa_stream_create(C.c_int32(8), win_nseq.ctypes.data_as(C.c_void_p), seq_len.ctypes.data_as(C.c_void_p),
                                          data.ctypes.data_as(C.c_void_p), C.c_int32(8), C.c_int32(-6), C.c_int32(-8), C.c_int32(2)))
    sec = np.zeros(8)
    cel = np.zeros(8)
    cnt = np.zeros(8, dtype=np.int64)
    done = C.c_int64(0)
    for _ in range(16):  # 2 threads x 4 windows x 8 reads, 2 reads per step
        lib.spoa_stream_step(h, C.c_int32(2), C.c_int32(8), sec.ctypes.data_as(C.c_void_p), cel.ctypes.data_as(C.c_void_p),
                             cnt.ctypes.data_as(C.c_void_p), C.byref(done))
    lib.spoa_stream_destroy(h)
    assert done.value == 8 and (cnt == 8).all()
    assert abs(cel.sum() - whole["cells"]) < 1e-6 * whole["cells"]
