"""GPU: SPOA_ACCURATE mode (cudapoa_kernels.cuh:508-530: racon's topological sort after every read) makes 3rdparty/spoa a bit-exact
oracle. BASELINE config C1 on the GPU: the 67 sample windows (first 8 reads, Test_CudapoaGenerateMSA2.cu:60-79 pattern) give the
same consensus as spoa on the host; the reference's own MSA case (500 reads of a 50-base backbone, :85-129) gives the same rows.
spoa's outputs are stored by reference_outputs.py."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
import reference_outputs as ref_out
from genomeworks_b200 import cudapoa, synth
from genomeworks_b200._lib import lib
from test_oracle_poa import load_sample_windows

pytestmark = pytest.mark.gpu


@pytest.fixture
def accurate():
    lib().gwb200_poa_set_spoa_accurate(C.c_int32(1))
    yield
    lib().gwb200_poa_set_spoa_accurate(C.c_int32(0))


def test_c1_sample_windows_consensus_equals_spoa(accurate):
    windows = [w[:8] for w in load_sample_windows()]
    win_nseq, seq_len, data = ol.flatten_windows(windows)
    spoa = ref_out.spoa_consensus(win_nseq, seq_len, data, n_threads=4)["consensus"]
    cfg = cudapoa.make_config(1024, 8, 256, "full_band")
    b = cudapoa.CudaPoaBatch(8, 1024, 4 << 30, output_type="consensus", config=cfg)
    rc, added = b.add_poa_groups_flat(win_nseq, seq_len, data)
    assert rc == 0 and added == len(windows)
    b.generate_poa()
    cons, cov, status = b.get_consensus()
    b.close()
    assert all(s == 0 for s in status)
    assert cons == spoa


def test_reference_msa_case_equals_spoa(accurate):
    win_nseq, seq_len, data = synth.poa_windows(1, 50, 500, 10, 5, 10, seed0=1)
    reads = list(synth.split_windows(win_nseq, seq_len, data)[0])
    spoa_rows = ref_out.spoa_msa(reads)
    cfg = cudapoa.make_config(1024, 500, 256, "full_band")
    b = cudapoa.CudaPoaBatch(500, 1024, 8 << 30, output_type="msa", config=cfg)
    rc, added = b.add_poa_groups_flat(win_nseq, seq_len, data)
    assert rc == 0 and added == 1
    b.generate_poa()
    msa, status = b.get_msa()
    b.close()
    assert status[0] == 0 and len(msa[0]) == 500
    assert [r.decode() if isinstance(r, bytes) else r for r in msa[0]] == spoa_rows


def test_default_mode_is_unchanged():
    assert lib().gwb200_poa_get_spoa_accurate() == 0
