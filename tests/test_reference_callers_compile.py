"""Source-level drop-in check: the reference's OWN caller programs compile and link, unmodified and from where they lie under
/root/reference, against this repo's headers (include/) and library (libgwb200.so) instead of the reference's:
  cudapoa/samples/sample_cudapoa.cpp, cudaaligner/samples/sample_cudaaligner.cpp, cudapoa/benchmarks/{multi,single}_batch.hpp.
Compile/link only. Those checks are skipped where the reference sources are absent."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"

needs_reference = pytest.mark.skipif(not os.path.exists(os.path.join(REF, "cudapoa", "samples", "sample_cudapoa.cpp")),
                                     reason="reference sources absent")


@pytest.fixture(scope="module")
def workdir(tmp_path_factory):
    import __graft_entry__ as g
    g.build()
    d = tmp_path_factory.mktemp("refcallers")
    # the reference generates this header at configure time (cudapoa/CMakeLists.txt); it only carries the data directory
    (d / "file_location.hpp").write_text('#define CUDAPOA_BENCHMARK_DATA_DIR "%s"\n' % os.path.join(REF, "cudapoa", "data"))
    return d


def _gxx(args):
    r = subprocess.run(["g++", "-std=c++14", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include"] + args, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]


@needs_reference
@pytest.mark.parametrize("src", ["cudapoa/samples/sample_cudapoa.cpp", "cudaaligner/samples/sample_cudaaligner.cpp"])
def test_reference_sample_links_against_this_engine(workdir, src):
    out = str(workdir / os.path.basename(src).replace(".cpp", ""))
    _gxx(["-O1", "-I", str(workdir), os.path.join(REF, src), "-o", out, "-L", os.path.join(ROOT, "genomeworks_b200"), "-lgwb200",
          "-L", "/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath," + os.path.join(ROOT, "genomeworks_b200"), "-Wl,-rpath,/usr/local/cuda/lib64"])
    assert os.path.exists(out)
    # the binary must be bound to this engine, not to the reference's libraries
    ldd = subprocess.run(["ldd", out], capture_output=True, text=True).stdout
    assert "libgwb200.so" in ldd and "libcudapoa" not in ldd and "libcudaaligner" not in ldd


@needs_reference
def test_reference_benchmark_helpers_compile(workdir):
    tu = workdir / "tu.cpp"
    tu.write_text('#include <file_location.hpp>\n#include "multi_batch.hpp"\n#include "single_batch.hpp"\nint main() { return 0; }\n')
    _gxx(["-fsyntax-only", "-I", str(workdir), "-I", os.path.join(REF, "cudapoa", "benchmarks"), str(tu)])


def test_nvtx_range_is_real_under_gw_profiling(workdir):
    """GW_NVTX_RANGE (reference cudautils.hpp:155-184): a scoped range object when GW_PROFILING is defined, nothing otherwise."""
    src = workdir / "nvtx_probe.cpp"
    src.write_text('#include <claraparabricks/genomeworks/utils/cudautils.hpp>\n'
                   'int main() { GW_NVTX_RANGE(r, "probe"); return 0; }\n')
    out = str(workdir / "nvtx_probe")
    for flags in ([], ["-DGW_PROFILING"]):
        _gxx(flags + [str(src), "-o", out, "-L", "/usr/local/cuda/lib64", "-lcudart", "-ldl"])
        assert subprocess.run([out]).returncode == 0
    pre = subprocess.run(["g++", "-std=c++14", "-E", "-DGW_PROFILING", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include", str(src)],
                         capture_output=True, text=True).stdout
    assert "nvtx_range r(" in pre.replace("::claraparabricks::genomeworks::cudautils::", "")
