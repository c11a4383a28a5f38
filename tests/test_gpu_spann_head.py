"""Row f4 -- SPANN head search on the device, end to end.  tests/cpp/spann_head_dropin.cpp builds a SPANN index with the
unmodified reference (SelectHead -> BuildHead -> BuildSSDIndex, the parameters of Test/src/AlgoTest.cpp:23-42), wraps
its in-memory head index in the real VectorIndex subclass (SPTAG::B200::Index) and
  A. drives the head exactly as SPANNIndex.cpp:197-203 (SearchIndex with K = SearchInternalResultNum) and :259-285
     (RentWorkSpace -> SearchIndexIterativeFromNeareast x n -> End) do, against the reference's CPU head;
  B. puts the wrapped head INTO the reference's own SPANN::Index and runs SPANN::Index::SearchIndex / GetIterator end
     to end (head on the B200, posting lists on the CPU) against an all-CPU copy.
Every (VID, Dist) is compared bit for bit in-process.  No SSD kernels, no posting lists on the device."""
import os
import subprocess
import tempfile

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "oracle", "_ref", "spann_head_dropin")


def test_spann_head_search_on_the_device():
    import __graft_entry__
    __graft_entry__.build_dropin_test()
    if not os.path.exists(EXE):
        pytest.skip("oracle/_ref/spann_head_dropin was not built (needs the reference sources at build time)")
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([EXE, tmp], capture_output=True, text=True, timeout=900, cwd=tmp)
    lines = [l for l in r.stdout.splitlines() if l.startswith(("PASS", "FAIL"))]
    assert r.returncode == 0, r.stdout + r.stderr
    assert len(lines) == 4 and all(l.startswith("PASS") for l in lines), r.stdout
