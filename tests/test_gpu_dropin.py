"""GPU test of the drop-in boundary itself: `SPTAG::B200::Index` (sptag_b200/csrc/sptag_vector_index.hpp), a real
`class Index : public SPTAG::VectorIndex` compiled against the reference's own headers, is driven through the reference's
types (BasicResult with Meta, QueryResult, ResultIterator, WorkSpace) next to the unmodified reference index it wraps
(oracle/_ref), and every returned result is compared bit for bit in-process by tests/cpp/vector_index_dropin.cpp:
SearchIndex(batch) with and without metadata, the AnnIndex::BatchSearch / Search patterns (Wrappers/src/CoreInterface.cpp
:206-238), p_searchDeleted, SearchIndexWithFilter, RefineSearchIndex, GetIterator (the reference's ResultIterator class
on top of the overridden virtuals), SPANN's head-index pattern (SPANNIndex.cpp:259-285) and a DeleteIndex + re-sync.
The binary is built into oracle/_ref by build() where the reference sources exist."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import data_folder

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "oracle", "_ref", "vector_index_dropin")


@pytest.mark.parametrize("name,k,mc", [("bkt_l2_10k_128", 10, 1024), ("bkt_cos_3k_768", 10, 8192),
                                       ("bkt_l2_deleted_6k_32", 12, 2048), ("bkt_cos_deleted_5k_64", 5, 512),
                                       ("bkt_l2_dups", 10, 1024), ("kdt_l2_10k_64", 10, 2048),
                                       ("bkt_i8_l2_5k_100", 10, 1024), ("bkt_i16_cos_5k_40", 8, 1024),
                                       ("bkt_u8_l2_6k_128", 10, 1024)])
def test_vector_index_subclass_matches_the_reference(name, k, mc):
    import __graft_entry__
    __graft_entry__.build_dropin_test()
    if not os.path.exists(EXE):
        pytest.skip("oracle/_ref/vector_index_dropin was not built (needs the reference sources at build time)")
    folder = data_folder(name)
    q = np.load(os.path.join(folder, "queries.npy"))[:96]
    with tempfile.TemporaryDirectory() as tmp:
        qf = os.path.join(tmp, "q.bin")
        np.ascontiguousarray(q).tofile(qf)
        r = subprocess.run([EXE, folder, qf, str(q.shape[0]), str(k), str(mc)], capture_output=True, text=True,
                           timeout=600)
    lines = [l for l in r.stdout.splitlines() if l.startswith(("PASS", "FAIL"))]
    assert r.returncode == 0, r.stdout + r.stderr
    assert len(lines) >= 9 and all(l.startswith("PASS") for l in lines), r.stdout
