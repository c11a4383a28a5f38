"""CPU tests: pin the C restatement (oracle/sptag_oracle.c) against

1. the reference's own known-answer tests (Test/src/AlgoTest.cpp:163-201,
   Test/cuda/distance_tests.cu:15-17, Test/src/DistanceTest.cpp:36-50),
2. committed golden vectors produced by the UNMODIFIED reference (tests/golden/*.npz,
   generator tests/golden/make_golden.py),
3. the reference itself (oracle/_ref/libsptag_ref.so), bit for bit, where it is available.
"""
import glob
import os

import numpy as np
import pytest

import reflib
from conftest import data_folder

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_ref = pytest.mark.skipif(not reflib.have_ref(), reason="oracle/_ref not built on this box")


def _ora_dist(metric, width, a, b):
    L = reflib.ora()
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    return L.ora_distance(metric, reflib.VT_FLOAT, width, a.ctypes.data, b.ctypes.data, a.shape[0])


# ---------------------------------------------------------------------------------------------
# known answers from the reference's tests
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [4, 10, 16, 100, 128, 384, 768])
@pytest.mark.parametrize("width", [16, 8, 4, 1])
def test_static_distances_known_answer(oracle_lib, dim, width):
    # Test/cuda/distance_tests.cu:15-17: vectors (0..), (1..), (2..): L2 = {D, 4D, D}, cosine = {BASE, BASE, BASE-2D}
    v = [np.full(dim, i, np.float32) for i in range(3)]
    assert _ora_dist(0, width, v[0], v[1]) == dim
    assert _ora_dist(0, width, v[0], v[2]) == 4 * dim
    assert _ora_dist(0, width, v[1], v[2]) == dim
    assert _ora_dist(1, width, v[0], v[1]) == 1
    assert _ora_dist(1, width, v[0], v[2]) == 1
    assert _ora_dist(1, width, v[1], v[2]) == 1 - 2 * dim


@pytest.mark.parametrize("width", [16, 8, 4, 1])
def test_simd_tree_close_to_naive(oracle_lib, width):
    # Test/src/DistanceTest.cpp:36-50: SIMD result within 1e-5 relative of the naive scalar loop,
    # cosine convention base^2 - dot, random dimension in [2, 256), values in (-1, 1)
    rng = np.random.default_rng(123)
    for _ in range(200):
        dim = int(rng.integers(2, 256))
        x = rng.uniform(-1, 1, dim).astype(np.float32)
        y = rng.uniform(-1, 1, dim).astype(np.float32)
        l2 = float(((x.astype(np.float64) - y.astype(np.float64)) ** 2).sum())
        cos = 1.0 - float((x.astype(np.float64) * y.astype(np.float64)).sum())
        assert _ora_dist(0, width, x, y) == pytest.approx(l2, rel=1e-5)
        assert _ora_dist(1, width, x, y) == pytest.approx(cos, rel=1e-5, abs=1e-5)


def test_algo_line_known_answer(oracle_lib):
    # Test/src/AlgoTest.cpp:163-201: vec[i] = (i)*10, n = 2000, queries 0/2/4, k = 3, L2
    # expected id sets {0,1,2}, {2,1,3}, {4,3,5}; distances 0, 10, 40
    path = os.path.join(GOLDEN, "algo_line_bkt.npz")
    g = np.load(path)
    files = reflib.IndexFiles.__new__(reflib.IndexFiles)
    _files_from_npz(files, g)
    o = reflib.OracleIndex(files)
    q = np.array([[0] * 10, [2] * 10, [4] * 10], np.float32)
    ids, dists, _ = o.search(q, 3)
    assert [set(r) for r in ids.tolist()] == [{0, 1, 2}, {2, 1, 3}, {4, 3, 5}]
    assert dists.tolist() == [[0, 10, 40], [0, 10, 10], [0, 10, 10]]


# ---------------------------------------------------------------------------------------------
# committed golden vectors (index arrays + the reference's outputs on them)
# ---------------------------------------------------------------------------------------------
def _files_from_npz(files, g):
    files.folder = None
    files.params = {k: str(v) for k, v in zip(g["param_names"].tolist(), g["param_values"].tolist())}
    files.algo = files.params["IndexAlgoType"]
    files.value_type = reflib.VT_OF_NAME[files.params["ValueType"]]
    files.metric = reflib.METRIC_OF_NAME[files.params["DistCalcMethod"]]
    files.vectors = np.ascontiguousarray(g["vectors"])
    files.n, files.dim = files.vectors.shape
    files.graph = np.ascontiguousarray(g["graph"])
    files.degree = files.graph.shape[1]
    files.tree_starts = np.ascontiguousarray(g["tree_starts"])
    files.tree_num = files.tree_starts.shape[0]
    files.nodes = np.ascontiguousarray(g["nodes"])
    files.node_count = files.nodes.shape[0]
    files.deleted = np.ascontiguousarray(g["deleted"]) if "deleted" in g.files else None
    files.num_deleted = int(g["num_deleted"]) if "num_deleted" in g.files else 0


def golden_cases():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))


@pytest.mark.parametrize("name", golden_cases())
def test_oracle_matches_golden_reference_outputs(oracle_lib, name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    files = reflib.IndexFiles.__new__(reflib.IndexFiles)
    _files_from_npz(files, g)
    q = g["queries"]
    for i, mc in enumerate(g["max_checks"].tolist()):
        o = reflib.OracleIndex(files)
        o.max_check = int(mc)
        k = int(g["k"])
        ids, dists, stats = o.search(q, k)
        assert np.array_equal(ids, g["ref_ids"][i]), (name, mc)
        assert np.array_equal(dists.view(np.int32), g["ref_dists"][i].view(np.int32)), (name, mc)
        # WorkSpace counters of the reference (m_iNumberOfCheckedLeaves, NGQueue/SPTQueue sizes)
        assert np.array_equal(stats[:, reflib.ST_CHECKED], g["ref_stats"][i][:, 0]), (name, mc)
        assert np.array_equal(stats[:, reflib.ST_NG_LEFT], g["ref_stats"][i][:, 2]), (name, mc)
        assert np.array_equal(stats[:, reflib.ST_SPT_LEFT], g["ref_stats"][i][:, 3]), (name, mc)


def refine_golden_cases():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "refine", "*.npz")))


@pytest.mark.parametrize("name", refine_golden_cases())
def test_oracle_refine_matches_golden_reference_outputs(oracle_lib, name):
    """SURVEY.md 8 f2: the reference's RefineSearchIndex lists + RebuildNeighbors rows on the committed indexes
    (tests/golden/make_golden_refine.py) against ora_refine_nodes."""
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    r = np.load(os.path.join(GOLDEN, "refine", name + ".npz"))
    files = reflib.IndexFiles.__new__(reflib.IndexFiles)
    _files_from_npz(files, g)
    o = reflib.OracleIndex(files)
    o.max_check_refine = int(r["max_check_refine"])
    num = r["rows"].shape[0]
    rows, ids, dists = o.refine_nodes(0, num, int(r["cef"]), int(r["neighborhood"]), float(r["rng_factor"]))
    assert np.array_equal(ids, r["res_ids"]), name
    assert np.array_equal(dists.view(np.int32), r["res_dists"].view(np.int32)), name
    assert np.array_equal(rows, r["rows"]), name


def rebuild_golden_cases():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "rebuild", "*.npz")))


@pytest.mark.parametrize("name", rebuild_golden_cases())
def test_oracle_rebuild_graph_matches_golden_reference_outputs(oracle_lib, name):
    """SURVEY.md 8 f2: the reference's own NeighborhoodGraph::RebuildGraph (one thread) on the committed indexes' rows and
    on a skewed copy (tests/golden/make_golden_rebuild.py) against ora_rebuild_graph.  Needs no reference at test time."""
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    r = np.load(os.path.join(GOLDEN, "rebuild", name + ".npz"))
    nbh = int(r["neighborhood"])
    own = g["graph"].astype(np.int32).copy()
    own[own < 0] = -1
    assert np.array_equal(reflib.oracle_rebuild_graph(own, nbh)[:, :nbh], r["own_rows"]), name
    assert np.array_equal(reflib.oracle_rebuild_graph(r["skewed_in"], nbh)[:, :nbh], r["skewed_rows"]), name


def quantized_golden_cases():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "quantized", "*.npz")))


@pytest.mark.parametrize("name", quantized_golden_cases())
def test_oracle_matches_golden_quantized_reference_outputs(oracle_lib, tmp_path, name):
    """SURVEY.md 8a row A10 + 8 f2 on committed fixtures (tests/golden/make_golden_quantized.py): an index the reference built
    over PQ / OPQ codes, its SDC and ADC searches on raw queries, ReconstructVector, and RefineNode on the quantized index --
    all produced by the reference, checked against the oracle without the reference present."""
    g = np.load(os.path.join(GOLDEN, "quantized", name + ".npz"))
    files = reflib.IndexFiles.__new__(reflib.IndexFiles)
    _files_from_npz(files, g)
    qpath = str(tmp_path / "quantizer.bin")
    g["quantizer_blob"].tofile(qpath)
    files.quantizer = reflib.Quantizer.read(qpath)
    q, k = g["queries"], int(g["k"])
    for adc, tag in ((False, "sdc"), (True, "adc")):
        for i, mc in enumerate(g["max_checks"].tolist()):
            o = reflib.OracleIndex(files)
            o.max_check = int(mc)
            o.enable_adc = adc
            ids, dists, _ = o.search(q, k)
            assert np.array_equal(ids, g["ref_ids_" + tag][i]), (name, tag, mc)
            assert np.array_equal(dists.view(np.int32), g["ref_dists_" + tag][i].view(np.int32)), (name, tag, mc)
    oq = reflib.OracleQuantizer(files.quantizer)
    rec = oq.reconstruct(files.vectors[:64], g["reconstructed"].dtype)
    assert np.array_equal(rec.view(np.uint8), g["reconstructed"].view(np.uint8)), name
    o = reflib.OracleIndex(files)
    o.max_check_refine = int(g["refine_max_check"])
    num = g["refine_rows"].shape[0]
    rows, ids, dists = o.refine_nodes(0, num, int(g["refine_cef"]), int(g["refine_neighborhood"]), float(g["refine_rng_factor"]))
    assert np.array_equal(ids, g["refine_ids"]), name
    assert np.array_equal(dists.view(np.int32), g["refine_dists"].view(np.int32)), name
    assert np.array_equal(rows, g["refine_rows"]), name


def iterator_golden_cases():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "iterator", "*.npz")))


def check_iterator_golden(name, make_iterators):
    """make_iterators(files, queries, max_check) -> object with next(batch) -> (counts, ids, dists, relaxed) over all
    queries; shared by the oracle (here) and the device (tests/test_gpu_iterator.py)."""
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    r = np.load(os.path.join(GOLDEN, "iterator", name + ".npz"))
    files = reflib.IndexFiles.__new__(reflib.IndexFiles)
    _files_from_npz(files, g)
    nq = int(r["nq"])
    q = np.ascontiguousarray(g["queries"][:nq])
    its = make_iterators(files, q, int(r["max_check"]))
    for s, b in enumerate(r["schedule"].tolist()):
        counts, ids, dists, relaxed = its.next(b)
        assert np.array_equal(counts, r["counts"][:, s]), (name, s)
        assert np.array_equal(ids, r["ids"][:, s, :b]), (name, s)
        assert np.array_equal(np.ascontiguousarray(dists).view(np.int32),
                              np.ascontiguousarray(r["dists"][:, s, :b]).view(np.int32)), (name, s)
        assert np.array_equal(np.asarray(relaxed, bool), r["relaxed"][:, s] != 0), (name, s)
    its.close()


class _OracleIteratorBatch:
    def __init__(self, files, q, max_check):
        o = reflib.OracleIndex(files)
        o.max_check = max_check
        self.its = [o.iterator(qq) for qq in q]

    def next(self, b):
        out = [it.next(b) for it in self.its]
        return (np.array([x[0] for x in out], np.int32), np.stack([x[1] for x in out]),
                np.stack([x[2] for x in out]), np.array([x[3] for x in out]))

    def close(self):
        for it in self.its:
            it.close()


@pytest.mark.parametrize("name", iterator_golden_cases())
def test_oracle_iterator_matches_golden_reference_outputs(oracle_lib, name):
    """SURVEY.md 8 f3: the reference's ResultIterator outputs on the committed indexes
    (tests/golden/make_golden_iterator.py) against ora_iter_*."""
    check_iterator_golden(name, _OracleIteratorBatch)


# ---------------------------------------------------------------------------------------------
# the reference's outputs on seeded inputs, stored in tests/golden/pin/ (tests/golden/make_golden_pin.py)
# ---------------------------------------------------------------------------------------------
ISA_WIDTHS = [(512, 16), (256, 8), (128, 4), (0, 1)]
F32_DIMS = [1, 2, 3, 4, 5, 7, 8, 9, 12, 15, 16, 17, 20, 24, 28, 31, 32, 33, 48, 63, 64, 100, 127, 128, 131, 200,
            256, 384, 768, 960, 1000, 1024]
F32_PAIRS = 300
F32_PAIRS_KEPT = 48          # pairs per dimension whose reference distances are stored
INT_CASES = [(reflib.VT_INT8, np.int8, -127, 128), (reflib.VT_UINT8, np.uint8, 0, 256),
             (reflib.VT_INT16, np.int16, -32768, 32768), (reflib.VT_INT16, np.int16, -3000, 3000)]
INT_DIMS = [1, 3, 4, 5, 15, 16, 17, 31, 32, 33, 47, 48, 63, 64, 65, 79, 80, 95, 96, 100, 127, 128, 131, 192, 200, 256, 258]
INT_PAIRS = 25
QUANTIZER_CASES = [(False, reflib.VT_FLOAT), (True, reflib.VT_FLOAT), (True, reflib.VT_INT8)]
QUANT_ROWS_KEPT, QUANT_RECON_KEPT = 1000, 128


def pin_golden(name):
    return np.load(os.path.join(GOLDEN, "pin", name + ".npz"))


def f32_distance_inputs():
    """(dim, a [F32_PAIRS, dim], b [F32_PAIRS, dim]) per dimension of F32_DIMS."""
    rng = np.random.default_rng(7)
    for dim in F32_DIMS:
        a = rng.standard_normal((F32_PAIRS, dim), dtype=np.float32)
        b = rng.standard_normal((F32_PAIRS, dim), dtype=np.float32)
        yield dim, a, b


def int_distance_inputs(dt, lo, hi):
    """(metric, dim, a, b) in the order the pairs are drawn."""
    rng = np.random.default_rng(9)
    for metric in (0, 1):
        for dim in INT_DIMS:
            for _ in range(INT_PAIRS):
                a = rng.integers(lo, hi, dim).astype(dt)
                b = rng.integers(lo, hi, dim).astype(dt)
                yield metric, dim, a, b


def int_case_key(vt, lo, hi):
    return "vt%d_%d_%d" % (vt, lo, hi)


def quantizer_rows(rtype):
    """Low-rank raw rows (reflib.gen_lowrank's model) drawn without BLAS: the rank-6 product is summed term by term in
    float32, so the rows are the same bits on every CPU."""
    rng = np.random.default_rng(51)
    a = rng.standard_normal((6, 24), dtype=np.float32) / np.float32(np.sqrt(6))
    z = rng.standard_normal((3000, 6), dtype=np.float32)
    x = np.zeros((3000, 24), np.float32)
    for j in range(6):
        x += z[:, j:j + 1] * a[j]
    x += np.float32(0.1) * rng.standard_normal((3000, 24), dtype=np.float32)
    return x if rtype == reflib.VT_FLOAT else np.clip(np.round(x * 32), -127, 127).astype(np.int8)


def quantizer_case_key(opq, rtype):
    return "%s_vt%d" % ("opq" if opq else "pq", rtype)


@pytest.mark.parametrize("metric", [0, 1])
def test_distance_bit_exact_vs_reference_all_trees(oracle_lib, metric):
    """The reference's float DistanceUtils variants (AVX-512, AVX, SSE, scalar) against the oracle's SIMD trees."""
    ref = pin_golden("distance_f32")["dists"][metric]                     # [dim, isa, pair]
    for i, (dim, a, b) in enumerate(f32_distance_inputs()):
        for j, (isa, width) in enumerate(ISA_WIDTHS):
            out_o = np.empty(F32_PAIRS, np.float32)
            oracle_lib.ora_distance_f32_many(metric, width, a.ctypes.data, b.ctypes.data, dim, F32_PAIRS, out_o.ctypes.data)
            assert np.array_equal(out_o[:F32_PAIRS_KEPT].view(np.int32), ref[i, j].view(np.int32)), (dim, isa)


# ---------------------------------------------------------------------------------------------
# the reference itself, on the index folders it built (tests/make_test_data.py)
# ---------------------------------------------------------------------------------------------
@needs_ref
@pytest.mark.parametrize("name", ["algo_line_bkt", "bkt_l2_20k_32", "bkt_cos_10k_128", "bkt_l2_5k_100",
                                  "bkt_l2_3k_30", "bkt_l2_dups", "kdt_l2_10k_64", "bkt2_l2_6k_32", "kdt2_l2_6k_32"])
def test_search_bit_exact_vs_reference(oracle_lib, name):
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    q = np.load(os.path.join(folder, "queries.npy"))
    r = reflib.RefIndex.load(folder)
    width = {512: 16, 256: 8, 128: 4, 0: 1}[reflib.ref().ref_isa()]
    k = 10 if files.n > 100 and name != "algo_line_bkt" else 3
    for mc in [8192, 2048, 512, 64]:
        r.set_param("MaxCheck", mc)
        ids_r, d_r, _ = r.search(q, k, threads=4)
        o = reflib.OracleIndex(files, simd_width=width)
        o.max_check = mc
        ids_o, d_o, _ = o.search(q, k, threads=4)
        assert np.array_equal(ids_r, ids_o), (name, mc)
        assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32)), (name, mc)


@needs_ref
def test_counters_match_reference_workspace(oracle_lib):
    folder = data_folder("bkt_l2_20k_32")
    files = reflib.IndexFiles(folder)
    q = np.load(os.path.join(folder, "queries.npy"))[:40]
    r = reflib.RefIndex.load(folder)
    assert r.enable_stats() == 0
    for mc in [4096, 256]:
        r.set_param("MaxCheck", mc)
        o = reflib.OracleIndex(files)
        o.max_check = mc
        _, _, st = o.search(q, 10)
        for i in range(q.shape[0]):
            _, _, rs = r.search_one_stats(q[i], 10)
            assert rs[0] == st[i, reflib.ST_CHECKED]
            assert rs[2] == st[i, reflib.ST_NG_LEFT]
            assert rs[3] == st[i, reflib.ST_SPT_LEFT]


# ---------------------------------------------------------------------------------------------
# PQ / OPQ quantized indexes (SURVEY.md 8a row A10)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("opq,rtype", QUANTIZER_CASES)
def test_quantizer_bit_exact_vs_reference(oracle_lib, tmp_path, opq, rtype):
    """PQ / OPQ QuantizeVector, SDC L2, ReconstructVector and re-quantisation of the reference, on the stored quantizer."""
    g = pin_golden("quantizer_" + quantizer_case_key(opq, rtype))
    xs = quantizer_rows(rtype)
    path = str(tmp_path / "q.bin")
    g["quantizer_blob"].tofile(path)
    oq = reflib.OracleQuantizer(reflib.Quantizer.read(path))
    co = oq.encode(xs)
    assert np.array_equal(co[:QUANT_ROWS_KEPT], g["codes"])                   # QuantizeVector (incl. the OPQ rotation)
    do = np.array([oq.l2(co[i], co[i + 1]) for i in range(500)], np.float32)
    assert np.array_equal(do.view(np.int32), g["sdc_l2"].view(np.int32))     # SDC table sum
    ro = oq.reconstruct(co, xs.dtype)
    # ReconstructVector (incl. the OPQ back-rotation + cast) and what RefineNode makes of it (SetTarget)
    assert np.array_equal(ro[:QUANT_RECON_KEPT].view(np.uint8), g["reconstructed"].view(np.uint8))
    assert np.array_equal(oq.encode(ro)[:QUANT_ROWS_KEPT], g["recoded"])


@needs_ref
@pytest.mark.parametrize("name", ["bkt_pq_6k_32", "bkt_opq_6k_48", "bkt_opq_i8_8k_100"])
def test_quantized_search_bit_exact_vs_reference(oracle_lib, name):
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    assert files.quantizer is not None and files.value_type == reflib.VT_UINT8
    q = np.load(os.path.join(folder, "queries.npy"))
    r = reflib.RefIndex.load(folder)
    for mc in [8192, 1024, 128]:
        r.set_param("MaxCheck", mc)
        ids_r, d_r, _ = r.search_each(q, 10, threads=4)   # per-query overload on RAW queries
        o = reflib.OracleIndex(files)
        o.max_check = mc
        ids_o, d_o, _ = o.search(q, 10, threads=4)
        assert np.array_equal(ids_r, ids_o), (name, mc)
        assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32)), (name, mc)


# ---------------------------------------------------------------------------------------------
# int8 / uint8 element types (DistanceUtils.cpp:305-558, :684-874)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("vt,dt,lo,hi", INT_CASES)
def test_integer_distance_bit_exact_vs_reference(oracle_lib, vt, dt, lo, hi):
    """The reference's integer DistanceUtils, run through its own cpuid dispatch; `width` is the SIMD tree it picked."""
    g = pin_golden("distance_int")
    width = int(g["width"])
    if vt == reflib.VT_INT16 and width != 16:
        pytest.skip("the int16 restatement covers the AVX-512 variants only")
    ref = g[int_case_key(vt, lo, hi)]
    for i, (metric, dim, a, b) in enumerate(int_distance_inputs(dt, lo, hi)):
        o = np.float32(oracle_lib.ora_distance(metric, vt, width, a.ctypes.data, b.ctypes.data, dim))
        assert ref[i].view(np.int32) == o.view(np.int32), (vt, metric, dim)


@needs_ref
@pytest.mark.parametrize("name", ["bkt_i8_cos_6k_64", "bkt_u8_l2_6k_128", "bkt_i8_l2_5k_100", "kdt_i8_l2_6k_32",
                                  "bkt_i16_l2_5k_64", "bkt_i16_cos_5k_40", "bkt_i16_l2_4k_27", "kdt_i16_l2_5k_32"])
def test_integer_index_search_bit_exact_vs_reference(oracle_lib, name):
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    q = np.load(os.path.join(folder, "queries.npy"))
    r = reflib.RefIndex.load(folder)
    width = {512: 16, 256: 8, 128: 4, 0: 1}[reflib.ref().ref_isa()]
    for mc in [8192, 1024, 128]:
        r.set_param("MaxCheck", mc)
        ids_r, d_r, _ = r.search(q, 10, threads=4)
        o = reflib.OracleIndex(files, simd_width=width)
        o.max_check = mc
        ids_o, d_o, _ = o.search(q, 10, threads=4)
        assert np.array_equal(ids_r, ids_o), (name, mc)
        assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32)), (name, mc)


@needs_ref
@pytest.mark.parametrize("name", ["bkt_pq_6k_32", "bkt_opq_6k_48", "bkt_opq_i8_8k_100"])
def test_quantized_adc_search_bit_exact_vs_reference(oracle_lib, name):
    # VectorIndex::SetQuantizerADC(true): asymmetric distance tables (PQQuantizer.h:114-119, :141-157)
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    q = np.load(os.path.join(folder, "queries.npy"))
    r = reflib.RefIndex.load(folder)
    r.set_adc(True)
    for mc in [8192, 256]:
        r.set_param("MaxCheck", mc)
        ids_r, d_r, _ = r.search_each(q, 10, threads=4)
        o = reflib.OracleIndex(files)
        o.max_check = mc
        o.enable_adc = True
        ids_o, d_o, _ = o.search(q, 10, threads=4)
        assert np.array_equal(ids_r, ids_o), (name, mc)
        assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32)), (name, mc)


# ---------------------------------------------------------------------------------------------
# SearchIndexWithFilter (SURVEY.md 8 f3; Test/src/FilterTest.cpp:40-60)
# ---------------------------------------------------------------------------------------------
def test_filter_known_answer(oracle_lib):
    # FilterTest.cpp: line data, queries (0..),(2..),(4..), k = 3, the filter rejects metadata "2" -> id 2 never returned
    g = np.load(os.path.join(GOLDEN, "algo_line_bkt.npz"))
    files = reflib.IndexFiles.__new__(reflib.IndexFiles)
    _files_from_npz(files, g)
    allowed = np.ones(files.n, np.uint8)
    allowed[2] = 0
    o = reflib.OracleIndex(files)
    o.filter = allowed
    ids, _, _ = o.search(np.array([[0] * 10, [2] * 10, [4] * 10], np.float32), 3)
    assert 2 not in ids.ravel().tolist()
    assert ids.tolist() == [[0, 1, 3], [1, 3, 0], [4, 3, 5]]


@needs_ref
@pytest.mark.parametrize("name", ["algo_line_bkt", "bkt_l2_20k_32", "bkt_l2_dups", "bkt_cos_10k_128"])
def test_filtered_search_bit_exact_vs_reference(oracle_lib, name):
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    q = np.load(os.path.join(folder, "queries.npy"))[:100]
    allowed = (np.random.default_rng(5).random(files.n) < 0.5).astype(np.uint8)
    r = reflib.RefIndex.load(folder)
    k = 3 if name == "algo_line_bkt" else 10
    for mc in [0, 512]:
        ids_r, d_r = r.search_filtered(q, k, allowed, max_check=mc, threads=4)
        o = reflib.OracleIndex(files)
        o.filter = allowed
        if mc:
            o.max_check = mc
        ids_o, d_o, _ = o.search(q, k, threads=4)
        assert np.array_equal(ids_r, ids_o), (name, mc)
        assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32)), (name, mc)
        assert allowed[ids_r[ids_r >= 0]].all()


@needs_ref
@pytest.mark.parametrize("name,cef,mcr", [("bkt_l2_dups", 20, 256), ("bkt_l2_20k_32", 100, 2048),
                                          ("bkt_cos_3k_768", 1000, 8192), ("kdt_l2_10k_64", 64, 1024),
                                          ("bkt_i8_cos_6k_64", 50, 512), ("bkt_u8_l2_6k_128", 50, 512),
                                          ("bkt_l2_3k_30", 64, 1024), ("bkt_i16_l2_4k_27", 40, 512),
                                          ("bkt_i16_cos_5k_40", 40, 512)])
def test_refine_bit_exact_vs_reference(oracle_lib, name, cef, mcr):
    """NeighborhoodGraph::RefineNode per node on the loaded index (RefineSearchIndex + RebuildNeighbors run by the
    reference itself) against the oracle's restatement."""
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    r = reflib.RefIndex.load(folder)
    r.set_param("MaxCheckForRefineGraph", mcr)
    o = reflib.OracleIndex(files)
    o.max_check_refine = mcr
    num = min(files.n, 300)
    first = files.n // 3
    for nbh, factor in [(files.degree, 1.0), (12, 1.3)]:
        rows_r, ids_r, d_r = r.refine_nodes(first, num, cef, nbh, factor, threads=4)
        rows_o, ids_o, d_o = o.refine_nodes(first, num, cef, nbh, factor, threads=4)
        assert np.array_equal(ids_r, ids_o), name
        assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32)), name
        assert np.array_equal(rows_r, rows_o), name


@needs_ref
@pytest.mark.parametrize("name,cef,mcr", [("bkt_pq_6k_32", 64, 1024), ("bkt_opq_6k_48", 100, 2048),
                                          ("bkt_opq_i8_8k_100", 40, 512)])
def test_quantized_refine_bit_exact_vs_reference(oracle_lib, name, cef, mcr):
    """RefineNode on a quantized index (NeighborhoodGraph.h:538-543): the node's code row is reconstructed, SetTarget
    quantizes the reconstruction again, RefineSearchIndex runs on that and RebuildNeighbors compares code rows through
    the quantizer's distance -- the reference itself against the oracle's restatement.  (ADC off, as at build time:
    with SetQuantizerADC(true) the reference's RebuildNeighbors hands two CODE rows to the ADC branch of L2Distance,
    which reads the first one as a float table -- out of bounds; neither the oracle nor the device offers that.)"""
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    r = reflib.RefIndex.load(folder)
    r.set_param("MaxCheckForRefineGraph", mcr)
    o = reflib.OracleIndex(files)
    o.max_check_refine = mcr
    num = min(files.n, 300)
    first = files.n // 3
    for nbh, factor in [(files.degree, 1.0), (12, 1.3)]:
        rows_r, ids_r, d_r = r.refine_nodes(first, num, cef, nbh, factor, threads=4)
        rows_o, ids_o, d_o = o.refine_nodes(first, num, cef, nbh, factor, threads=4)
        assert np.array_equal(ids_r, ids_o), name
        assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32)), name
        assert np.array_equal(rows_r, rows_o), name


@needs_ref
@pytest.mark.parametrize("name,nbh", [("bkt_l2_20k_32", 16), ("bkt_l2_10k_128", 16), ("bkt_l2_dups", 16), ("kdt_l2_10k_64", 8),
                                      ("bkt_i8_cos_6k_64", 12)])
def test_rebuild_graph_bit_exact_vs_reference(oracle_lib, name, nbh):
    """NeighborhoodGraph::RebuildGraph (EnableRebuild's in-degree repair, NeighborhoodGraph.h:404-456) run by the
    reference itself, single-threaded, on rows of 2 x nbh candidates -- the index's own graph rows (32 wide), a widened
    copy with -1 padding, and a copy with a skewed in-degree -- against the oracle's restatement."""
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    r = reflib.RefIndex.load(folder)
    g0 = files.graph[:, :2 * nbh].copy()
    g0[g0 < 0] = -1                       # (duplicate back-pointers are re-attached after RebuildGraph, :395-401)
    rng = np.random.default_rng(7)
    g1 = np.concatenate([g0, -np.ones((files.n, 5), np.int32)], axis=1)        # stride > 2 x nbh
    g2 = g0.copy()                                                            # many edges into few nodes + holes
    g2[:, nbh // 2:nbh] = rng.integers(0, 50, size=(files.n, nbh - nbh // 2))
    g2[rng.random(g2.shape) < 0.05] = -1
    for g in (g0, g1, g2):
        a = r.rebuild_graph(g, nbh)
        b = reflib.oracle_rebuild_graph(g, nbh)
        assert np.array_equal(a, b), name
        assert not np.array_equal(a[:, :nbh], g[:, :nbh])   # it did something


@needs_ref
def test_iterator_known_answer_of_the_reference(oracle_lib):
    """Test/src/IterativeScanTest.cpp: line data, MaxCheck 5, query (0,...): two Next(5) calls return ids 0..9 in order
    with RelaxedMono set -- run on the reference itself and on the oracle."""
    folder = data_folder("algo_line_bkt")
    files = reflib.IndexFiles(folder)
    q = np.zeros(10, np.float32)
    r = reflib.RefIndex.load(folder)
    r.set_param("MaxCheck", 5)
    o = reflib.OracleIndex(files)
    o.max_check = 5
    for make in (r.iterator, o.iterator):
        it = make(q)
        got = []
        for _ in range(2):
            count, ids, dists, relaxed = it.next(5)
            assert count == 5 and relaxed
            got += ids.tolist()
        it.close()
        assert got == list(range(10))


@needs_ref
@pytest.mark.parametrize("name,mc", [("bkt_l2_20k_32", 8192), ("bkt_l2_20k_32", 64), ("bkt_cos_10k_128", 1024),
                                     ("bkt_l2_dups", 256), ("bkt_l2_3k_30", 512), ("bkt_i8_cos_6k_64", 512),
                                     ("bkt2_l2_6k_32", 256), ("bkt_i16_l2_4k_27", 300)])
def test_iterator_bit_exact_vs_reference(oracle_lib, name, mc):
    """ResultIterator::Next sequences (growing/shrinking batches, long scans, exhaustion) on the reference itself
    against ora_iter_*: count, ids, distances and RelaxedMono per call."""
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    qs = np.load(os.path.join(folder, "queries.npy"))[:10]
    r = reflib.RefIndex.load(folder)
    r.set_param("MaxCheck", mc)
    o = reflib.OracleIndex(files)
    o.max_check = mc
    for qi, q in enumerate(qs):
        ir, io = r.iterator(q), o.iterator(q)
        batches = [10, 10, 5, 7, 10, 3, 10, 1, 4] if qi % 2 == 0 else [32, 32, 16, 32, 8]
        if qi == 5:
            batches = [50] * 40
        if qi == 7:
            batches = [1000] * 6
        for b in batches:
            a, c = ir.next(b), io.next(b)
            assert a[0] == c[0], (name, qi, b)
            assert np.array_equal(a[1], c[1]), (name, qi, b)
            assert np.array_equal(a[2].view(np.int32), c[2].view(np.int32)), (name, qi, b)
            assert a[3] == c[3], (name, qi, b)
        ir.close()
        io.close()


@needs_ref
@pytest.mark.parametrize("name", ["bkt_l2_deleted_6k_32", "bkt_cos_deleted_5k_64"])
def test_tombstones_bit_exact_vs_reference(oracle_lib, name):
    """Row A9 (Labelset::Contains via CheckIfNotDeleted): indexes the reference built, deleted ~30 % of (including the
    true nearest neighbours of the first queries) with VectorIndex::DeleteIndex and saved with deletes.bin -- search,
    one refine step and iterator scans on the reference itself against the oracle with the same tombstone map."""
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    assert files.num_deleted > 1000 and int((files.deleted == 1).sum()) == files.num_deleted
    q = np.load(os.path.join(folder, "queries.npy"))
    r = reflib.RefIndex.load(folder)
    o = reflib.OracleIndex(files)
    for mc in (8192, 512, 64):
        r.set_param("MaxCheck", mc)
        o.max_check = mc
        ids_r, d_r, _ = r.search(q, 10, threads=4)
        ids_o, d_o, _ = o.search(q, 10, threads=4)
        assert np.array_equal(ids_r, ids_o), (name, mc)
        assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32)), (name, mc)
        assert not (files.deleted[ids_r[ids_r >= 0]] == 1).any()
    r.set_param("MaxCheckForRefineGraph", 512)
    o.max_check_refine = 512
    for a, b in zip(r.refine_nodes(100, 400, 48, files.degree, 1.0), o.refine_nodes(100, 400, 48, files.degree, 1.0)):
        assert np.array_equal(a.view(np.int32), b.view(np.int32)), name
    r.set_param("MaxCheck", 256)
    o.max_check = 256
    for qi in range(12):
        ir, io = r.iterator(q[qi]), o.iterator(q[qi])
        for b in [10, 10, 5, 10, 10, 10]:
            a, c = ir.next(b), io.next(b)
            assert a[0] == c[0] and np.array_equal(a[1], c[1]) and a[3] == c[3], (name, qi, b)
            assert np.array_equal(a[2].view(np.int32), c[2].view(np.int32)), (name, qi, b)
        ir.close()
        io.close()


@needs_ref
@pytest.mark.parametrize("name,k,mc", [("bkt_l2_10k_128", 2048, 8192), ("bkt_l2_10k_128", 10, 20000),
                                       ("bkt_i8_l2_5k_100", 2048, 8192), ("bkt_cos_3k_768", 1100, 8192)])
def test_large_k_and_budget_bit_exact_vs_reference(oracle_lib, name, k, mc):
    """K up to 2048 and MaxCheck beyond 16384 (m_Results capacity > 1024), plus a refine step with the reference's
    default first-pass CEF x CEFScale = 2000: the reference itself against the oracle."""
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    q = np.load(os.path.join(folder, "queries.npy"))[:60]
    r = reflib.RefIndex.load(folder)
    r.set_param("MaxCheck", mc)
    o = reflib.OracleIndex(files)
    o.max_check = mc
    if mc > 8192:
        r.set_param("MaxCheckForRefineGraph", mc)
        o.max_check_refine = mc
    ids_r, d_r, _ = r.search(q, k, threads=4)
    ids_o, d_o, _ = o.search(q, k, threads=4)
    assert np.array_equal(ids_r, ids_o)
    assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32))
    if mc <= 8192:
        r.set_param("MaxCheckForRefineGraph", 8192)
        o.max_check_refine = 8192
        for a, b in zip(r.refine_nodes(10, 100, 2000, files.degree, 1.0), o.refine_nodes(10, 100, 2000, files.degree, 1.0)):
            assert np.array_equal(a.view(np.int32), b.view(np.int32))


@needs_ref
@pytest.mark.parametrize("name", ["bkt_l2_deleted_6k_32", "bkt_cos_deleted_5k_64"])
def test_search_deleted_flag_vs_reference(oracle_lib, name):
    """p_searchDeleted = true (VectorIndex.h:41, dispatch flag BKTIndex.cpp:473): tombstoned vectors are eligible
    results again -- SearchIndex and GetIterator on the reference itself against the oracle without its tombstone map."""
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    q = np.load(os.path.join(folder, "queries.npy"))
    r = reflib.RefIndex.load(folder)
    r.set_param("MaxCheck", 1024)
    o = reflib.OracleIndex(files)
    o.max_check = 1024
    o.search_deleted = True
    ids_r, d_r = r.search_flag(q, 10, True, threads=4)
    ids_o, d_o, _ = o.search(q, 10, threads=4)
    assert np.array_equal(ids_r, ids_o)
    assert np.array_equal(d_r.view(np.int32), d_o.view(np.int32))
    assert (files.deleted[ids_r[ids_r >= 0]] == 1).sum() > 100      # deleted vectors do come back
    for qi in range(8):
        a, b = r.iterator(q[qi], True), o.iterator(q[qi])
        for bt in [10, 10, 10]:
            x, y = a.next(bt), b.next(bt)
            assert x[0] == y[0] and np.array_equal(x[1], y[1]) and x[3] == y[3]
            assert np.array_equal(x[2].view(np.int32), y[2].view(np.int32))
        a.close()
        b.close()


@needs_ref
@pytest.mark.parametrize("name,mc,k", [("bkt_l2_20k_32", 8192, 10), ("bkt_l2_20k_32", 128, 32), ("bkt_cos_10k_128", 1024, 64),
                                       ("bkt_l2_dups", 256, 16), ("bkt_l2_3k_30", 512, 8), ("bkt_i8_cos_6k_64", 512, 10),
                                       ("bkt_l2_deleted_6k_32", 512, 10), ("bkt_i16_l2_4k_27", 300, 5)])
def test_iterative_from_nearest_bit_exact_vs_reference(oracle_lib, name, mc, k):
    """VectorIndex::SearchIndexIterativeFromNeareast driven the way SPANN drives its head index (RentWorkSpace(k), one
    call per batch on a Reset() QueryResult, SearchIndexIterativeEnd) on the reference itself, against the oracle."""
    folder = data_folder(name)
    files = reflib.IndexFiles(folder)
    qs = np.load(os.path.join(folder, "queries.npy"))[:8]
    r = reflib.RefIndex.load(folder)
    r.set_param("MaxCheck", mc)
    o = reflib.OracleIndex(files)
    o.max_check = mc
    for qi, q in enumerate(qs):
        a, b = reflib.RefNearestScan(r, q, k), o.iterator(q)
        for rd in range(12 if qi != 3 else 300):
            x, y = a.next(), b.next_from_nearest(k)
            assert x[0] == y[0], (name, qi, rd)
            assert np.array_equal(x[1], y[1]), (name, qi, rd)
            assert np.array_equal(x[2].view(np.int32), y[2].view(np.int32)), (name, qi, rd)
            if not x[0]:
                break
        a.close()
        b.close()
