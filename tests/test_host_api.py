"""CPU tests of the host-side mirror of the reference API (options, data layer, chunk feed, metrics,
serialization).  The data fixtures are the reference's own known answers (tests/data/test_mm.py:15,62-68,
tests/data/test_stream.py:44-112, tests/util/test_aux.py)."""
import os

import numpy as np
import pytest
import scipy.sparse

import buffalo
from buffalo import MatrixMarket, MatrixMarketOptions, Stream, StreamOptions
from buffalo.algo.base import Algo, Serializable
from buffalo.algo.options import ALSOption, BPRMFOption, WARPOption
from buffalo.data.buffered_data import BufferedDataMatrix
from buffalo.evaluate import Evaluable
from buffalo.misc import aux


@pytest.fixture()
def mm_files(tmp_path):
    mm = tmp_path / "main.mtx"
    mm.write_text("%%MatrixMarket matrix coordinate integer general\n%\n%\n5 3 5\n1 1 1\n2 1 3\n3 3 1\n4 2 1\n5 2 2")
    uid = tmp_path / "uid"
    uid.write_text("lucas\ngony\njason\nlomego\nhan")
    iid = tmp_path / "iid"
    iid.write_text("apple\nmango\nbanana")
    return str(mm), str(uid), str(iid), str(tmp_path)


def test_option_attr_access():
    opt = aux.Option({"a": 1, "b": {"c": 2}})
    assert opt.a == 1 and opt.b.c == 2 and opt.missing is None
    opt.b.c = 7
    assert opt["b"]["c"] == 7
    assert ALSOption().get_default_option().optimizer == "manual_cg"
    assert WARPOption().get_default_option().max_trials == 500 and BPRMFOption().get_default_option().lr == 0.002


def test_option_validation():
    opt = ALSOption().get_default_option()
    assert ALSOption().is_valid_option(opt)
    opt.optimizer = "nope"
    with pytest.raises(RuntimeError):
        ALSOption().is_valid_option(opt)
    opt = ALSOption().get_default_option()
    opt.d = "20"
    with pytest.raises(RuntimeError):
        ALSOption().is_valid_option(opt)
    o = MatrixMarketOptions().get_default_option()
    assert MatrixMarketOptions().is_valid_option(o)
    o["type"] = 1
    with pytest.raises(RuntimeError):
        MatrixMarketOptions().is_valid_option(o)


@pytest.mark.parametrize("with_ids", [True, False])
def test_matrix_market_known_answer(mm_files, with_ids):
    mm_path, uid, iid, tmp = mm_files
    opt = MatrixMarketOptions().get_default_option()
    opt.input.main = mm_path
    opt.input.uid, opt.input.iid = (uid, iid) if with_ids else (None, None)
    opt.data.path = os.path.join(tmp, "mm.h5py")
    mm = MatrixMarket(opt)
    mm.create()
    assert sorted(mm.handle.keys()) == sorted(["vali", "idmap", "rowwise", "colwise"])
    h = mm.get_header()
    assert (h["num_nnz"], h["num_users"], h["num_items"]) == (5, 5, 3)
    data = list(mm.iterate())
    assert [int(k) for _, k, _ in data] == [0, 0, 2, 1, 1]
    assert (data[2][0], int(data[2][1]), float(data[2][2])) == (2, 2, 1.0)
    assert [int(k) for _, k, _ in mm.iterate(axis="colwise")] == [0, 1, 3, 4, 2]
    assert list(mm.get_group("rowwise")["indptr"][:]) == [1, 2, 3, 4, 5]       # exclusive END offsets
    if with_ids:
        assert [u for u, _, _ in mm.iterate(use_repr_name=True)][:2] == ["lucas", "gony"]
    # cache reuse keyed on the file (mm.py:241-245)
    opt.data.use_cache = True
    mm2 = MatrixMarket(opt)
    mm2.create()
    assert mm2.get_header()["num_nnz"] == 5


def test_matrix_market_array_inputs(tmp_path):
    for main in (scipy.sparse.random(32, 4, density=0.33, random_state=1), np.random.default_rng(0).random((32, 4))):
        opt = MatrixMarketOptions().get_default_option()
        opt.input.main = main
        opt.data.path = str(tmp_path / "a.h5py")
        mm = MatrixMarket(opt)
        mm.create()
        assert mm.get_header()["num_users"] == 32
    opt = MatrixMarketOptions().get_default_option()
    opt.input.main = [[10, 123], [1, 2]]
    with pytest.raises((AssertionError, RuntimeError)):
        MatrixMarketOptions().is_valid_option(opt)
    with pytest.raises((RuntimeError, TypeError)):
        MatrixMarket(opt).create()
    opt = MatrixMarketOptions().get_default_option()
    opt.input.main = np.array([[1, 2], [1, 2], [2, 1]])
    opt.input.uid, opt.input.iid = [1, 2.0, "3"], np.array(["1", "a"])
    opt.data.path = str(tmp_path / "b.h5py")
    MatrixMarket(opt).create()
    opt.input.uid = [1, 2.0]
    with pytest.raises(TypeError):
        MatrixMarket(opt).create()


def test_matrix_market_validation_split(tmp_path):
    rng = np.random.default_rng(0)
    M = scipy.sparse.random(300, 200, density=0.05, random_state=2, data_rvs=lambda n: rng.integers(1, 6, n))
    opt = MatrixMarketOptions().get_default_option()
    opt.input.main = M
    opt.data.validation.p, opt.data.validation.max_samples = 0.1, 50
    opt.data.path = str(tmp_path / "v.h5py")
    mm = MatrixMarket(opt)
    mm.create()
    assert mm.get_group("vali").attrs["num_samples"] == 50
    assert mm.get_header()["num_nnz"] == M.nnz - 50
    mm._prepare_validation_data()
    v = mm.vali_data
    for r, c in zip(v["row"][:10], v["col"][:10]):
        assert int(c) not in v["validation_seen"][int(r)] and int(c) in v["vali_gt"][int(r)]
    # both orientations describe the same training matrix
    rw = sorted((u, int(k)) for u, k, _ in mm.iterate())
    cw = sorted((int(k), i) for i, k, _ in mm.iterate(axis="colwise"))
    assert rw == cw


@pytest.mark.parametrize("text,uids,expect", [
    ("apple mango mango apple pie juice coke\npie\njuice coke grape", "kim\nlee\npark",
     ["apple", "mango", "mango", "apple", "pie", "juice", "pie", "juice", "coke"]),
    ("사과 망고 망고 사과 파이 주스 콜라\n파이\n주스 콜라 포도", "김씨\n이씨\n박씨",
     ["사과", "망고", "망고", "사과", "파이", "주스", "파이", "주스", "콜라"])])
def test_stream_known_answer(tmp_path, text, uids, expect):
    (tmp_path / "main").write_text(text)
    (tmp_path / "uid").write_text(uids)
    opt = StreamOptions().get_default_option()
    assert StreamOptions().is_valid_option(opt)
    opt.input.main, opt.input.uid = str(tmp_path / "main"), str(tmp_path / "uid")
    opt.data.path = str(tmp_path / "s.h5py")
    st = Stream(opt)
    st.create()
    assert sorted(st.handle.keys()) == sorted(["idmap", "rowwise", "colwise", "vali"])
    h = st.get_header()
    assert (h["num_nnz"], h["num_users"], h["num_items"]) == (9, 3, 6)      # newest-1 held out per line
    assert [k for _, k in st.iterate(use_repr_name=True)] == expect
    opt.data.internal_data_type = "matrix"
    st = Stream(opt)
    st.create()
    assert st.get_header()["num_nnz"] == 7
    assert [u for u, _, _ in st.iterate()] == [0, 0, 0, 0, 1, 2, 2]
    assert len(sorted(u for u, _, _ in st.iterate(axis="colwise", use_repr_name=True))) == 7


def test_prepro():
    from buffalo.data import prepro
    v = np.array([1.0, 3.0, 5.0], dtype=np.float32)
    assert np.array_equal(prepro.OneBased(aux.Option({}))(v.copy()), np.ones(3, np.float32))
    assert np.allclose(prepro.ImplicitALS(aux.Option({"epsilon": 0.5}))(v), np.log(1 + v / 0.5))
    mms = prepro.MinMaxScalar(aux.Option({"min": 1.0, "max": 2.0}))
    mms(v)
    db = {"val": v.copy()}
    mms.post(db)
    assert np.allclose(db["val"], [1.0, 1.5, 2.0])


def _mm_data(tmp_path, U=400, I=90, density=0.08, batch_mb=1024):
    M = scipy.sparse.random(U, I, density=density, random_state=3)
    opt = MatrixMarketOptions().get_default_option()
    opt.input.main = M
    opt.data.validation = aux.Option({})
    opt.data.batch_mb = batch_mb
    opt.data.path = str(tmp_path / "d.h5py")
    mm = MatrixMarket(opt)
    mm.create()
    return mm, M


def test_buffered_data_chunks_cover_every_row_once(tmp_path):
    mm, M = _mm_data(tmp_path)
    for limit in (None, 150, 40):
        buf = BufferedDataMatrix()
        buf.initialize(mm)
        for G, rows in (("rowwise", 400), ("colwise", 90)):
            if limit:
                buf.major[G]["limit"] = max(limit, int(np.max(np.diff(buf.major[G]["indptr"], prepend=0))) + 1)
            buf.set_group(G)
            covered, total = [], 0
            for sz in buf.fetch_batch():
                start_x, next_x, indptr, keys, vals = buf.get()
                beg = 0 if start_x == 0 else indptr[start_x - 1]
                assert indptr[next_x - 1] - beg == sz and sz <= max(buf.major[G]["limit"], 1) or limit is None
                assert np.array_equal(keys[:sz], mm.get_group(G)["key"][beg:beg + sz])
                covered.append((start_x, next_x))
                total += sz
            assert covered[0][0] == 0 and covered[-1][1] == rows
            assert all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
            assert total == M.nnz
            if limit and limit < M.nnz:
                assert len(covered) > 1


class _Mock(Algo, ALSOption, Evaluable, Serializable):
    def __init__(self, data=None):
        Algo.__init__(self)
        Serializable.__init__(self)
        self.opt = ALSOption().get_default_option()
        self.data = data
        import logging
        self.logger = logging.getLogger("mock")

    def normalize(self, group="item"):
        pass

    def _get_feature(self, index, group="item"):
        return self.Q[index]

    def _get_topk_recommendation(self, rows, topk, pool=None):
        return zip(rows, Algo._get_topk_recommendation(self, self.P[rows], self.Q, None, None, pool, topk, 1))

    def _get_most_similar_item(self, col, topk, pool):
        return Algo._get_most_similar_item(self, col, topk, self.Q, False, pool)

    def _get_scores(self, row, col):
        return (self.P[row] * self.Q[col]).sum(1)

    def _get_data(self):
        return super()._get_data() + [("opt", self.opt), ("Q", self.Q), ("P", self.P)]


def test_serialization_roundtrip_and_queries(tmp_path, mm_files):
    mm_path, uid, iid, tmp = mm_files
    opt = MatrixMarketOptions().get_default_option()
    opt.input.main, opt.input.uid, opt.input.iid = mm_path, uid, iid
    opt.data.path = os.path.join(tmp, "q.h5py")
    mm = MatrixMarket(opt)
    mm.create()
    m = _Mock(mm)
    m.initialize()
    m.P = np.eye(5, 3, dtype=np.float32) + 0.1
    m.Q = np.array([[1, 0, 0], [0.9, 0.1, 0], [0, 0, 1]], dtype=np.float32)
    assert m.topk_recommendation("lucas", topk=2) == ["apple", "mango"]
    assert set(m.topk_recommendation(["lucas", "gony"], topk=1).keys()) == {"lucas", "gony"}
    sims = m.most_similar("apple", topk=1)
    assert sims[0][0] == "mango"
    assert m.get_index("banana") == 2 and m.get_index("zzz") is None
    path = str(tmp_path / "model")
    m.save(path)
    m2 = _Mock(mm)
    m2.load(path)
    assert np.array_equal(m2.Q, m.Q) and m2.opt.d == 20 and m2._idmanager.itemids == ["apple", "mango", "banana"]
    m3 = _Mock(mm)
    m3.load(path, data_fields=["Q"])
    assert not hasattr(m3, "P")


def test_early_stopping_and_periodical():
    m = _Mock()
    m.initialize()
    m.opt.early_stopping_rounds = 2
    assert [m.early_stopping(x) for x in (1.0, 0.9, 0.95, 0.97)] == [False, False, False, True]   # base.py:213-224
    assert m.periodical(3, 2) and not m.periodical(3, 1) and m.periodical(0, 5)


def test_ranking_metrics_match_bruteforce(tmp_path):
    rng = np.random.default_rng(0)
    M = scipy.sparse.random(60, 40, density=0.2, random_state=5)
    opt = MatrixMarketOptions().get_default_option()
    opt.input.main = M
    opt.data.validation.p, opt.data.validation.max_samples = 0.2, 60
    opt.data.path = str(tmp_path / "e.h5py")
    np.random.seed(3)
    mm = MatrixMarket(opt)
    mm.create()
    m = _Mock(mm)
    m.initialize()
    m.opt.validation = aux.Option({"topk": 5})
    m.P = rng.normal(size=(60, 8)).astype(np.float32)
    m.Q = rng.normal(size=(40, 8)).astype(np.float32)
    res = m.get_validation_results()
    mm._prepare_validation_data()
    v = mm.vali_data
    acc = ndcg = 0.0
    n = 0
    for u in v["vali_rows"]:
        seen, gt = v["validation_seen"][int(u)], v["vali_gt"][int(u)]
        if not seen:
            continue
        order = [i for i in np.argsort(-(m.P[u] @ m.Q.T), kind="stable") if i not in seen][:5]
        acc += len(set(order) & gt) / len(gt)
        dcg = sum(1.0 / np.log2(r + 2) for r, i in enumerate(order) if i in gt)
        ndcg += dcg / sum(1.0 / np.log2(r + 2) for r in range(min(len(gt), 5)))
        n += 1
    assert abs(res["accuracy"] - acc / n) < 1e-9 and abs(res["ndcg"] - ndcg / n) < 1e-9
    assert 0.0 <= res["auc"] <= 1.0 and res["rmse"] > 0


def test_package_surface():
    # names the reference exports + the superset needed by examples/example_als.py (SURVEY.md Appendix A)
    for name in ["ALS", "BPRMF", "WARP", "Algo", "ALSOption", "BPRMFOption", "WARPOption", "AlgoOption", "MatrixMarket",
                 "MatrixMarketOptions", "Stream", "StreamOptions", "aux", "log", "set_log_level", "inited_CUALS",
                 "inited_CUBPR", "ParALS", "ParBPRMF"]:
        assert hasattr(buffalo, name), name
    from buffalo.algo import ALS, ALSOption  # noqa: F401
    from buffalo.data import MatrixMarketOptions as _M  # noqa: F401
    from buffalo.misc import aux as _a, log as _l  # noqa: F401
    from buffalo.parallel import ParALS  # noqa: F401
    with pytest.raises(NotImplementedError):
        buffalo.W2V()


def test_csr_from_triples_device_sort_matches_host_sort():
    """The torch ordering (run here on CPU tensors; on a GPU box the same code runs on `cuda`) reproduces the NumPy
    build of both orientations: sorted by (major, minor), duplicates kept in input order, end offsets."""
    from buffalo_b200.data.base import csr_from_triples
    rng = np.random.default_rng(3)
    n, U, I = 20000, 300, 170
    rows = rng.integers(0, U, n).astype(np.int64)
    cols = rng.integers(0, I, n).astype(np.int64)
    vals = rng.normal(size=n).astype(np.float32)
    rows[:50], cols[:50] = 7, 9          # duplicates: the stable sort keeps their input order
    for stable in (True, False):
        for major, minor, nm in ((rows, cols, U), (cols, rows, I)):
            a = csr_from_triples(major, minor, vals, nm, stable_sort=stable)
            b = csr_from_triples(major, minor, vals, nm, stable_sort=stable, device="cpu")
            assert all(np.array_equal(x, y) and x.dtype == y.dtype for x, y in zip(a, b))


def test_bench_zipf_generator_chunked_equals_unchunked():
    """bench.py's C5 generator (SURVEY 8d: Zipf items, de-duplicated per user) builds the matrix in ranges so that no sort
    exceeds 2^31 elements at full scale; the ranges must not change the result, the rowwise CSR must be sorted and
    duplicate-free, and the colwise CSR must be its exact transpose in (item, user) order."""
    import torch
    import bench
    ref = None
    for lim in (1 << 29, 4096, 777):
        w = dict(users=2500, items=300, nnz=50000, d=32, zipf=1.1, _chunk_limit=lim)
        wl = bench.make_workload_zipf(w, torch.device("cpu"))
        U, I, nnz = wl["U"], wl["I"], wl["nnz"]
        ri, rk = wl["r_indptr"].numpy(), wl["r_keys"].numpy()
        ci, ck = wl["c_indptr"].numpy(), wl["c_keys"].numpy()
        assert ri[-1] == nnz == ci[-1] and len(rk) == nnz == len(ck)
        rows = np.repeat(np.arange(U), np.diff(np.concatenate([[0], ri])))
        assert (np.diff(rows.astype(np.int64) * I + rk) > 0).all()           # sorted, no duplicates
        order = np.lexsort((rows, rk))
        assert (ck == rows[order]).all()
        assert (np.diff(np.concatenate([[0], ci])) == np.bincount(rk, minlength=I)).all()
        deg_items = np.bincount(rk, minlength=I)
        assert deg_items[:10].mean() > 20 * max(1.0, deg_items[I // 2:].mean())   # a Zipf head
        if ref is None:
            ref = (ri.copy(), rk.copy(), ck.copy())
        else:
            assert (ref[0] == ri).all() and (ref[1] == rk).all() and (ref[2] == ck).all()


def test_bench_dump_outputs_is_a_fixed_bounded_sample(tmp_path):
    """bench.py --dump-outputs: a matrix larger than the per-array budget is cut to the same sorted row sample on every
    run, a small one is written whole, always as float32, and four arrays stay within 64 MB."""
    import torch
    import bench
    P = torch.arange(300000 * 16, dtype=torch.float32).reshape(300000, 16)     # row r holds 16 r .. 16 r + 15
    Qb = torch.arange(50, dtype=torch.float64).reshape(50, 1)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"P": P, "Qb": Qb})
    a, b = np.load(tmp_path / "a" / "P.npy"), np.load(tmp_path / "b" / "P.npy")
    assert a.dtype == np.float32 and a.shape[1] == 16 and 0 < a.shape[0] < 300000
    assert 4 * a.nbytes <= 64 << 20 and np.array_equal(a, b)
    rows = a[:, 0] / 16
    assert (np.diff(rows) > 0).all() and np.array_equal(a, P.numpy()[rows.astype(np.int64)])
    qb = np.load(tmp_path / "a" / "Qb.npy")
    assert qb.dtype == np.float32 and np.array_equal(qb, Qb.numpy())
