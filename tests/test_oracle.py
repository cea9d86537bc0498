"""CPU tests of the oracle (oracle/lux_oracle.c) against fixtures that do not come from the oracle itself:
the .lux byte image the reference's own converter produces, answers worked out by hand from the cited reference
lines, and an independent numpy restatement of the same semantics."""
import os

import numpy as np
import pytest

import oracle as O
from graphs import ALL_SMALL, hand5, rmat, star, symmetrize

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ---- independent numpy restatements (no shared code with the C oracle) -----------------------------------------
def np_edges(row_end, src):
    nv = len(row_end)
    starts = np.concatenate([[0], row_end[:-1]]).astype(np.int64)
    dst = np.repeat(np.arange(nv, dtype=np.int64), (row_end.astype(np.int64) - starts))
    return src.astype(np.int64), dst


def np_pagerank(row_end, src, iters):
    """pagerank_gpu.cu:255-259 (init), :86-100 + :144 (iteration); per-vertex sum in fp64 rounded once to f32."""
    nv = len(row_end)
    s, d = np_edges(row_end, src)
    deg = np.bincount(s, minlength=nv).astype(np.uint32)
    rank = np.float32(1.0) / np.float32(nv)
    x = np.where(deg == 0, rank, rank / np.maximum(deg, 1).astype(np.float32)).astype(np.float32)
    init = (np.float32(1) - np.float32(0.15)) / np.float32(nv)
    for _ in range(iters):
        acc = np.bincount(d, weights=x[s].astype(np.float64), minlength=nv).astype(np.float32)
        # fmaf(alpha, acc, init): emulate a single rounding with float64 (exact product, one rounding to f32)
        y = (np.float64(np.float32(0.15)) * acc.astype(np.float64) + np.float64(init)).astype(np.float32)
        x = np.where(deg == 0, y, y / np.maximum(deg, 1).astype(np.float32)).astype(np.float32)
    return x


def np_cc(row_end, src):
    """fixed point of label[v] = max(label[v], label[u]) over edges u->v (components_gpu.cu:112-122)."""
    nv = len(row_end)
    s, d = np_edges(row_end, src)
    lab = np.arange(nv, dtype=np.int64)
    while True:
        new = lab.copy()
        np.maximum.at(new, d, lab[s])
        if np.array_equal(new, lab):
            return lab.astype(np.uint32)
        lab = new


def np_bfs(row_end, src, start):
    """hop distance along directed edges, INF = nv (sssp_gpu.cu:733-744, :122)."""
    nv = len(row_end)
    s, d = np_edges(row_end, src)
    dist = np.full(nv, nv, dtype=np.int64)
    dist[start] = 0
    while True:
        new = dist.copy()
        np.minimum.at(new, d, dist[s] + 1)
        new = np.minimum(new, nv)
        if np.array_equal(new, dist):
            return dist.astype(np.uint32)
        dist = new


# ---- format / converter ----------------------------------------------------------------------------------------
def test_lux_bytes_match_reference_converter(tmp_path):
    """tests/golden/hand5.lux.hex is the byte image tools/converter.cc (g++ -O2, oracle/build_ref.py) writes for the
    edges {0->1,1->2,2->0,3->0,0->2}: u32 nv | u64 ne | u64 row_end[nv] | u32 src[ne] | u32 out_degree[nv].
    The converter's std::sort by dst is unstable, so inside one destination's block the source order is arbitrary
    (here dst 2 holds [1,0]); our canonical CSC sorts it.  Everything else must match byte for byte."""
    row_end, src = hand5()
    assert row_end.tolist() == [2, 3, 5, 5] and src.tolist() == [2, 3, 0, 0, 1]
    path = str(tmp_path / "hand5.lux")
    O.lux_write(path, row_end, src)
    want = bytes.fromhex(open(os.path.join(GOLDEN, "hand5.lux.hex")).read().strip())
    got = open(path, "rb").read()
    hdr = 12 + 8 * 4
    assert len(got) == len(want) and got[:hdr] == want[:hdr] and got[hdr + 20:] == want[hdr + 20:]
    ref_src = np.frombuffer(want[hdr:hdr + 20], np.uint32)
    lo = 0
    for v in range(4):
        hi = int(row_end[v])
        assert sorted(ref_src[lo:hi].tolist()) == src[lo:hi].tolist()
        lo = hi
    # the reference's own bytes load through the oracle's reader and give the same PageRank
    ref_path = str(tmp_path / "ref.lux")
    open(ref_path, "wb").write(want)
    re2, src2 = O.lux_read(ref_path)
    assert np.array_equal(re2, row_end)
    assert np.allclose(O.pagerank(re2, src2, 3), O.pagerank(row_end, src, 3), rtol=1e-7)


def test_lux_weighted_roundtrip(tmp_path):
    row_end, src, w = O.gen_bipartite_csc(50, 7, 300, 5)
    path = str(tmp_path / "w.lux")
    O.lux_write(path, row_end, src, w)
    re2, src2, w2 = O.lux_read(path, weighted=True)
    assert np.array_equal(re2, row_end) and np.array_equal(src2, src) and np.array_equal(w2, w)
    assert w.min() >= 1 and w.max() <= 5


# ---- partitioner (pull_model.inl:108-131) ------------------------------------------------------------------------
def py_partition(row_end, ne, P):
    cap = (ne + P - 1) // P
    bounds, cnt, left = [], 0, 0
    prev = 0
    for v, e in enumerate(row_end.tolist()):
        cnt += e - prev
        prev = e
        if cnt > cap:
            bounds.append((left, v))
            cnt, left = 0, v + 1
    if cnt > 0:
        bounds.append((left, len(row_end) - 1))
    return bounds


@pytest.mark.parametrize("P", [1, 2, 3, 4, 8])
def test_partitioner_matches_line_by_line_python(P):
    row_end, src = rmat(12)
    cnt, rl, rr, cl, fl, fr = O.partition(row_end, len(src), P)
    want = py_partition(row_end, len(src), P)
    assert cnt == len(want)
    for p, (a, b) in enumerate(want[:P]):
        assert (rl[p], rr[p]) == (a, b)
        assert cl[p] == (0 if a == 0 else row_end[a - 1])
    # frontier slots: 8-byte header + ((R-L)/16 + 100) ids (push_model.inl:393-397), laid out back to back
    off = 0
    for p, (a, b) in enumerate(want[:P]):
        assert fl[p] == off
        off += 8 + 4 * ((b - a) // 16 + 100)
        assert fr[p] == off - 1


def test_partitioner_hand_case():
    # in-degrees [100,1,1,1], P=4: cap = 26 -> vertex 0 alone closes partition 0, the rest never exceed cap:
    # the reference would assert (#parts = 2 != 4), SURVEY §8 a2.
    row_end = np.array([100, 101, 102, 103], np.uint64)
    cnt, rl, rr, cl, _, _ = O.partition(row_end, 103, 4)
    assert cnt == 2 and (rl[0], rr[0]) == (0, 0) and (rl[1], rr[1]) == (1, 3) and cl[1] == 100


# ---- PageRank ------------------------------------------------------------------------------------------------
def test_pagerank_hand5_by_hand():
    """One iteration worked by hand: nv=4, out-degrees [2,1,1,1]; x0 = [1/8,1/4,1/4,1/4];
    s = [x2+x3, x0, x0+x1, 0] = [1/2,1/8,3/8,0]; y = .85/4 + .15*s; x1 = y/deg."""
    row_end, src = hand5()
    x1 = O.pagerank(row_end, src, 1)
    init = np.float32(0.85) / np.float32(4)
    s = np.array([0.5, 0.125, 0.375, 0.0], np.float32)
    y = (np.float32(0.15) * s + init).astype(np.float32)
    want = y / np.array([2, 1, 1, 1], np.float32)
    assert np.allclose(x1, want, rtol=2e-7, atol=0)


@pytest.mark.parametrize("name", sorted(ALL_SMALL))
def test_pagerank_matches_numpy_restatement(name):
    row_end, src = ALL_SMALL[name]()
    for ni in (1, 4):
        a, b = O.pagerank(row_end, src, ni), np_pagerank(row_end, src, ni)
        assert np.allclose(a, b, rtol=3e-7, atol=0)


def test_pagerank_range_calls_compose():
    row_end, src = rmat(11)
    nv = len(row_end)
    deg = O.out_degree(nv, src)
    x0 = O.pagerank_init(deg)
    full = O.pagerank_iter(row_end, src, deg, x0)
    cnt, rl, rr, _, _, _ = O.partition(row_end, len(src), 4)
    assert cnt == 4
    out = np.zeros(nv, np.float32)
    for p in range(4):
        O.pagerank_iter(row_end, src, deg, x0, int(rl[p]), int(rr[p]), out=out)
    assert np.array_equal(out, full)


# ---- CC / SSSP -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(ALL_SMALL))
def test_cc_fixed_point_and_invariant(name):
    row_end, src = ALL_SMALL[name]()
    r = O.label_run(O.APP_CC, row_end, src)
    assert np.array_equal(r["labels"], np_cc(row_end, src))
    assert O.label_check(O.APP_CC, row_end, src, r["labels"]) == 0
    assert r["active"][-1] == 0 and (len(r["active"]) == 1 or r["active"][-2] > 0)


@pytest.mark.parametrize("name", sorted(ALL_SMALL))
def test_sssp_is_bfs_depth(name):
    row_end, src = ALL_SMALL[name]()
    for start in (0, len(row_end) // 2):
        r = O.label_run(O.APP_SSSP, row_end, src, start=start)
        assert np.array_equal(r["labels"], np_bfs(row_end, src, start))
        assert O.label_check(O.APP_SSSP, row_end, src, r["labels"]) == 0


def test_cc_on_symmetric_graph_is_max_id_of_component():
    row_end, src = symmetrize(*rmat(10, ef=2))
    lab = O.label_run(O.APP_CC, row_end, src)["labels"]
    s, d = np_edges(row_end, src)
    assert np.array_equal(lab[s], lab[d])  # constant on every edge => constant per component
    for c in np.unique(lab):
        assert c == np.nonzero(lab == c)[0].max()


@pytest.mark.parametrize("P", [1, 2, 4])
def test_labels_do_not_depend_on_partition_count(P):
    row_end, src = rmat(12)
    base = O.label_run(O.APP_SSSP, row_end, src, P=1, start=3)
    r = O.label_run(O.APP_SSSP, row_end, src, P=P, start=3)
    assert np.array_equal(r["labels"], base["labels"])
    assert np.array_equal(r["active"], base["active"]) and np.array_equal(r["pull"], base["pull"])


def test_direction_rule_and_frontier_types():
    """pull iff #active > nv/16 (components_gpu.cu:414); CC starts all-active dense (:733-737)."""
    row_end, src = star()
    nv = len(row_end)
    r = O.label_run(O.APP_CC, row_end, src, P=1)
    assert r["pull"][0] == 1  # all nv vertices active
    prev_active = [nv] + r["active"].tolist()[:-1]
    for a, p in zip(prev_active, r["pull"].tolist()):
        assert p == (1 if a > nv // 16 else 0)
    assert set(np.unique(r["ftype"])) <= {O.DENSE_BITMAP, O.SPARSE_QUEUE}


def test_push_csr_is_transpose_of_partition():
    row_end, src = rmat(10)
    cnt, rl, rr, _, _, _ = O.partition(row_end, len(src), 2)
    s, d = np_edges(row_end, src)
    for p in range(2):
        out_end, out_dst = O.build_push_csr(row_end, src, int(rl[p]), int(rr[p]))
        sel = (d >= rl[p]) & (d <= rr[p])
        want = sorted(zip(s[sel].tolist(), d[sel].tolist()))
        starts = np.concatenate([[0], out_end[:-1]]).astype(np.int64)
        got_src = np.repeat(np.arange(len(row_end)), out_end.astype(np.int64) - starts)
        assert sorted(zip(got_src.tolist(), out_dst.tolist())) == want


# ---- collaborative filtering ---------------------------------------------------------------------------------
def test_colfilter_one_vertex_by_hand():
    """Single edge u->v with weight 3: x = sqrt(1/20) everywhere; dot = 20 * (1/20) = 1; err = 2;
    acc = 2 * x; x_v' = x + GAMMA * (2x - LAMBDA x) (colfilter_gpu.cu:83-100)."""
    row_end = np.array([0, 1], np.uint64)
    src = np.array([0], np.uint32)
    w = np.array([3], np.int32)
    x1 = O.colfilter(row_end, src, w, 1)
    x = np.float32(np.sqrt(np.float32(1.0 / 20)))
    want_v = x + np.float32(3.5e-7) * (np.float32(2) * x - np.float32(1e-3) * x)
    want_u = x + np.float32(3.5e-7) * (np.float32(0) - np.float32(1e-3) * x)
    assert np.allclose(x1[1], want_v, rtol=1e-6) and np.allclose(x1[0], want_u, rtol=1e-6)


def test_colfilter_matches_numpy_restatement():
    row_end, src, w = O.gen_bipartite_csc(60, 9, 700, 5)
    nv = len(row_end)
    s, d = np_edges(row_end, src)
    x = np.full((nv, 20), np.float32(np.sqrt(np.float32(1 / 20))), np.float32)
    for _ in range(3):
        dot = np.einsum("ek,ek->e", x[s].astype(np.float64), x[d].astype(np.float64))
        err = w.astype(np.float64) - dot
        acc = np.zeros((nv, 20))
        np.add.at(acc, d, err[:, None] * x[s].astype(np.float64))
        x = (x + np.float32(3.5e-7) * (acc.astype(np.float32) - np.float32(1e-3) * x)).astype(np.float32)
    got = O.colfilter(row_end, src, w, 3)
    assert np.allclose(got, x, rtol=1e-6, atol=0)


def test_colfilter_step_is_minus_gamma_times_the_gradient_of_the_regularised_squared_error():
    """Mathematical pin of the col_filter oracle (the reference kernel is racy and mis-indexed, SURVEY §2.2, so it
    cannot be pinned by execution).  What the reference INTENDS (colfilter_gpu.cu:83-100 with LAMBDA / GAMMA of
    col_filter/app.h:26-27) is one Jacobi gradient-descent step on
        L_v(x_v) = 1/2 * sum_{(u,w) in in(v)} (w - <x_u, x_v>)^2 + 1/2 * LAMBDA * |x_v|^2        (x_u held fixed)
    i.e. x_v' - x_v = -GAMMA * grad L_v(x_v).  The gradient is taken here by CENTRAL FINITE DIFFERENCES of L_v in
    float64 — no line of this test restates the update formula."""
    lam, gamma = 1e-3, 3.5e-7
    row_end, src, w = O.gen_bipartite_csc(300, 40, 20000, 5)
    nv = len(row_end)
    rng = np.random.default_rng(3)
    x = (0.1 + 0.4 * rng.random((nv, 20))).astype(np.float32)  # not the uniform start: every factor gets its own slope
    x_new = O.cf_iter(row_end, src, w, x)
    starts = np.concatenate([[0], row_end[:-1]]).astype(np.int64)
    x64 = x.astype(np.float64)

    def loss(v, xv):
        b, e = starts[v], int(row_end[v])
        err = w[b:e].astype(np.float64) - x64[src[b:e]] @ xv
        return 0.5 * np.dot(err, err) + 0.5 * lam * np.dot(xv, xv)

    checked = 0
    for v in list(range(0, 300, 37)) + list(range(300, 340, 5)):  # users (degree ~67) and items (degree ~500)
        if int(row_end[v]) - starts[v] == 0:
            continue
        grad = np.zeros(20)
        for k in range(20):
            h = 1e-5
            xp, xm = x64[v].copy(), x64[v].copy()
            xp[k] += h
            xm[k] -= h
            grad[k] = (loss(v, xp) - loss(v, xm)) / (2 * h)
        step = (x_new[v].astype(np.float64) - x64[v]) / (-gamma)
        # x' - x is a difference of f32 numbers near 0.3: resolution ulp(0.5)/gamma ~ 0.1 in gradient units
        assert np.allclose(step, grad, rtol=2e-3, atol=0.1), (v, np.abs(step - grad).max(), np.abs(grad).max())
        assert np.abs(grad).max() > 5  # the comparison is not vacuous (atol is < 2 % of it)
        checked += 1
    assert checked >= 10


# ---- generators ----------------------------------------------------------------------------------------------
def test_rmat_generator_properties():
    scale, nv = 12, 3000
    ne = 16 * nv
    row_end, src = O.gen_rmat_csc(scale, nv, ne, 3)
    assert row_end[-1] == ne and src.max() < nv and np.all(np.diff(row_end.astype(np.int64)) >= 0)
    s, d = np_edges(row_end, src)
    key = d * (1 << 32) + s
    assert np.all(np.diff(key) >= 0)  # canonical (dst, src) order, duplicates kept
    # edge multiset equals the per-edge generator
    want = sorted((O.rmat_edge(3, i, scale, nv)[1] << 32) | O.rmat_edge(3, i, scale, nv)[0] for i in range(0, 2000))
    assert set(want) <= set(key.tolist())
    # skew: P(src bit = 0) = a + b = 0.76 at the top level (only approximately once endpoints >= nv are rejected)
    row_end, src = O.gen_rmat_csc(12, 4096, 65536, 27)
    assert abs((src < 2048).mean() - 0.76) < 0.01


def test_golden_vectors():
    """Regression pin: oracle outputs frozen in tests/golden/oracle_rmat10.npz (made by tests/golden/make_golden.py)."""
    g = np.load(os.path.join(GOLDEN, "oracle_rmat10.npz"))
    row_end, src = O.gen_rmat_csc(10, 1000, 16000, 27)
    assert np.array_equal(row_end, g["row_end"]) and np.array_equal(src, g["src"])
    assert np.array_equal(O.pagerank(row_end, src, 10), g["pagerank10"])
    assert np.array_equal(O.label_run(O.APP_CC, row_end, src)["labels"], g["cc"])
    assert np.array_equal(O.label_run(O.APP_SSSP, row_end, src, start=0)["labels"], g["sssp0"])
    assert np.array_equal(O.label_run(O.APP_SSSP, row_end, src, start=0)["active"], g["sssp0_active"])


# ---- the real reference converter: tests/golden/ref_converter.npz holds edge lists and the bytes tools/converter.cc
# (built as is by oracle/build_ref.py) wrote for them (tests/golden/make_golden.py) ----------------------------------
def test_oracle_lux_writer_matches_reference_converter_binary(tmp_path):
    """tools/converter.cc run on an edge list must produce exactly what oracle.lux_write produces (the converter's
    std::sort by dst is unstable, so compare per-destination source MULTISETS plus every other byte)."""
    g = np.load(os.path.join(GOLDEN, "ref_converter.npz"))
    nv, ne = 300, 4000
    s, d = g["n300_src"], g["n300_dst"]
    assert len(s) == len(d) == ne
    row_end, src = O.edges_to_csc(nv, s, d)
    mine = str(tmp_path / "mine.lux")
    O.lux_write(mine, row_end, src)
    a, b = g["n300_lux"].tobytes(), open(mine, "rb").read()
    assert len(a) == len(b)
    hdr = 12 + 8 * nv
    assert a[:hdr] == b[:hdr]                      # header + row_end
    assert a[hdr + 4 * ne:] == b[hdr + 4 * ne:]    # out-degree trailer
    ra = np.frombuffer(a[hdr:hdr + 4 * ne], np.uint32)
    lo = 0
    for v in range(nv):
        hi = int(row_end[v])
        assert sorted(ra[lo:hi].tolist()) == src[lo:hi].tolist()
        lo = hi


# ---- pinned by REFERENCE EXECUTION: outputs of the reference's own CUDA kernels, replayed on a B200 --------------
def test_oracle_matches_reference_replay():
    """tests/golden/ref_replay_golden.npz holds what the reference's OWN task bodies and kernels (pagerank_gpu.cu,
    components_gpu.cu, sssp_gpu.cu compiled unmodified behind oracle/ref_replay/shim) produced on a B200
    (scripts/make_ref_golden.py).  CC / SSSP labels: bit-exact.  Per-iteration active counts: equal, except where a
    sparse frontier overflows and is promoted to a bitmap — there the reference re-counts into a header that already
    holds the sparse count (defect B5, components_gpu.cu:482-490) and reports exactly twice the true number.
    PageRank: the reference sums with float atomicAdd in arbitrary order (pagerank_gpu.cu:90), so it matches the
    fp64-accumulating oracle to ~1e-6 on low-degree graphs and ~5e-5 on a 10^4-in-degree hub (SURVEY Appendix E)."""
    g = np.load(os.path.join(GOLDEN, "ref_replay_golden.npz"))
    names = sorted({k[: -len("_row_end")] for k in g.files if k.endswith("_row_end")})
    assert len(names) >= 5
    for name in names:
        row_end, src = g[name + "_row_end"], g[name + "_src"]
        pr = O.pagerank(row_end, src, 10)
        rel = (np.abs(pr - g[name + "_pagerank10"]) / np.abs(pr)).max()
        assert rel <= (1e-4 if name == "star" else 1.5e-6), (name, rel)
        for oapp, key in ((O.APP_CC, "_cc"), (O.APP_SSSP, "_sssp0")):
            r = O.label_run(oapp, row_end, src, start=0)
            assert np.array_equal(r["labels"], g[name + key]), (name, key)
            ref_active = g[name + key + "_active"].astype(np.int64)
            assert len(ref_active) == r["iters"]
            for it, (a_ref, a_or) in enumerate(zip(ref_active, r["active"].astype(np.int64))):
                promoted = r["pull"][it] == 0 and r["ftype"][it, 0] == O.DENSE_BITMAP and (
                    it == 0 and oapp == O.APP_SSSP or it > 0 and r["ftype"][it - 1, 0] == O.SPARSE_QUEUE)
                assert a_ref == a_or or (promoted and a_ref == 2 * a_or), (name, key, it, a_ref, a_or)
