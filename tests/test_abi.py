"""No-GPU checks of the drop-in boundary: libluxb.so builds/loads, exports every symbol include/lux_b200.h declares,
the host-side partitioner (pure host code behind the C ABI) matches the oracle, and the product refuses to run
without a GPU instead of falling back to anything."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import lux_b200 as L
import oracle as O
from graphs import rmat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = L.load_library()
    names = L.declared_symbols()
    assert len(names) >= 24
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    assert b"sm_100a" in lib.luxb_version()


def test_header_cites_the_reference_interface():
    text = open(os.path.join(ROOT, "include", "lux_b200.h")).read()
    for cite in ("pull_model.inl", "push_model.inl", "pagerank_gpu.cu", "components_gpu.cu", "core/graph.h"):
        assert cite in text
    assert "torch" not in text.lower()  # plain pointers and sizes only


def test_product_sources_never_touch_the_oracle():
    """The product must not import, include, link or dlopen anything under oracle/ (comments may mention it)."""
    bad = re.compile(r"^\s*(import\s+oracle|from\s+oracle|#\s*include\s*[\"<][^\">]*oracle)|liblux_oracle|lo_[a-z_]+\(")
    for d in ("lux_b200", "lux_b200/csrc", "include"):
        for f in os.listdir(os.path.join(ROOT, d)):
            p = os.path.join(ROOT, d, f)
            if os.path.isfile(p) and f.endswith((".py", ".cu", ".cuh", ".h")):
                for ln, line in enumerate(open(p, errors="ignore"), 1):
                    if line.lstrip().startswith(("//", "*", "/*", "#  ", '"""')):
                        continue
                    assert not bad.search(line), "%s:%d %s" % (p, ln, line.strip())


@pytest.mark.parametrize("P", [1, 2, 4, 8])
def test_host_partitioner_matches_oracle(P):
    row_end, src = rmat(12)
    cnt, rl, rr, cl = L.partition_csc(row_end, len(src), P)
    ocnt, orl, orr, ocl, _, _ = O.partition(row_end, len(src), P)
    assert cnt == ocnt
    assert np.array_equal(rl[:cnt], orl[:cnt]) and np.array_equal(rr[:cnt], orr[:cnt]) and np.array_equal(cl[:cnt], ocl[:cnt])


def test_partitioner_keeps_trailing_zero_indegree_vertices():
    # reference would assert (count 1 != P 2); we keep vertex 3 in an edge-free last partition
    row_end = np.array([2, 3, 5, 5], np.uint64)
    cnt, rl, rr, cl = L.partition_csc(row_end, 5, 2)
    assert cnt == 1 and (rl[0], rr[0]) == (0, 2) and (rl[1], rr[1]) == (3, 3) and cl[1] == 5


def test_bad_arguments_return_errors_not_exits():
    lib = L.load_library()
    with pytest.raises(L.LuxError):
        L.partition_csc(np.array([3, 2], np.uint64), 2, 1)  # decreasing row_end (pull_model.inl:100-101)
    assert lib.luxb_graph_info(None, None, None, None) < 0
    assert b"NULL" in lib.luxb_last_error()


def test_no_cpu_fallback_without_gpu(gpu_count):
    if gpu_count:
        pytest.skip("GPU present")
    with pytest.raises(L.LuxError, match="no CPU fallback"):
        L.pagerank(np.array([1, 2], np.uint64), np.array([1, 0], np.uint32), num_iter=1)


# ---- .lux writer / edge-list converter of the product (host-only entry points: run without a GPU) -----------------
def test_write_lux_bytes_equal_the_oracle_writer(tmp_path):
    import oracle as O
    import lux_b200 as L
    row_end, src = O.gen_rmat_csc(9, 500, 6000, 4)
    a, b = str(tmp_path / "a.lux"), str(tmp_path / "b.lux")
    L.write_lux(a, row_end, src)
    O.lux_write(b, row_end, src)
    assert open(a, "rb").read() == open(b, "rb").read()
    row_end, src, w = O.gen_bipartite_csc(40, 9, 300, 5)
    L.write_lux(a, row_end, src, w)
    O.lux_write(b, row_end, src, w)
    assert open(a, "rb").read() == open(b, "rb").read()
    # the reference converter's own bytes for {0->1, 1->2, 2->0, 3->0, 0->2} (tests/golden/hand5.lux.hex): identical except
    # for the order inside destination 2's block (its std::sort by dst is unstable: [1, 0]; ours is canonical: [0, 1])
    re5, src5 = O.edges_to_csc(4, [0, 1, 2, 3, 0], [1, 2, 0, 0, 2])
    L.write_lux(a, re5, src5)
    golden = bytes.fromhex(open(os.path.join(ROOT, "tests", "golden", "hand5.lux.hex")).read().strip())
    got = open(a, "rb").read()
    hdr = 12 + 8 * 4
    assert len(got) == len(golden) and got[:hdr] == golden[:hdr] and got[hdr + 20:] == golden[hdr + 20:]
    assert sorted(np.frombuffer(golden[hdr + 12:hdr + 20], np.uint32).tolist()) == np.frombuffer(got[hdr + 12:hdr + 20], np.uint32).tolist()


def test_convert_edgelist_matches_reference_converter(tmp_path):
    """luxb_convert_edgelist vs tools/converter.cc built as is (its output for this edge list is stored in
    tests/golden/ref_converter.npz): header, offsets and out-degree trailer byte-identical, per-destination source
    multisets equal (the reference's std::sort by dst is unstable), and byte-identical to the oracle's canonical writer."""
    import oracle as O
    import lux_b200 as L
    golden = np.load(os.path.join(ROOT, "tests", "golden", "ref_converter.npz"))
    nv, ne = 257, 5000
    s, d = golden["n257_src"], golden["n257_dst"]
    assert len(s) == len(d) == ne
    txt = tmp_path / "edges.txt"
    txt.write_text("".join("%d %d\n" % (a, b) for a, b in zip(s, d)))
    mine = str(tmp_path / "mine.lux")
    L.convert_edgelist(str(txt), mine, nv, ne)
    row_end, src = O.edges_to_csc(nv, s, d)
    canon = str(tmp_path / "canon.lux")
    O.lux_write(canon, row_end, src)
    a = open(mine, "rb").read()
    assert a == open(canon, "rb").read()
    b = golden["n257_lux"].tobytes()
    hdr = 12 + 8 * nv
    assert len(a) == len(b) and a[:hdr] == b[:hdr] and a[hdr + 4 * ne:] == b[hdr + 4 * ne:]
    ra, rb = np.frombuffer(a[hdr:hdr + 4 * ne], np.uint32), np.frombuffer(b[hdr:hdr + 4 * ne], np.uint32)
    lo = 0
    for v in range(nv):
        hi = int(row_end[v])
        assert sorted(rb[lo:hi].tolist()) == ra[lo:hi].tolist()
        lo = hi
    with pytest.raises(L.LuxError):
        L.convert_edgelist(str(txt), mine, nv, ne + 1)      # fewer edges in the file than announced
    with pytest.raises(L.LuxError):
        L.convert_edgelist(str(txt), mine, 10, ne)          # endpoint out of range: an error code, not an assert
