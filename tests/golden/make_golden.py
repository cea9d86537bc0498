"""Regenerates the committed golden fixtures.  Run from the repo root:  python tests/golden/make_golden.py
hand5.lux.hex is NOT produced by the oracle: it is the byte image that the reference's tools/converter.cc writes for
edges {0->1,1->2,2->0,3->0,0->2}: python oracle/build_ref.py && printf '0 1\\n1 2\\n2 0\\n3 0\\n0 2\\n' > e5.txt &&
oracle/_ref/converter -nv 4 -ne 5 -input e5.txt -output e5.lux  (hex dump of e5.lux).
ref_converter.npz is NOT produced by the oracle either: random edge lists and the .lux bytes tools/converter.cc writes for
them (oracle/_ref/converter, built by python oracle/build_ref.py); it is rewritten only when that binary exists."""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle as O  # noqa: E402

row_end, src = O.gen_rmat_csc(10, 1000, 16000, 27)
ss = O.label_run(O.APP_SSSP, row_end, src, start=0)
np.savez_compressed(os.path.join(HERE, "oracle_rmat10.npz"), row_end=row_end, src=src,
                    pagerank10=O.pagerank(row_end, src, 10), cc=O.label_run(O.APP_CC, row_end, src)["labels"],
                    sssp0=ss["labels"], sssp0_active=ss["active"])
print("wrote oracle_rmat10.npz")

# (rng seed, nv, ne) of each edge list; the key prefix is n<nv>
CONVERTER_CASES = [(1, 300, 4000), (2, 257, 5000)]
converter = os.path.join(HERE, "..", "..", "oracle", "_ref", "converter")
if os.path.exists(converter):
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for seed, nv, ne in CONVERTER_CASES:
            rng = np.random.default_rng(seed)
            s = rng.integers(0, nv, ne).astype(np.uint32)
            d = rng.integers(0, nv, ne).astype(np.uint32)
            txt, lux = os.path.join(tmp, "edges.txt"), os.path.join(tmp, "ref.lux")
            with open(txt, "w") as f:
                f.write("".join("%d %d\n" % (a, b) for a, b in zip(s, d)))
            subprocess.check_call([converter, "-nv", str(nv), "-ne", str(ne), "-input", txt, "-output", lux],
                                  stdout=subprocess.DEVNULL)
            out["n%d_src" % nv], out["n%d_dst" % nv] = s, d
            out["n%d_lux" % nv] = np.fromfile(lux, np.uint8)
    np.savez_compressed(os.path.join(HERE, "ref_converter.npz"), **out)
    print("wrote ref_converter.npz")
else:
    print("kept ref_converter.npz: %s not built" % os.path.normpath(converter))
