"""Golden fixture of the tests that compare with the reference itself (run where oracle/_ref is built).

Runs the UNMODIFIED reference compiled against the serial oneTBB stand-in (`make -C oracle ref ref_full`) on the
inputs the tests define and stores what they compare against in tests/golden/live_reference.npz:

  contract_a<algorithm>_{c_n,c_m,sha256}  contract_clustering with algorithm 0 / 1 / 2 on the graphs and clusterings
                                          of test_contraction_oracle.live_graphs / live_clusterings, canonicalised
                                          and stored as digests (the coarse graphs themselves are ~1.3 MB)
  multigraph<i>_*, multigraph_c_n         raw contract_clustering results (default algorithm) on
                                          test_contraction_oracle.multigraph_cases
  full_<run>_{cut,part}                   KaMinPar::compute_partition of the whole reference partitioner
                                          (libkaminpar_ref_full.so) for test_reference_full_cpu

    python tests/golden/make_live_reference_golden.py
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import bindings as B  # noqa: E402
from oracle import contraction_oracle as CO  # noqa: E402
from tests import helpers as H  # noqa: E402
from tests import test_contraction_oracle as T  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "live_reference.npz")
LIB_FULL = os.path.join(ROOT, "oracle", "_ref", "libkaminpar_ref_full.so")
# (run, graph, k, seed): walshaw_k16_s0 twice, the reference is deterministic for a seed
FULL_RUNS = [("walshaw_k16_s0", "walshaw_data", 16, 0), ("walshaw_k16_s0_again", "walshaw_data", 16, 0),
             ("walshaw_k16_s1", "walshaw_data", 16, 1), ("rgg2d_k4_s0", "rgg2d", 4, 0)]


def compute_partition(lib, g, k, seed):
    out = np.zeros(g.n, np.uint32)
    cut = lib.kmpfull_compute_partition(C.c_uint32(g.n), g.xadj.ctypes.data_as(C.c_void_p),
                                        g.adjncy.ctypes.data_as(C.c_void_p), None, None, C.c_uint32(k),
                                        C.c_double(0.03), C.c_int(seed), C.c_int(1), out.ctypes.data_as(C.c_void_p))
    return int(cut), out


def main():
    assert B.have_reference() and os.path.exists(LIB_FULL), "build oracle/_ref first: make -C oracle ref ref_full"
    out = {}
    for algorithm in (0, 1, 2):
        rng = np.random.default_rng(algorithm)
        rows = []
        for g in T.live_graphs():
            for cl in T.live_clusterings(g, rng):
                o = CO.canonicalize(**B.ref_contract(g, cl, algorithm), clustering=cl)
                rows.append((o["c_n"], len(o["c_adjncy"]), T.digest(o)))
        out[f"contract_a{algorithm}_c_n"] = np.array([r[0] for r in rows], np.int64)
        out[f"contract_a{algorithm}_c_m"] = np.array([r[1] for r in rows], np.int64)
        out[f"contract_a{algorithm}_sha256"] = np.array([r[2] for r in rows])
    c_n = []
    for i, (g, cl) in enumerate(T.multigraph_cases()):
        r = B.ref_contract(g, cl, 1)
        c_n.append(r.pop("c_n"))
        out.update({f"multigraph{i}_{k}": v for k, v in r.items()})
    out["multigraph_c_n"] = np.array(c_n, np.int64)
    lib = C.CDLL(LIB_FULL)
    lib.kmpfull_compute_partition.restype = C.c_longlong
    for run, name, k, seed in FULL_RUNS:
        cut, part = compute_partition(lib, H.load_graph(name), k, seed)
        out[f"full_{run}_cut"] = np.array([cut], np.int64)
        out[f"full_{run}_part"] = part.astype(np.uint8 if k <= 256 else np.uint32)
        print(run, "cut", cut)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
