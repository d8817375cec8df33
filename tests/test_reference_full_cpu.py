"""CPU: the whole UNMODIFIED reference partitioner (oracle/_ref/libkaminpar_ref_full.so: every kaminpar-shm /
kaminpar-common translation unit on the serial oneTBB stand-in, `make -C oracle ref_full`) through the same C entry
point the B200-integrated build exports (integration/partition_driver.cc). Pins the harness of
tests/test_gpu_integration.py against the reference's own end-to-end properties
(tests/endtoend/shm_endtoend_test.cc:142-247). The partitions and cuts the reference returned are stored in
tests/golden/live_reference.npz by tests/golden/make_live_reference_golden.py."""
import os

import numpy as np

from oracle import bindings as B
from tests import helpers as H


def test_reference_compute_partition_properties():
    d = np.load(os.path.join(H.GOLDEN, "live_reference.npz"))

    def run(key):
        return int(d[f"full_{key}_cut"][0]), d[f"full_{key}_part"]

    g = H.load_graph("walshaw_data")
    cut, p = run("walshaw_k16_s0")
    assert len(p) == g.n and (p < 16).all() and cut == B.oracle_edge_cut(g, p) and cut <= 2000
    cut2, p2 = run("walshaw_k16_s0_again")
    assert cut2 == cut and np.array_equal(p, p2)
    _, p3 = run("walshaw_k16_s1")
    assert not np.array_equal(p, p3)
    g = H.load_graph("rgg2d")
    cut, p = run("rgg2d_k4_s0")
    assert g.n == 1024 and g.m == 8226 and len(p) == g.n and (p < 4).all() and cut == B.oracle_edge_cut(g, p)
