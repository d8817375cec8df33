"""Graph IO (SURVEY §8f-3): METIS text and ParHIP binary readers / writers, partition files -- checked against the
reference's own sample files (misc/rgg2d*, stored gzip-compressed under tests/golden/) and by round trips."""
import gzip
import os

import numpy as np
import pytest

from kaminpar_b200.graph import (CSRGraph, random_weights, read_metis, read_parhip, read_partition, rmat, write_metis,
                                 write_parhip, write_partition)
from tests import helpers as H


def sample_file(fname, tmp_path):
    """The reference's sample file `fname`, unpacked from tests/golden/<fname>.gz into tmp_path."""
    path = str(tmp_path / fname)
    with gzip.open(os.path.join(H.GOLDEN, fname + ".gz"), "rb") as src, open(path, "wb") as dst:
        dst.write(src.read())
    return path


@pytest.mark.parametrize("fname", ["rgg2d-32bit.parhip", "rgg2d-64bit.parhip"])
def test_parhip_reader_on_the_references_sample_files(fname, tmp_path):
    g = read_parhip(sample_file(fname, tmp_path))
    gold = H.load_graph("rgg2d")  # parsed from misc/rgg2d.metis by the reference (tests/golden/make_golden.py)
    assert g.n == 1024 and g.m == 8226  # test_pykaminpar.py:78-92
    assert np.array_equal(g.xadj, gold.xadj) and np.array_equal(g.adjncy, gold.adjncy)
    assert g.vwgt is None and g.adjwgt is None
    m = read_metis(sample_file("rgg2d.metis", tmp_path))
    assert np.array_equal(m.xadj, g.xadj) and np.array_equal(m.adjncy, g.adjncy)


@pytest.mark.parametrize("weights", [(0, 0), (5, 0), (0, 7), (4, 9)])
def test_parhip_and_metis_round_trips(tmp_path, weights):
    g = random_weights(rmat(10, 8, 3), 2, max_vwgt=weights[0], max_adjwgt=weights[1])
    p = str(tmp_path / "g.parhip")
    write_parhip(g, p)
    h = read_parhip(p)
    for a, b in ((g.xadj, h.xadj), (g.adjncy, h.adjncy), (g.vwgt, h.vwgt), (g.adjwgt, h.adjwgt)):
        assert (a is None and b is None) or np.array_equal(a, b)
    q = str(tmp_path / "g.metis")
    write_metis(g, q)
    k = read_metis(q)
    assert np.array_equal(g.xadj, k.xadj) and np.array_equal(g.adjncy, k.adjncy)
    assert (g.vwgt is None and k.vwgt is None) or np.array_equal(g.vwgt, k.vwgt)
    assert (g.adjwgt is None and k.adjwgt is None) or np.array_equal(g.adjwgt, k.adjwgt)


def test_partition_file_round_trip(tmp_path):
    part = np.random.default_rng(0).integers(0, 17, 1000).astype(np.uint32)
    p = str(tmp_path / "part.txt")
    write_partition(p, part)
    assert open(p).read().splitlines()[:3] == [str(int(x)) for x in part[:3]]  # one block id per line
    assert np.array_equal(read_partition(p), part)
    write_partition(p, part[:1])
    assert np.array_equal(read_partition(p), part[:1])
