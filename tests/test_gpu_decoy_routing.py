"""Decoy attempts at the edges of the repair-pass routing, GPU against the CPU oracle: an attempt is grown once, repaired with
32-bit position masks up to 32 residues and with 64-bit ones from 33 on, and dropped when it needs a 61st residue.  The
precursors below give decoys of exactly 32, 33 and 60 residues (and attempts that grow past 60)."""
import numpy as np
import pytest

import maxdecoy
from maxdecoy import Modification, synth
from oracle_lib import oracle_engine
import workloads as wl

pytestmark = pytest.mark.gpu

PHOSPHO_S = Modification("x:21", "Phospho", "A", False, "S", 79.966331)


@pytest.fixture(scope="module")
def gpu():
    e = maxdecoy.Engine()
    yield e
    e.close()


@pytest.fixture(scope="module")
def cpu():
    e = oracle_engine(8)
    yield e
    e.close()


@pytest.mark.parametrize("mods,nvar", [((synth.CAM,), 0), ((synth.CAM, synth.OXM), 3), ((synth.CAM, synth.OXM, PHOSPHO_S), 2)])
def test_decoy_lengths_at_routing_edges_bit_exact(gpu, cpu, mods, nvar, monkeypatch):
    """No variable letter, one (the position-mask path) and two (the generic enumeration)."""
    for e in (gpu, cpu):
        e.digest(list(wl.proteins(300)), 2, 5, 50)
        e.set_modifications(list(mods), nvar)
        e.index_build()
    pre = wl.routing_precursors()
    dc = cpu.generate_decoys(pre, 60, maxdecoy.DECOY_REFERENCE_RANDOM, seed=5)
    dg = gpu.generate_decoys(pre, 60, maxdecoy.DECOY_REFERENCE_RANDOM, seed=5)
    for k in dc:
        assert np.array_equal(dg[k], dc[k]), k
    lens = set(np.diff(dg["seq_off"]).tolist())
    assert {32, 33, 60} <= lens
    monkeypatch.setenv("MD_DECOY_WIDE_ONLY", "1")
    dw = gpu.generate_decoys(pre, 60, maxdecoy.DECOY_REFERENCE_RANDOM, seed=5)
    for k in dc:
        assert np.array_equal(dw[k], dc[k]), k
