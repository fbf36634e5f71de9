"""Decoy generation across rounds, GPU against the CPU oracle, bit for bit.

The host plans REFERENCE_RANDOM / PERMUTE_TARGET decoys in rounds: every unfinished spectrum gets a budget of attempts,
split into list entries of at most MD_ROUND_ATTEMPTS (4096) consecutive attempt ordinals, and a select kernel per level
keeps each spectrum's first distinct successes -- through a shared-memory hash set, or, when that set would not fit, an
exact quadratic scan (k_decoy_select's two routes, "hash" and "n2" in the trace).  The results must depend on (seed,
spectrum_id, attempt) alone: not on the entry size, the select route, the repair loop's refill constants, the precursor
order or the round budgets.

- Test builds of decoy.cu with 64-attempt entries and either 6-bit hashes or the quadratic select (and the repair loop's
  refill threshold, ring size and ring period at their extremes, with the device-side substitution check) run the usual
  workloads through many rounds and levels.
- The default build reaches several levels and the quadratic select with 12000 decoys per spectrum.
- Precursor order, duplicate precursors, round budgets, extreme seeds and spectrum ids, attempt caps and the 32-bit
  residual refusals.

Which select kernel ran at which level comes from the engine's trace (MD_TRACE, one line per select launch)."""
import re

import numpy as np
import pytest

import maxdecoy
from maxdecoy import Modification, SearchParams, synth
from oracle_lib import oracle_engine
import testbuild
import workloads as wl

pytestmark = pytest.mark.gpu

RANDOM, PERMUTE = maxdecoy.DECOY_REFERENCE_RANDOM, maxdecoy.DECOY_PERMUTE_TARGET
PHOSPHO_S = Modification("x:21", "Phospho", "A", False, "S", 79.966331)
K_CTERM_FIX = Modification("x:259", "Label:13C(6)15N(2)", "C", True, "K", 8.014199)
Q_NTERM_VAR = Modification("unimod:28", "Gln->pyro-Glu", "N", False, "Q", -17.026549)

VARIANTS = {
    # 6-bit hashes: the exact-compare fallback of k_decoy_select in most entries; a refill whenever one lane is free, the
    # smallest ring (every lane runs dry) topped up at every step
    "tiny_rounds_hash": ["-DMD_ROUND_ATTEMPTS=64", "-DMD_SELECT_HASH_MASK=0x3Full", "-DMD_REFILL_MIN=1", "-DMD_RNG_RING=4", "-DMD_RNG_PERIOD=1",
                         "-DMD_DECOY_CHECK"],
    # every level through the exact scan of k_decoy_select; a refill only when the whole warp is free
    "tiny_rounds_n2": ["-DMD_ROUND_ATTEMPTS=64", "-DMD_SELECT_SMEM_MAX=0", "-DMD_REFILL_MIN=32", "-DMD_RNG_RING=16", "-DMD_RNG_PERIOD=5", "-DMD_DECOY_CHECK"],
}
VARIANT_KERNEL = {"tiny_rounds_hash": "hash", "tiny_rounds_n2": "n2"}

# name -> (modifications, max variable modifications, precursors, decoys per spectrum, mode, seed)
WORKLOADS = {
    "cam": ((synth.CAM,), 0, "spectra", 200, RANDOM, 11),
    "cam_oxm": ((synth.CAM, synth.OXM), 3, "spectra_ox", 200, RANDOM, 11),
    "two_var_letters": ((synth.CAM, synth.OXM, PHOSPHO_S), 2, "spectra_ox", 150, RANDOM, 13),
    "long_cam": ((synth.CAM,), 0, "long", 60, RANDOM, 3),
    "long_cam_oxm": ((synth.CAM, synth.OXM), 3, "long", 60, RANDOM, 3),
    "degenerate_fixed": wl.degenerate_mod_sets()[0] + ("spectra16", 150, RANDOM, 17),
    "degenerate_var": wl.degenerate_mod_sets()[1] + ("spectra16", 150, RANDOM, 17),
    "stored": ((synth.CAM,), 0, "spectra", 200, RANDOM, 21),
    "permuted_targets": ((synth.CAM,), 0, "spectra", 50, PERMUTE, 5),
    "terminal": ((synth.CAM, K_CTERM_FIX, Q_NTERM_VAR), 2, "spectra", 60, RANDOM, 9),
}

SELECT_RE = re.compile(r"decoy select round (\d+) level (\d+): entries=(\d+) kernel=(\w+)")


def _traced(lib=None):
    """An engine that writes the per-round trace to stderr (MD_TRACE is read when the engine is created)."""
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("MD_TRACE", "1")
        return maxdecoy.Engine(lib=lib)


def _selects(err):
    """(round, level, entries, kernel) of every select launch in a captured stderr."""
    return [(int(r), int(lv), int(n), k) for r, lv, n, k in SELECT_RE.findall(err)]


@pytest.fixture(scope="module")
def gpu():
    e = _traced()
    yield e
    e.close()


@pytest.fixture(scope="module")
def cpu():
    e = oracle_engine(8)
    yield e
    e.close()


@pytest.fixture(scope="module")
def variants():
    libs = testbuild.libraries(list(VARIANTS.values()))
    engines = {name: _traced(maxdecoy.load(so)) for name, so in zip(VARIANTS, libs)}
    yield engines
    for e in engines.values():
        e.close()


def _setup(engines, mods, nvar, n_prot=300):
    for e in engines:
        e.digest(list(wl.proteins(n_prot)), 2, 5, 50)
        e.set_modifications(list(mods), nvar)
        e.index_build()
        e.set_decoy_store([])


def _precursors(cpu, kind):
    if kind == "long":
        return wl.heavy_precursors() + wl.routing_precursors()
    sp, _ = wl.spectra(300, 16 if kind == "spectra16" else 24, 2, with_ox=kind == "spectra_ox")
    return wl.precursors_of(cpu, sp)


def _prepare(g, cpu, name):
    """Sets both engines up for workload `name`; returns (precursors, n, mode, seed)."""
    mods, nvar, kind, n, mode, seed = WORKLOADS[name]
    _setup((g, cpu), mods, nvar)
    pre = _precursors(cpu, kind)
    if name == "stored":    # some of the decoys the generator would find, plus sequences it never finds
        seqs = wl.decoy_strings(cpu.generate_decoys(pre, 80, RANDOM, seed=seed))
        store = seqs[::3] + seqs[1::7] + ["GGGGG", "A" * 60]
        for e in (g, cpu):
            e.set_decoy_store(store)
    return pre, n, mode, seed


def assert_tables_equal(a, b):
    assert sorted(a) == sorted(b) == ["attempt", "mod_weight", "off", "seq", "seq_off", "var_mask", "weight"]
    for k in a:
        assert a[k].shape == b[k].shape, k
        assert np.array_equal(a[k], b[k]), k


def assert_identify_equal(g, cpu, sp, prm):
    pg, stg, scg, offg = g.identify(sp, prm, want_all_scores=True)
    pc, stc, scc, offc = cpu.identify(sp, prm, want_all_scores=True)
    assert np.array_equal(offg, offc) and np.array_equal(scg, scc)
    for k in pg.dtype.names:
        if k != "_pad":
            assert np.array_equal(pg[k], pc[k]), k
    assert stg["n_decoys"] == stc["n_decoys"]


def _rows(table):
    """Per precursor row: its decoys (sequences, masks, weights, ordinals), in the table's order."""
    seqs = wl.decoy_strings(table)
    off = table["off"]
    cols = [table[k].tolist() for k in ("var_mask", "weight", "mod_weight", "attempt")]
    return [(seqs[a:b],) + tuple(c[a:b] for c in cols) for a, b in zip(off[:-1].tolist(), off[1:].tolist())]


def _by_id(table, pre):
    return dict(zip((p[4] for p in pre), _rows(table)))


def _subset(sp, idx):
    off = sp.peak_off.astype(np.int64)
    parts = [np.arange(off[i], off[i + 1]) for i in idx]
    new_off = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.uint64)
    take = np.concatenate(parts)
    return maxdecoy.Spectra(sp.precursor_mz[idx], sp.charge[idx], new_off, sp.peak_mz[take], sp.peak_intensity[take])


# ------------------------------------------------------------------------------------------------ test builds
@pytest.mark.parametrize("workload", list(WORKLOADS))
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_variant_build_decoys_bit_exact(variants, cpu, variant, workload, capfd):
    g = variants[variant]
    try:
        pre, n, mode, seed = _prepare(g, cpu, workload)
        capfd.readouterr()
        dg = g.generate_decoys(pre, n, mode, seed=seed)
        sel = _selects(capfd.readouterr().err)
        dc = cpu.generate_decoys(pre, n, mode, seed=seed)
        assert_tables_equal(dg, dc)
        assert len(dc["attempt"]) > 0
    finally:
        for e in (g, cpu):
            e.set_decoy_store([])
    assert sel and {k for _, _, _, k in sel} == {VARIANT_KERNEL[variant]}
    assert max(lv for _, lv, _, _ in sel) >= 1                # several 64-attempt entries of one spectrum in a round
    if workload == "stored":
        assert np.any(dg["attempt"] == maxdecoy.DECOY_STORED)
    if workload.startswith("long"):
        assert {32, 33, 60} <= set(np.diff(dg["seq_off"]).tolist())


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_variant_build_identify_bit_exact(variants, cpu, variant, capfd):
    """Decoy scores are laid out by the decoys' order: after many rounds and levels they must still be the oracle's."""
    g = variants[variant]
    _setup((g, cpu), (synth.CAM, synth.OXM), 3, n_prot=600)
    sp, _ = wl.spectra(600, 96, 2, with_ox=True)
    capfd.readouterr()
    assert_identify_equal(g, cpu, sp, SearchParams(10, 10, n_decoys=200, seed=3, top_k=5))
    sel = _selects(capfd.readouterr().err)
    assert max(r for r, _, _, _ in sel) >= 1 and max(lv for _, lv, _, _ in sel) >= 1


# ------------------------------------------------------------------------------------------------ default build
def _two_heavy(cpu):
    sp, _ = wl.spectra(300, 24, 2)
    pre = [p for p in wl.precursors_of(cpu, sp) if 1_800_000_000 < p[0] < 2_600_000_000][:2]
    assert len(pre) == 2
    return sp, pre


def test_large_counts_take_several_levels_and_quadratic_select(gpu, cpu, capfd):
    """12000 decoys: round 0 asks for 13232 attempts per spectrum, entries of 4096, 4096, 4096 and 944.  Level 0 fits the
    hash set; levels 1-3 would need more than 220 KB of shared memory and run the exact scan.  5000 decoys: two levels,
    both hashed."""
    _setup((gpu, cpu), (synth.CAM,), 0)
    _, pre = _two_heavy(cpu)
    for n, kernels in ((12000, ["hash", "n2", "n2", "n2"]), (5000, ["hash", "hash"])):
        capfd.readouterr()
        dg = gpu.generate_decoys(pre, n, RANDOM, seed=7)
        sel = _selects(capfd.readouterr().err)
        assert [k for r, _, _, k in sel if r == 0] == kernels, sel
        assert all(e == 2 for r, _, e, _ in sel if r == 0)
        dc = cpu.generate_decoys(pre, n, RANDOM, seed=7)
        assert_tables_equal(dg, dc)
        assert np.all(np.diff(dg["off"]) == n)
        assert int(dg["attempt"].max()) >= len(kernels[:-1]) * 4096   # decoys from the last level were kept


def test_large_counts_identify_bit_exact(gpu, cpu, capfd):
    _setup((gpu, cpu), (synth.CAM,), 0)
    sp, pre = _two_heavy(cpu)
    sub = _subset(sp, [p[4] for p in pre])
    capfd.readouterr()
    assert_identify_equal(gpu, cpu, sub, SearchParams(10, 10, n_decoys=12000, seed=7, top_k=5))
    assert "n2" in {k for _, _, _, k in _selects(capfd.readouterr().err)}


def test_precursor_order_and_duplicates_do_not_change_decoys(gpu, cpu):
    """The host sorts spectra into mass buckets to schedule the attempts; the order only steers which attempts run side by
    side.  Reversed, shuffled and repeated precursors give every spectrum the same decoys."""
    _setup((gpu, cpu), (synth.CAM, synth.OXM), 3)
    pre = _precursors(cpu, "spectra_ox")
    ref = gpu.generate_decoys(pre, 200, RANDOM, seed=11)
    assert_tables_equal(ref, cpu.generate_decoys(pre, 200, RANDOM, seed=11))
    want = _by_id(ref, pre)
    shuffled = [pre[i] for i in np.random.default_rng(5).permutation(len(pre))]
    for order in (pre[::-1], shuffled):
        assert _by_id(gpu.generate_decoys(order, 200, RANDOM, seed=11), order) == want
    rows = _rows(gpu.generate_decoys(pre + pre, 200, RANDOM, seed=11))
    assert rows[: len(pre)] == rows[len(pre):] == _rows(ref)


@pytest.mark.parametrize("want0", [100, 400])
@pytest.mark.parametrize("later", [100, 300])
def test_round_budgets_do_not_change_decoys(gpu, cpu, want0, later, monkeypatch, capfd):
    """MD_DECOY_WANT0_PCT / MD_DECOY_LATER_PCT set how many attempts round 0 and the later rounds ask for.  At 400 % and
    1200 decoys round 0 asks for 4832 attempts per spectrum: two levels."""
    _setup((gpu, cpu), (synth.CAM,), 0)
    pre = _precursors(cpu, "spectra")
    monkeypatch.setenv("MD_DECOY_WANT0_PCT", str(want0))
    monkeypatch.setenv("MD_DECOY_LATER_PCT", str(later))
    capfd.readouterr()
    dg = gpu.generate_decoys(pre, 1200, RANDOM, seed=11)
    sel = _selects(capfd.readouterr().err)
    assert_tables_equal(dg, cpu.generate_decoys(pre, 1200, RANDOM, seed=11))
    assert max(lv for r, lv, _, _ in sel if r == 0) == (1 if want0 == 400 else 0)


EDGE = [
    (500_000_000, 500_000_000, 500_000_000, 2, 0xFFFFFFF0),       # zero-width window
    (60_000_000, 59_000_000, 61_000_000, 1, 0xFFFFFFFF),          # lighter than any residue plus water
    (9_000_000_000, 8_999_900_000, 9_000_100_000, 3, 7),          # every attempt grows past 60 residues
    (1_200_000_000, 1_199_988_000, 1_200_012_000, 2, 8),          # 10 ppm: one decoy within the attempt cap
]


def test_input_edges_in_one_batch(gpu, cpu):
    """Spectra that use up their attempt cap (16 n + 1024) without n decoys, spectrum ids near 2^32 and a seed with its high
    32 bits set (the second word of the Philox key), next to ordinary precursors; 1 and 0 decoys per spectrum."""
    _setup((gpu, cpu), (synth.CAM,), 0)
    pre = EDGE + _precursors(cpu, "spectra")[:6]
    seed = 0xFEDCBA9876543210
    for n in (50, 1, 0):
        dg = gpu.generate_decoys(pre, n, RANDOM, seed=seed)
        dc = cpu.generate_decoys(pre, n, RANDOM, seed=seed)
        assert_tables_equal(dg, dc)
        if n == 50:
            assert np.diff(dc["off"]).tolist() == [0, 0, 0, 1] + [50] * 6
    # the high word of the seed is part of the key
    assert not np.array_equal(gpu.generate_decoys(pre[4:], 50, RANDOM, seed=seed)["seq"],
                              gpu.generate_decoys(pre[4:], 50, RANDOM, seed=seed & 0xFFFFFFFF)["seq"])


def test_residual_range_refusals(gpu, cpu):
    """Decoy generation works in 32-bit residuals: a window reaching further than 2^30 - 1 uDa from its precursor mass, or a
    residue whose mass with its fixed modification reaches 2^29 uDa, is refused with MD_ERR_UNSUPPORTED (the oracle accepts
    both).  The limits are exact, and the engine's next call is unaffected."""
    _setup((gpu, cpu), (synth.CAM,), 0)
    pre = _precursors(cpu, "spectra")[:6]
    m = 1_200_000_000

    def check_normal():
        assert_tables_equal(gpu.generate_decoys(pre, 40, RANDOM, seed=1), cpu.generate_decoys(pre, 40, RANDOM, seed=1))

    edge = pre + [(m, m - (2**30 - 1), m + 10_000, 2, 40)]
    assert_tables_equal(gpu.generate_decoys(edge, 5, RANDOM, seed=1), cpu.generate_decoys(edge, 5, RANDOM, seed=1))
    for lo, hi in ((m - 2**30, m + 10_000), (m - 1_100_000_000, m + 1_100_000_000)):
        wide = pre + [(m, lo, hi, 2, 40)]
        with pytest.raises(maxdecoy.MaxDecoyError) as ei:
            gpu.generate_decoys(wide, 5, RANDOM, seed=1)
        assert ei.value.status == -5 and "left the 32-bit range" in str(ei.value)
        assert len(cpu.generate_decoys(wide, 5, RANDOM, seed=1)["attempt"]) > 0
        check_normal()
    w = 186_079_310                                              # W, the heaviest residue
    for delta, ok in ((2**29 - 1 - w, True), (2**29 - w, False), (400_000_000, False)):
        heavy_w = Modification("x:9", "Heavy", "A", True, "W", delta / 1e6)
        assert heavy_w.mono_mass_int == delta
        _setup((gpu, cpu), (synth.CAM, heavy_w), 0)
        if ok:
            assert_tables_equal(gpu.generate_decoys(pre, 40, RANDOM, seed=1), cpu.generate_decoys(pre, 40, RANDOM, seed=1))
        else:
            with pytest.raises(maxdecoy.MaxDecoyError) as ei:
                gpu.generate_decoys(pre, 40, RANDOM, seed=1)
            assert ei.value.status == -5 and "below 536 Da" in str(ei.value)
            assert len(cpu.generate_decoys(pre, 40, RANDOM, seed=1)["attempt"]) > 0
        _setup((gpu, cpu), (synth.CAM,), 0)
        check_normal()
