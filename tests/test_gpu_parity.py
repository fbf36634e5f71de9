"""GPU parity: the CUDA library (through the C ABI) against the CPU oracle on identical seeded inputs.
Bit-exact for peptides, integer masses, windows, candidates, decoys and raw scores."""
import numpy as np
import pytest

import maxdecoy
from maxdecoy import SearchParams, synth
from oracle_lib import oracle_engine
import workloads as wl

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    e = maxdecoy.Engine()
    assert e.backend == "cuda-sm100a"
    yield e
    e.close()


@pytest.fixture(scope="module")
def cpu():
    e = oracle_engine(8)
    yield e
    e.close()


def assert_tables_equal(a, b, keys=None):
    for k in (keys or a.keys()):
        assert a[k].shape == b[k].shape, k
        assert np.array_equal(a[k], b[k]), k


def test_digest_golden_p77377(gpu):
    g = wl.p77377()
    n = gpu.digest([g["sequence"]], **g["params"])
    assert n == 71
    got = set(gpu.sequences_of(gpu.peptides()))
    want = {s.replace("I", "J").replace("L", "J") for s in g["peptides"]}
    assert got == want


@pytest.mark.parametrize("n_prot,mc,min_len,max_len", [(300, 1, 5, 50), (2000, 2, 5, 50), (200, 0, 1, 60), (150, 5, 6, 30)])
def test_digest_matches_oracle(gpu, cpu, n_prot, mc, min_len, max_len):
    prots = list(wl.proteins(n_prot))
    ng = gpu.digest(prots, mc, min_len, max_len)
    nc = cpu.digest(prots, mc, min_len, max_len)
    assert ng == nc
    assert_tables_equal(gpu.peptides(), cpu.peptides())


def test_digest_edge_cases(gpu, cpu):
    cases = ["", "K", "KR", "KP", "MKPR", "AAAAKAAAAR", "RRRRRR", "KKKKPKKKK", "MSLREKTISGAK" * 3, "ILILIKLILIR", "ABZXUOK", "A" * 70 + "K" + "C" * 10]
    for mc in (0, 2):
        ng = gpu.digest(cases, mc, 1, 60)
        nc = cpu.digest(cases, mc, 1, 60)
        assert ng == nc
        assert_tables_equal(gpu.peptides(), cpu.peptides())
    assert gpu.digest([], 2, 5, 50) == 0
    assert gpu.digest(["", ""], 2, 5, 50) == 0


def _setup(e, n_prot, mc, mods, nvar):
    e.digest(list(wl.proteins(n_prot)), mc, 5, 50)
    e.set_modifications(list(mods), nvar)
    e.index_build()


@pytest.mark.parametrize("mods,nvar", [((synth.CAM,), 0), ((synth.CAM, synth.OXM), 3)])
def test_index_and_candidates(gpu, cpu, mods, nvar):
    for e in (gpu, cpu):
        _setup(e, 600, 2, mods, nvar)
    sg, sc = gpu.index_stats(), cpu.index_stats()
    for k in ("n_peptides", "seq_bytes", "min_key", "max_key"):
        assert sg[k] == sc[k]
    n = sg["n_peptides"]
    pg, kg = gpu.index_export(0, n)
    pc, kc = cpu.index_export(0, n)
    assert np.array_equal(kg, kc) and np.array_equal(pg, pc)
    sp, _ = wl.spectra(600, 200, 2, with_ox=len(mods) > 1)
    pre = wl.precursors_of(cpu, sp)
    assert pre == wl.precursors_of(gpu, sp)
    lo = [p[1] for p in pre] + [0, -5, 10**12, 2000000000]
    hi = [p[2] for p in pre] + [10**12, -1, 10**12 + 5, 1999999999]
    bg, eg = gpu.window_search(lo, hi)
    bc, ec = cpu.window_search(lo, hi)
    assert np.array_equal(bg, bc) and np.array_equal(eg, ec)
    # wide windows exercise the variable-modification enumeration
    wide = [(p[0], p[0] - 40_000_000, p[0] + 40_000_000, p[3], p[4]) for p in pre[:40]]
    for prs in (pre, wide):
        assert_tables_equal(gpu.candidates(prs), cpu.candidates(prs))


@pytest.mark.parametrize("mods,nvar", [((synth.CAM,), 0), ((synth.CAM, synth.OXM), 3)])
def test_decoys_random_bit_exact(gpu, cpu, mods, nvar):
    for e in (gpu, cpu):
        _setup(e, 300, 2, mods, nvar)
    sp, _ = wl.spectra(300, 24, 2, with_ox=len(mods) > 1)
    pre = wl.precursors_of(cpu, sp)
    dg = gpu.generate_decoys(pre, 200, maxdecoy.DECOY_REFERENCE_RANDOM, seed=11)
    dc = cpu.generate_decoys(pre, 200, maxdecoy.DECOY_REFERENCE_RANDOM, seed=11)
    assert_tables_equal(dg, dc)
    assert len(dg["attempt"]) > 0


@pytest.mark.parametrize("mods,nvar", [((synth.CAM,), 0), ((synth.CAM, synth.OXM), 3)])
def test_decoys_random_long_sequences_bit_exact(gpu, cpu, mods, nvar, monkeypatch):
    """Heavy precursors: attempts grow past 32 residues, which the kernel hands from its 32-bit-mask pass to the 64-bit
    one; sequences near the 60-residue cap are dropped.  Also: the 64-bit pass alone gives the same decoys."""
    for e in (gpu, cpu):
        _setup(e, 300, 2, mods, nvar)
    pre = wl.heavy_precursors()
    dc = cpu.generate_decoys(pre, 120, maxdecoy.DECOY_REFERENCE_RANDOM, seed=3)
    dg = gpu.generate_decoys(pre, 120, maxdecoy.DECOY_REFERENCE_RANDOM, seed=3)
    assert_tables_equal(dg, dc)
    lens = np.diff(dg["seq_off"])
    assert lens.max() > 32 and lens.min() <= 32
    monkeypatch.setenv("MD_DECOY_WIDE_ONLY", "1")
    dw = gpu.generate_decoys(pre, 120, maxdecoy.DECOY_REFERENCE_RANDOM, seed=3)
    assert_tables_equal(dw, dc)


def test_decoys_random_degenerate_masses_bit_exact(gpu, cpu):
    """The modification sets of workloads.degenerate_mod_sets make letters collide (equal masses, near-ties on either side
    of a midpoint) and add two variable letters, one of them also fixed (the generic variable-modification path).  The
    substitution search of the kernel (bucket tables) must agree with the oracle's literal 20-way scan."""
    sp, _ = wl.spectra(300, 16, 2)
    for mods, nvar in wl.degenerate_mod_sets():
        for e in (gpu, cpu):
            _setup(e, 300, 2, mods, nvar)
        pre = wl.precursors_of(cpu, sp)
        dg = gpu.generate_decoys(pre, 150, maxdecoy.DECOY_REFERENCE_RANDOM, seed=17)
        dc = cpu.generate_decoys(pre, 150, maxdecoy.DECOY_REFERENCE_RANDOM, seed=17)
        assert_tables_equal(dg, dc)
        assert len(dg["attempt"]) > 0


@pytest.mark.parametrize("mods,nvar", [((synth.CAM,), 0), ((synth.CAM, synth.OXM), 3)])
def test_stored_decoys_bit_exact(gpu, cpu, mods, nvar):
    """Decoy reuse (tasks/identification.rs:259-283): same stored decoys taken, in the same order, the same remainder
    generated -- through md_generate_decoys and through md_identify (scores of the reused decoys included)."""
    for e in (gpu, cpu):
        _setup(e, 300, 2, mods, nvar)
        e.set_decoy_store([])
    sp, _ = wl.spectra(300, 24, 2, with_ox=len(mods) > 1)
    pre = wl.precursors_of(cpu, sp)
    seqs = wl.decoy_strings(cpu.generate_decoys(pre, 80, maxdecoy.DECOY_REFERENCE_RANDOM, seed=21))
    store = seqs[::3] + seqs[1::7] + ["GGGGG", "AAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAA"]
    try:
        for e in (gpu, cpu):
            e.set_decoy_store(store)
        for n in (10, 80, 200):
            dg = gpu.generate_decoys(pre, n, maxdecoy.DECOY_REFERENCE_RANDOM, seed=21)
            dc = cpu.generate_decoys(pre, n, maxdecoy.DECOY_REFERENCE_RANDOM, seed=21)
            assert_tables_equal(dg, dc)
            assert np.any(dg["attempt"] == maxdecoy.DECOY_STORED)
        prm = SearchParams(10, 10, n_decoys=60, decoy_mode=0, seed=21, top_k=5)
        pg, stg, scg, offg = gpu.identify(sp, prm, want_all_scores=True)
        pc, stc, scc, offc = cpu.identify(sp, prm, want_all_scores=True)
        assert np.array_equal(offg, offc) and np.array_equal(scg, scc)
        for k in pg.dtype.names:
            if k != "_pad":
                assert np.array_equal(pg[k], pc[k]), k
        # the other modes ignore the store
        de = gpu.generate_decoys(pre[:4], 20, maxdecoy.DECOY_EXHAUSTIVE, seed=0)
        assert not np.any(de["attempt"] == maxdecoy.DECOY_STORED)
    finally:
        for e in (gpu, cpu):
            e.set_decoy_store([])


def test_expanded_variable_mode_bit_exact(gpu, cpu):
    """MD_VARMOD_EXPANDED: the same candidates in the same order (count vectors, fixed-weight order, placements in NChooseK
    order), the same scores and PSM rows -- with one and with two variable letters, narrow and wide windows."""
    from maxdecoy import Modification
    var_s = Modification("x:21", "Phospho", "A", False, "S", 79.966331)
    try:
        for mods, nvar in (((synth.CAM, synth.OXM), 3), ((synth.CAM, synth.OXM, var_s), 2)):
            for e in (gpu, cpu):
                e.digest(list(wl.proteins(300)), 2, 5, 50)
                e.set_modifications(list(mods), nvar)
                e.set_variable_mode(maxdecoy.VARMOD_EXPANDED)
                e.index_build()
            sp, _ = wl.spectra(300, 32, 2, with_ox=True)
            pre = wl.precursors_of(cpu, sp)
            wide = [(p[0], p[0] - 30_000_000, p[0] + 30_000_000, p[3], p[4]) for p in pre[:12]]
            for prs in (pre, wide):
                cg, cc = gpu.candidates(prs), cpu.candidates(prs)
                assert_tables_equal(cg, cc)
            assert len(cg["peptide_id"]) > 1000
            prm = SearchParams(10, 10, n_decoys=40, decoy_mode=0, seed=5, top_k=5)
            pg, stg, scg, offg = gpu.identify(sp, prm, want_all_scores=True)
            pc, stc, scc, offc = cpu.identify(sp, prm, want_all_scores=True)
            assert np.array_equal(offg, offc) and np.array_equal(scg, scc)
            for k in pg.dtype.names:
                if k != "_pad":
                    assert np.array_equal(pg[k], pc[k]), k
    finally:
        for e in (gpu, cpu):
            e.set_variable_mode(maxdecoy.VARMOD_REFERENCE)


def test_expanded_variable_mode_finds_partially_modified_peptides(gpu):
    """What the mode is for (SURVEY A.4 / 8(f) row 4): a peptide with two methionines of which ONE is oxidised is invisible
    to the reference's lookup (only the fully modified weight is queried) and is identified, placement included, in
    expanded mode."""
    prots = list(wl.proteins(400))
    sp, truth = synth.synthetic_spectra(prots, 400, 2, mods=(synth.CAM, synth.OXM), seed=11, frac_random=0.0, ox_prob=0.6, max_var=1)
    partial = [i for i, (q, m) in enumerate(truth) if m and q.count("M") >= 2]
    assert len(partial) >= 8
    won = {}
    try:
        for mode in (maxdecoy.VARMOD_REFERENCE, maxdecoy.VARMOD_EXPANDED):
            gpu.digest(prots, 2, 5, 50)
            gpu.set_modifications([synth.CAM, synth.OXM], 3)
            gpu.set_variable_mode(mode)
            gpu.index_build()
            seqs = gpu.sequences_of(gpu.peptides())
            psms, _ = gpu.identify(sp, SearchParams(10, 10, n_decoys=50, seed=1, top_k=1))
            top = psms[:, 0]
            won[mode] = sum(1 for i in partial if top["rank"][i] and not top["is_decoy"][i] and seqs[int(top["candidate"][i]) - 1] == truth[i][0]
                            and int(top["var_mask"][i]) == truth[i][1])
    finally:
        gpu.set_variable_mode(maxdecoy.VARMOD_REFERENCE)
    assert won[maxdecoy.VARMOD_REFERENCE] == 0
    assert won[maxdecoy.VARMOD_EXPANDED] >= 0.7 * len(partial)


def test_decoys_permute_bit_exact(gpu, cpu):
    for e in (gpu, cpu):
        _setup(e, 300, 2, (synth.CAM,), 0)
    sp, _ = wl.spectra(300, 24, 2)
    pre = wl.precursors_of(cpu, sp)
    dg = gpu.generate_decoys(pre, 50, maxdecoy.DECOY_PERMUTE_TARGET, seed=5)
    dc = cpu.generate_decoys(pre, 50, maxdecoy.DECOY_PERMUTE_TARGET, seed=5)
    assert_tables_equal(dg, dc)


@pytest.mark.parametrize("mods,nvar", [((synth.CAM,), 0), ((synth.CAM, synth.OXM), 2)])
def test_decoys_exhaustive_bit_exact(gpu, cpu, mods, nvar):
    """Exhaustive-enumeration mode (north star): identical sequences, order, weights and ordinals."""
    for e in (gpu, cpu):
        _setup(e, 300, 2, mods, nvar)
    sp, _ = wl.spectra(300, 48, 2)
    pre = wl.precursors_of(cpu, sp)
    # plus tiny precursors (few compositions: fewer decoys than requested) and a wide window
    pre += [(300_000_000, 299_000_000, 301_000_000, 2, 1000), (75_031_000, 75_000_000, 75_100_000, 1, 1001),
            (900_400_000, 800_000_000, 1_000_000_000, 2, 1002), (10_000_000, 9_000_000, 11_000_000, 1, 1003)]
    for n in (1, 37, 400):
        dg = gpu.generate_decoys(pre, n, maxdecoy.DECOY_EXHAUSTIVE, seed=0)
        dc = cpu.generate_decoys(pre, n, maxdecoy.DECOY_EXHAUSTIVE, seed=0)
        assert_tables_equal(dg, dc)
        assert len(dg["attempt"]) > 0


@pytest.mark.parametrize("mods,nvar,mode,nd", [((synth.CAM,), 0, 0, 100), ((synth.CAM, synth.OXM), 3, 0, 60), ((synth.CAM,), 0, 2, 30), ((synth.CAM,), 0, 0, 0),
                                               ((synth.CAM,), 0, 1, 40)])
def test_identify_bit_exact(gpu, cpu, mods, nvar, mode, nd):
    for e in (gpu, cpu):
        _setup(e, 600, 2, mods, nvar)
    sp, truth = wl.spectra(600, 96, 2, with_ox=len(mods) > 1)
    prm = SearchParams(10, 10, n_decoys=nd, decoy_mode=mode, seed=3, top_k=5)
    pg, stg, scg, offg = gpu.identify(sp, prm, want_all_scores=True)
    pc, stc, scc, offc = cpu.identify(sp, prm, want_all_scores=True)
    assert np.array_equal(offg, offc)
    assert np.array_equal(scg, scc)
    for f in ("spectrum_id", "rank", "is_decoy", "charge", "candidate", "var_mask", "mod_weight", "raw_score", "n_targets", "n_decoys"):
        assert np.array_equal(pg[f], pc[f]), f
    # scores: 1e-5 relative tolerance (north star); they are in fact derived from the same integer
    assert np.allclose(pg["score"], pc["score"], rtol=1e-5, atol=0)
    assert stg["n_targets"] == stc["n_targets"] and stg["n_decoys"] == stc["n_decoys"]
    assert stg["n_kernel_launches"] > 0


def _dense_spectra(n, n_peaks, seed=1):
    """Spectra with thousands of peaks (more unique bins than the kernel stages in shared memory)."""
    rng = np.random.default_rng(seed)
    sp, _ = wl.spectra(600, n, 2)
    off, mzs, ints = [0], [], []
    for s in range(n):
        base = np.sort(np.concatenate([sp.peak_mz[int(sp.peak_off[s]):int(sp.peak_off[s + 1])], rng.uniform(60.0, 2400.0, n_peaks)]))
        mzs.append(base)
        ints.append(rng.lognormal(4.0, 1.0, len(base)).astype(np.float32))
        off.append(off[-1] + len(base))
    return maxdecoy.Spectra(sp.precursor_mz, sp.charge, np.array(off, dtype=np.uint64), np.concatenate(mzs), np.concatenate(ints))


@pytest.mark.parametrize("case", ["wide_window_chunked", "wide_window_running_lists", "wide_window_split", "top_k_generic", "dense_peaks", "low_res_bins", "high_charge",
                                  "few_peaks_and_empty", "classic_kernel", "many_decoys_unsorted", "wide_window_split_classic", "wide_window_split_16"])
def test_identify_kernel_paths(gpu, cpu, case, monkeypatch):
    """The branches of k_score the 10-ppm / top-5 cases never reach: candidate chunks beyond shared memory with the
    generic top-k merge, the same with per-warp running top-k lists (top_k <= 8), spectra split into parts over several CTAs
    (what an open search over few spectra does), top_k > 8, spectra whose binned peaks do not fit shared memory, 1.0005-Da bins (one tile),
    fragment charges up to 3, and spectra that are not scored at all.  Since round 2 the usual batch goes through k_score_pipe
    (tables prebuilt, streamed in; split batches too, `wide_window_split_classic` is k_score's split): `classic_kernel` forces k_score for it, `many_decoys_unsorted` gives every spectrum more
    candidates than k_cand_order sorts (natural order), `dense_peaks` are the spectra the pipelined kernel leaves to k_score on
    the side stream, `wide_window_running_lists` its many-units-per-spectrum case."""
    for e in (gpu, cpu):
        _setup(e, 600, 2, (synth.CAM, synth.OXM), 2)
    sp, _ = wl.spectra(600, 24, 2, with_ox=True)
    kw = dict(n_decoys=30, seed=9, top_k=5)
    if case == "wide_window_chunked":
        kw.update(abs_lower_uda=60_000_000, abs_upper_uda=60_000_000, n_decoys=10, top_k=12)     # thousands of targets per spectrum
    elif case == "wide_window_running_lists":
        kw.update(abs_lower_uda=60_000_000, abs_upper_uda=60_000_000, n_decoys=10, top_k=5)
    elif case == "wide_window_split":
        kw.update(abs_lower_uda=60_000_000, abs_upper_uda=60_000_000, n_decoys=10, top_k=8)
        monkeypatch.setenv("MD_SCORE_SPLIT_MIN", "1")
    elif case == "wide_window_split_classic":
        kw.update(abs_lower_uda=60_000_000, abs_upper_uda=60_000_000, n_decoys=10, top_k=8)
        monkeypatch.setenv("MD_SCORE_SPLIT_MIN", "1")
        monkeypatch.setenv("MD_SCORE_SPLIT_CLASSIC", "1")
    elif case == "wide_window_split_16":
        kw.update(abs_lower_uda=60_000_000, abs_upper_uda=60_000_000, n_decoys=10, top_k=8)
        monkeypatch.setenv("MD_SCORE_PARTS", "16")
    elif case == "top_k_generic":
        kw.update(top_k=40)
    elif case == "classic_kernel":
        monkeypatch.setenv("MD_SCORE_CLASSIC", "1")
    elif case == "many_decoys_unsorted":
        kw.update(n_decoys=2300, top_k=8)
    elif case == "dense_peaks":
        sp = _dense_spectra(12, 2500)
    elif case == "low_res_bins":
        kw.update(fragment_tolerance=1.0005)
    elif case == "high_charge":
        sp = maxdecoy.Spectra(sp.precursor_mz * sp.charge / 5.0 - 1.007276 * sp.charge / 5.0 + 1.007276, np.full(len(sp), 5, dtype=np.uint8), sp.peak_off, sp.peak_mz,
                              sp.peak_intensity)
    elif case == "few_peaks_and_empty":
        off = sp.peak_off.copy()
        keep = np.ones(len(sp.peak_mz), dtype=bool)
        for s in (0, 5, 6):                                   # 3 peaks, no peaks, 9 peaks (minimum_peaks = 10)
            a, b = int(off[s]), int(off[s + 1])
            keep[a + (3 if s == 0 else (0 if s == 5 else 9)):b] = False
        lens = np.add.reduceat(keep.astype(np.int64), off[:-1].astype(np.int64))
        sp = maxdecoy.Spectra(sp.precursor_mz, sp.charge, np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64), sp.peak_mz[keep], sp.peak_intensity[keep])
    prm = SearchParams(10, 10, **kw)
    pg, stg, scg, offg = gpu.identify(sp, prm, want_all_scores=True)
    pc, stc, scc, offc = cpu.identify(sp, prm, want_all_scores=True)
    assert np.array_equal(offg, offc) and np.array_equal(scg, scc)
    for f in ("spectrum_id", "rank", "is_decoy", "charge", "candidate", "var_mask", "mod_weight", "raw_score", "score", "n_targets", "n_decoys"):
        assert np.array_equal(pg[f], pc[f]), f
    if case.startswith("wide_window"):
        assert int(np.diff(offg).max()) > 2 * 1536          # more candidates than two shared-memory chunks
    if case == "few_peaks_and_empty":
        assert np.all(pg["rank"][[0, 5, 6]] == 0) and np.any(pg["rank"][1] > 0)
    # without the per-candidate score output the PSM rows must be the same
    pg2, _ = gpu.identify(sp, prm)
    assert pg2.tobytes() == pg.tobytes()


def test_error_reporting(gpu):
    """The ABI reports what the reference panics on (and what lies outside the hot path) as status codes."""
    e = maxdecoy.Engine()
    with pytest.raises(maxdecoy.MaxDecoyError) as ei:
        e.index_build()                                       # no digest yet
    assert ei.value.status == -2
    e.digest(list(wl.proteins(50)), 2, 5, 50)
    with pytest.raises(maxdecoy.MaxDecoyError) as ei:
        e.set_modifications([maxdecoy.Modification("x:1", "bad position", "Q", True, "A", 42.0)], 0)
    assert ei.value.status == -1                              # position must be A, N or C (modification.rs:24-33)
    with pytest.raises(maxdecoy.MaxDecoyError):
        e.digest(["MKR"], 2, 5, 61)
    e.set_modifications([synth.CAM], 0)
    e.index_build()
    sp, _ = wl.spectra(600, 4, 2)
    with pytest.raises(maxdecoy.MaxDecoyError) as ei:
        e.identify(sp, SearchParams(10, 10, top_k=500))
    assert ei.value.status in (-1, -5)
    bad = maxdecoy.Spectra(sp.precursor_mz[:1], sp.charge[:1], np.array([0, 12], dtype=np.uint64), np.arange(12, 0, -1) * 50.0, np.ones(12, dtype=np.float32))
    with pytest.raises(maxdecoy.MaxDecoyError) as ei:
        e.identify(bad, SearchParams(10, 10, n_decoys=0))
    assert ei.value.status == -1 and "sorted" in str(ei.value)
    empty = maxdecoy.Spectra(np.zeros(0), np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64), np.zeros(0), np.zeros(0, dtype=np.float32))
    psms, st = e.identify(empty, SearchParams(10, 10))
    assert psms.shape == (0, 5) and st["n_spectra"] == 0
    e.close()


def test_passes_do_not_change_results(gpu, cpu, monkeypatch):
    """Batches too large for the workspaces run as several passes (open searches, 100k-spectrum files); forcing tiny
    passes must give the same PSM rows and the same per-candidate scores as one pass and as the oracle."""
    for e in (gpu, cpu):
        _setup(e, 600, 2, (synth.CAM, synth.OXM), 3)
    sp, _ = wl.spectra(600, 50, 2, with_ox=True)
    prm = SearchParams(10, 10, n_decoys=40, seed=3, top_k=5)
    one, st1, sc1, off1 = gpu.identify(sp, prm, want_all_scores=True)
    monkeypatch.setenv("MD_MAX_PASS_SPECTRA", "7")
    many, stm, scm, offm = gpu.identify(sp, prm, want_all_scores=True)
    monkeypatch.delenv("MD_MAX_PASS_SPECTRA")
    assert many.tobytes() == one.tobytes() and np.array_equal(scm, sc1) and np.array_equal(offm, off1)
    assert (stm["n_targets"], stm["n_decoys"], stm["n_pairs"]) == (st1["n_targets"], st1["n_decoys"], st1["n_pairs"])
    pc, _, scc, offc = cpu.identify(sp, prm, want_all_scores=True)
    assert np.array_equal(scm, scc) and np.array_equal(many["raw_score"], pc["raw_score"]) and np.array_equal(many["candidate"], pc["candidate"])


def test_gather_psms_single_rank_and_device_pointers(gpu):
    """md_gather_psms without a communicator is a copy -- host to host, and in place on device pointers (the buffer
    md_identify_device wrote is the send buffer)."""
    import ctypes as C
    import torch
    from maxdecoy import _abi, parallel
    prots = list(wl.proteins(150))
    gpu.digest(prots, 2, 5, 50)
    gpu.set_modifications([synth.CAM], 0)
    gpu.index_build()
    sp, _ = wl.spectra(150, 40, 2)
    prm = SearchParams(10, 10, n_decoys=30, seed=9, top_k=3)
    gpu.comm_init(0, 1, None)
    want, _ = gpu.identify(sp, prm)
    got, _ = parallel.identify_sharded_comm(gpu, sp, prm, 0, 1, block=8)
    assert got.tobytes() == want.tobytes()
    dev = {k: torch.from_numpy(getattr(sp, k).view(np.int64) if getattr(sp, k).dtype == np.uint64 else getattr(sp, k)).cuda()
           for k in ("precursor_mz", "charge", "peak_off", "peak_mz", "peak_intensity")}
    sd = _abi.md_spectra()
    sd.n = len(sp)
    for k, v in dev.items():
        setattr(sd, k, v.data_ptr())
    rows = torch.zeros(len(sp) * 3 * 56, dtype=torch.uint8, device="cuda")
    allr = torch.zeros_like(rows)
    gpu.identify_device(sd, prm, rows.data_ptr())
    gpu.gather_psms_device(rows.data_ptr(), len(sp) * 3, allr.data_ptr())
    gpu.sync()
    assert allr.cpu().numpy().tobytes() == want.tobytes()
    gpu.comm_destroy()


def test_decoy_selection_is_exact_when_hashes_collide(cpu):
    """k_decoy_select finds duplicates through a hash set; a success whose hash is already carried by a different sequence
    must still be kept.  A test build of the library that keeps only 6 bits of the hashes makes such collisions the rule:
    its decoys must still equal the oracle's (which compares strings)."""
    import testbuild
    g = testbuild.engine(["-DMD_SELECT_HASH_MASK=0x3Full"])
    try:
        prots = list(wl.proteins(300))
        for e in (g, cpu):
            e.digest(prots, 2, 5, 50)
            e.set_modifications([synth.CAM], 0)
            e.index_build()
        sp, _ = wl.spectra(300, 24, 2)
        pre = wl.precursors_of(g, sp)
        dg = g.generate_decoys(pre, 200, seed=11)
        dc = cpu.generate_decoys(pre, 200, seed=11)
        assert len(dg["attempt"]) > 3000
        assert_tables_equal(dg, dc)
    finally:
        g.close()
