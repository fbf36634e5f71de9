"""The candidate lookup (K2: window search, fan-out test, placement search, expanded mode, stored-decoy reuse) against the
CPU oracle at its limits.  Every case is built from crafted proteins without K/R inside: digested with no missed
cleavage, each protein is exactly one peptide, so index sizes, equal keys and letter counts are chosen here.  Before a
limit case, a few lines compute on which side of the limit it lies (subset counts, count vectors, placements, K_a)."""
import itertools
import math
import random

import numpy as np
import pytest

import maxdecoy
from maxdecoy import MaxDecoyError, Modification, SearchParams, synth
from oracle_lib import oracle_engine
import pyref

pytestmark = pytest.mark.gpu

I64_MIN, I64_MAX = -2 ** 63, 2 ** 63 - 1
UNSUPPORTED = -5
REF, EXP = maxdecoy.VARMOD_REFERENCE, maxdecoy.VARMOD_EXPANDED

CAM, OXM = synth.CAM, synth.OXM
PHOS_S = Modification("unimod:21", "Phospho", "A", False, "S", 79.966331)
PHOS_T = Modification("unimod:21", "Phospho", "A", False, "T", 79.966331)
PHOS_Y = Modification("unimod:21", "Phospho", "A", False, "Y", 79.966331)
METH_T = Modification("unimod:34", "Methyl", "A", False, "T", 14.01565)
NEG_T = Modification("x:1", "Tminus", "A", False, "T", -79.966331)          # cancels one phospho-S exactly
DEAM_N = Modification("unimod:7", "Deamidated", "A", False, "N", 0.984016)
DEAM_Q = Modification("unimod:7", "Deamidated", "A", False, "Q", 0.984016)
PYRO_Q = Modification("unimod:28", "Gln->pyro-Glu", "N", False, "Q", -17.026549)
ACET_S = Modification("unimod:1", "Acetyl", "N", False, "S", 42.010565)     # variable, N-terminal S only
FIX_S = Modification("x:2", "Sfix", "A", True, "S", 0.984016)               # holds the slot of PHOS_S
VAR_C = Modification("x:3", "Cvar", "A", False, "C", 0.984016)              # its slot holds CAM
OX_W = Modification("unimod:35", "Oxidation", "A", False, "W", 15.994915)
SIX = (OXM, DEAM_N, DEAM_Q, PHOS_S, PHOS_T, PHOS_Y)                         # six variable letters


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


def _load(engines, proteins, mods, nvar, mode=REF):
    """Digest (no missed cleavage, lengths 1..60), set the modifications and the mode, build the index.  Returns the
    peptide sequences in canonical order (peptide id - 1)."""
    seqs = []
    for e in engines:
        e.set_decoy_store([])
        n = e.digest(list(proteins), 0, 1, 60)
        assert n == len(set(proteins))
        e.set_modifications(list(mods), nvar)
        e.set_variable_mode(mode)
        e.index_build()
        seqs.append(e.sequences_of(e.peptides()))
    assert all(s == seqs[0] for s in seqs)
    return seqs[0]


def _merged(mods):
    d = {m.amino_acid: m.mono_mass_int for m in mods if m.is_fix}
    d.update({m.amino_acid: m.mono_mass_int for m in mods if not m.is_fix})   # variable overrides fixed
    return d


def _wstar(e, seq, mods):
    """Index key: weight + sum over the modifiable letters of count * merged delta."""
    return e.get_sequence_weight(seq) + sum(seq.count(a) * d for a, d in _merged(mods).items())


def _wfix(e, seq, mods):
    assert all(m.position == "A" for m in mods if m.is_fix)
    return e.get_sequence_weight(seq) + sum(seq.count(m.amino_acid) * m.mono_mass_int for m in mods if m.is_fix)


def _letter_mass(e, mods, a):
    """m'_a: the divisor of K_a = P / m'_a."""
    return e.residue_mass(a) + _merged(mods)[a]


def _same_candidates(gpu, cpu, pre):
    cg, cc = gpu.candidates(pre), cpu.candidates(pre)
    for k in cc:
        assert cg[k].shape == cc[k].shape and np.array_equal(cg[k], cc[k]), k
    return cc


def _rows(c, s):
    a, b = int(c["off"][s]), int(c["off"][s + 1])
    return list(zip(c["peptide_id"][a:b].tolist(), c["var_mask"][a:b].tolist(), c["mod_weight"][a:b].tolist()))


def _refused(fn, *args):
    with pytest.raises(MaxDecoyError) as ei:
        fn(*args)
    assert ei.value.status == UNSUPPORTED


def _perms(comp, n, seed=1):
    """n distinct orders of one composition (one key), sorted."""
    assert math.factorial(len(comp)) >= n
    rng, s, out = random.Random(seed), list(comp), set()
    while len(out) < n:
        rng.shuffle(s)
        out.add("".join(s))
    return sorted(out)


def _spectra(masses, z=2, seed=0):
    """One spectrum per precursor mass (uDa), 16 peaks each."""
    rng = np.random.default_rng(seed)
    pmz = np.array([(m / 1e6 + pyref.PROTON * z) / z for m in masses])
    mz = [np.sort(rng.uniform(100.0, max(200.0, m / 1e6), 16)) for m in masses]
    off = np.concatenate([[0], np.cumsum([len(x) for x in mz])]).astype(np.uint64)
    return maxdecoy.Spectra(pmz, np.full(len(masses), z, dtype=np.uint8), off, np.concatenate(mz) if mz else np.zeros(0),
                            rng.lognormal(4.0, 1.0, int(off[-1])).astype(np.float32))


def _identify_equal(gpu, cpu, sp, prm):
    pg, stg, scg, offg = gpu.identify(sp, prm, want_all_scores=True)
    pc, stc, scc, offc = cpu.identify(sp, prm, want_all_scores=True)
    assert np.array_equal(offg, offc) and np.array_equal(scg, scc)
    for k in pg.dtype.names:
        if k != "_pad":
            assert np.array_equal(pg[k], pc[k]), k
    assert stg["n_targets"] == stc["n_targets"]
    return pg, stg


# ------------------------------------------------------------------------------------------------------------------
# 1. window search: k_window_search's 32-ary warp search (one level below 1025 entries, three at 32769)
# ------------------------------------------------------------------------------------------------------------------
LIGHT = "GASTVDENQ"   # 4-residue fillers, at most 534 Da
HEAVY = "EMHFYW"      # 8-residue fillers, at least 1050 Da
RUN = "GGAASSTTVV"    # 848 Da between them; 113400 distinct orders share one key


def _sized_index(n, run):
    """n proteins; entries [b, e) of the index are distinct orders of RUN, the lighter ones come before, heavier after."""
    b, e = run if run else (n, n)
    light = ["".join(t) for t in itertools.islice(itertools.product(LIGHT, repeat=4), b)]
    heavy = ["".join(t) for t in itertools.islice(itertools.product(HEAVY, repeat=8), n - e)]
    return light + _perms(RUN, e - b) + heavy


def _window_runs(n):
    """Runs of equal keys that start and end one before, on and one after a probe position of the first level
    (probes at (lane + 1) * stride - 1, stride = ceil(n / 32)), plus runs at either end of the index."""
    if n < 1000:
        return [None] + ([(0, n)] if n >= 33 else [])
    s = -(-n // 32)
    if n > 32 * 1024:
        return [(s - 2, 2 * s), (s - 1, 2 * s - 2), (s, 2 * s - 1)]
    p1, p3 = s - 1, 3 * s - 1
    return [(b, e) for b in (p1 - 1, p1, p1 + 1) for e in (p3 - 1, p3, p3 + 1)] + [(0, 40), (n - 40, n)]


def _windows(keys):
    u = np.unique(keys).tolist()
    w = []
    for k in u:
        w += [(k, k), (k - 1, k - 1), (k + 1, k + 1), (k + 1, k), (k, k - 1)]
    mn, mx = (u[0], u[-1]) if u else (0, 0)
    w += [(mn - 1, mn - 1), (mx + 1, mx + 1), (I64_MIN, I64_MAX), (I64_MIN, I64_MIN), (I64_MAX, I64_MAX), (I64_MIN, mn - 1),
          (mx + 1, I64_MAX), (mx, mn - 1), (mn, mx), (0, -1), (1, 0), (I64_MAX, I64_MIN)]
    return np.array([a for a, _ in w], dtype=np.int64), np.array([b for _, b in w], dtype=np.int64)


@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 1023, 1024, 1025, 32769])
def test_window_search(gpu, cpu, n):
    """(begin, end) of every key, its neighbours, empty and reversed windows and the int64 extremes, against the oracle and
    np.searchsorted on the exported keys."""
    if n > 32 * 1024:
        assert -(-n // 32) == 1025       # first stride 1025 leaves 1024 entries: a second level of stride 32, then the scan
    for run in _window_runs(n):
        _load((gpu, cpu), _sized_index(n, run), (CAM, OXM), 2)
        assert gpu.index_stats()["n_peptides"] == cpu.index_stats()["n_peptides"] == n
        pg, kg = gpu.index_export(0, n)
        pc, kc = cpu.index_export(0, n)
        assert np.array_equal(kg, kc) and np.array_equal(pg, pc)
        if run:
            b, e = run
            assert e - b >= 33 and np.all(kg[b:e] == kg[b]) and (b == 0 or kg[b - 1] < kg[b]) and (e == n or kg[e] > kg[b])
        lo, hi = _windows(kg)
        bg, eg = gpu.window_search(lo, hi)
        bc, ec = cpu.window_search(lo, hi)
        assert np.array_equal(bg, bc) and np.array_equal(eg, ec)
        want_b = np.searchsorted(kg, lo, "left")
        want_e = np.maximum(np.searchsorted(kg, hi, "right"), want_b)
        assert np.array_equal(bg, want_b) and np.array_equal(eg, want_e)


# ------------------------------------------------------------------------------------------------------------------
# 2. the fan-out test of k_filter: count_a < K_a = P / m'_a, and cur_lo > 0 at every level
# ------------------------------------------------------------------------------------------------------------------
def test_fanout_count_limit(gpu, cpu):
    """A run of c methionines: P = c*m'-1, c*m', (c+1)*m'-1, (c+1)*m'.  K = c drops the peptide, K = c + 1 keeps it.
    The window is the single point W*, which the placement search reaches with all c residues oxidised."""
    mods = (CAM, OXM)
    seqs = _load((gpu, cpu), ["M" * c + "G" for c in range(1, 7)], mods, 8)
    mp, mc = _letter_mass(cpu, mods, "M"), _letter_mass(cpu, mods, "C")
    pre, want = [], []
    for c in range(1, 7):
        q = "M" * c + "G"
        w = _wstar(cpu, q, mods)
        for P, K in ((c * mp - 1, c - 1), (c * mp, c), ((c + 1) * mp - 1, c), ((c + 1) * mp, c + 1)):
            assert P // mp == K
            keep = K > c
            assert not keep or P // mc >= 1          # K_C > count_C = 0
            pre.append((P, w, w, 2, len(pre)))
            want.append([(seqs.index(q) + 1, (1 << c) - 1, w)] if keep else [])
    c = _same_candidates(gpu, cpu, pre)
    assert [_rows(c, s) for s in range(len(pre))] == want


def test_fanout_lower_limit(gpu, cpu):
    """cur_lo > 0: lo = -1, 0, 1, and lo at and one above what the C level subtracts (count_C * CAM) before the M level."""
    mods = (CAM, OXM)
    seqs = _load((gpu, cpu), ["CCMG", "CMMG", "MG", "MMG", "GGG"], mods, 3)
    cam = CAM.mono_mass_int
    hi = _wstar(cpu, "CCMG", mods)
    assert _wstar(cpu, "CMMG", mods) <= hi
    P = 10 ** 10
    assert all(P // _letter_mass(cpu, mods, a) < 2 ** 15 for a in "CM")
    los = [-1, 0, 1, cam - 1, cam, cam + 1, 2 * cam - 1, 2 * cam, 2 * cam + 1, 2 * cam + 2]
    pre = [(P, lo, hi, 2, i) for i, lo in enumerate(los)]
    c = _same_candidates(gpu, cpu, pre)
    for s, lo in enumerate(los):
        got = {pid: (m, w) for pid, m, w in _rows(c, s)}
        for q, n_c in (("CCMG", 2), ("CMMG", 1)):
            keep = lo > 0 and lo - n_c * cam > 0
            pid = seqs.index(q) + 1
            assert (pid in got) == keep, (q, lo)
            if keep:
                assert got[pid] == (0, _wfix(cpu, q, mods))


def test_fanout_negative_delta(gpu, cpu):
    """A variable N-terminal Q -17.03 Da (m'_Q = 111.03 Da): K_Q = c drops Q^c G, K_Q = c + 1 keeps it.  Only the first
    Q can take the modification, so the window [W*, w - 17.03 Da] is reached by the placement of residue 0 alone."""
    mods = (CAM, OXM, PYRO_Q)
    seqs = _load((gpu, cpu), ["Q" * c + "G" for c in range(1, 5)] + ["GQQG"], mods, 3)
    mq = _letter_mass(cpu, mods, "Q")
    assert mq < cpu.residue_mass("Q")
    pre, want = [], []
    for c in range(1, 5):
        q = "Q" * c + "G"
        w, ws = cpu.get_sequence_weight(q), _wstar(cpu, q, mods)
        hit = w + PYRO_Q.mono_mass_int
        assert ws <= hit
        for P, K in ((c * mq - 1, c - 1), (c * mq, c), ((c + 1) * mq - 1, c), ((c + 1) * mq, c + 1)):
            assert P // mq == K
            keep = K > c
            assert not keep or min(P // _letter_mass(cpu, mods, a) for a in "CM") >= 1
            pre.append((P, ws, hit, 2, len(pre)))
            want.append((seqs.index(q) + 1, 1, hit) if keep else None)
    c = _same_candidates(gpu, cpu, pre)
    for s, row in enumerate(want):
        pids = {r[0]: r for r in _rows(c, s)}
        pid = seqs.index("Q" * (s // 4 + 1) + "G") + 1
        assert pids.get(pid) == row


def test_no_modifications_no_candidates(gpu, cpu):
    """No modifiable letter: the recursion emits no query, so reference mode finds nothing, on either side."""
    _load((gpu, cpu), ["GASG", "MMG", "CCG", "SSTG"], (), 0)
    pre = [(10 ** 10, 1, 10 ** 10, 2, 0), (10 ** 9, 1, 10 ** 9, 2, 1)]
    c = _same_candidates(gpu, cpu, pre)
    assert c["off"].tolist() == [0, 0, 0]


# ------------------------------------------------------------------------------------------------------------------
# 3. the placement search (md_try_variable): the one-letter shortcut and the generic NChooseK enumeration
# ------------------------------------------------------------------------------------------------------------------
PLACEMENT_SETS = {
    # one variable letter, no fixed modification on it, no terminal modification: var_simple_code
    "simple": ((CAM, PHOS_S), ["SAGSVGSAG", "CSGSSA", "GAVG"]),
    # the variable letter also fixed: its slot is taken, no placement changes the weight
    "fixed_and_variable": ((CAM, FIX_S, PHOS_S), ["SAGSVGSAG", "CSGSSA"]),
    # two variable letters with different deltas
    "two_deltas": ((CAM, PHOS_S, METH_T), ["STGSTGA", "TSAVT", "SGSSTG"]),
    # deltas that cancel: several placements share a weight, the first in NChooseK order wins
    "opposite_deltas": ((CAM, PHOS_S, NEG_T), ["SSTG", "STSTG", "TSSG"]),
    # a terminal variable letter that also sits away from the terminus: eligible positions != letter positions
    "terminal": ((CAM, ACET_S), ["SGSGSA", "GSSGSA", "SSSG"]),
}


def _placement_weights(pm, q):
    """Weight of every subset of the variable-letter positions of q, modified the reference's way (slots)."""
    pos = [i for i, ch in enumerate(q) if ch in pm.var]
    out = set()
    for n in range(len(pos) + 1):
        for sub in itertools.combinations(pos, n):
            sp = pyref.SlotPeptide(pm, q)
            for i in sub:
                sp.set_variable(i)
            out.add(sp.w)
    return len(pos), sorted(out)


@pytest.mark.parametrize("name", sorted(PLACEMENT_SETS))
def test_placement_search(gpu, cpu, name):
    """nvar = 0, 1, d-1, d, d+1 (d: variable-letter residues).  Windows: the single point W*, [X, X] and the span of X and
    W* for every placement weight X, and (wfix, W*] without the unmodified weight.  Against the oracle and, peptide by
    peptide, against the literal fan-out + filter of pyref."""
    mods, prots = PLACEMENT_SETS[name]
    pm0 = pyref.Mods(mods, 0)
    ds = {_placement_weights(pm0, q)[0] for q in prots} - {0}
    for nvar in sorted({0, 1} | {x for d in ds for x in (d - 1, d, d + 1)}):
        seqs = _load((gpu, cpu), prots, mods, nvar)
        pm = pyref.Mods(mods, nvar)
        table = cpu.peptides()
        peptides = [(q, int(table["weight"][i]), pyref.counts21(q)) for i, q in enumerate(seqs)]
        P = max((q.count(a) + 1) * _letter_mass(cpu, mods, a) for q in seqs for a in pm.letters) + 1_000_000   # every K_a > count_a
        wins = set()
        for q in seqs:
            ws = _wstar(cpu, q, mods)
            w0 = pyref.SlotPeptide(pm, q).w
            wins |= {(ws, ws), (w0 + 1, ws), (w0 + 1, max(ws, w0 + 1))}
            for x in _placement_weights(pm, q)[1]:
                wins |= {(x, x), (min(x, ws), max(x, ws))}
        pre = [(P, lo, hi, 2, i) for i, (lo, hi) in enumerate(sorted(wins))]
        c = _same_candidates(gpu, cpu, pre)
        for s, (_, lo, hi, _, _) in enumerate(pre):
            want = pyref.candidates_sql(pm, peptides, P, lo, hi)
            got = {pid - 1: (w, m) for pid, m, w in _rows(c, s)}
            assert got == want, (nvar, lo, hi)
        assert c["off"][-1] > 0


def test_lean_path_through_identify(gpu, cpu):
    """nvar = 0 with a variable modification configured: no per-entry mask / weight is written (the lean path), through
    md_candidates and md_identify."""
    mods, prots = PLACEMENT_SETS["two_deltas"]
    prots = prots + ["".join(t) for t in itertools.islice(itertools.product("GASTV", repeat=5), 400)]
    _load((gpu, cpu), prots, mods, 0)
    _, kg = gpu.index_export(0, len(set(prots)))
    masses = [int(k) for k in np.unique(kg)[::3]]
    sp = _spectra(masses)
    pre = [cpu.precursor_window(float(sp.precursor_mz[i]), 2, 10, 10) + (2, i) for i in range(len(sp))]
    c = _same_candidates(gpu, cpu, pre)
    assert c["off"][-1] > 0 and not np.any(c["var_mask"])
    pg, st = _identify_equal(gpu, cpu, sp, SearchParams(10, 10, n_decoys=3, seed=2, top_k=2))
    assert np.array_equal(pg[:, 0]["n_targets"], np.diff(c["off"].astype(np.int64)))


# ------------------------------------------------------------------------------------------------------------------
# 4. the enumeration cap of md_try_variable: 2^22 subsets per peptide
# ------------------------------------------------------------------------------------------------------------------
def test_reference_subset_cap(gpu, cpu):
    """S x20 T x20 K with phospho on S and T (the generic route), window at W* (all 40 residues modified): no subset of at
    most nvar residues reaches it, so every subset is tried.  nvar = 5 stays under the cap and equals the oracle;
    nvar = 6 goes over it and is refused through md_candidates and md_identify (the oracle, without a cap, answers)."""
    q = "S" * 20 + "T" * 20 + "K"
    mods = (PHOS_S, PHOS_T)
    d = 40

    def subsets(nvar):
        return sum(math.comb(d, n) for n in range(1, nvar + 1))
    assert subsets(5) == 760098 < 2 ** 22 < subsets(6) == 4598478
    _load((gpu, cpu), [q], mods, 5)
    ws = _wstar(cpu, q, mods)
    P = 2 * ws
    assert min(P // _letter_mass(cpu, mods, a) for a in "ST") > 20
    pre = [(P, ws, ws, 2, 0)]
    assert _same_candidates(gpu, cpu, pre)["off"].tolist() == [0, 0]
    for e in (gpu, cpu):
        e.set_modifications(list(mods), 6)
        e.index_build()
    assert cpu.candidates(pre)["off"].tolist() == [0, 0]
    _refused(gpu.candidates, pre)
    sp = _spectra([ws])
    _, lo, hi = gpu.precursor_window(float(sp.precursor_mz[0]), 2, 10, 10)
    assert lo <= ws <= hi and hi < ws + PHOS_S.mono_mass_int
    _refused(gpu.identify, sp, SearchParams(10, 10, n_decoys=0, top_k=1))


# ------------------------------------------------------------------------------------------------------------------
# 5. expanded mode: 6 letters, 96 count vectors, 2^20 - 1 placements per (window, peptide)
# ------------------------------------------------------------------------------------------------------------------
EXPANDED_PEPTIDES = ["SSSSG", "SMSMG", "MNQSTYG", "YTSQNMG", "SSTTYYG", "CSMQG", "NQNQWG", "GAVG", "WMSG"]


def _expanded_letters(mods):
    fix = {m.amino_acid: m.position for m in mods if m.is_fix}
    return sorted({m.amino_acid for m in mods if not m.is_fix and fix.get(m.amino_acid) != m.position})


def _expanded_windows(e, seqs, mods, nvar, P_factor=3):
    out = set()
    for q in seqs:
        w = _wfix(e, q, mods)
        out |= {(w, w), (w - 40_000_000, w + 250_000_000), (_wstar(e, q, mods),) * 2}
    return [(P_factor * max(hi, 1), lo, hi, 2, i) for i, (lo, hi) in enumerate(sorted(out))]


@pytest.mark.parametrize("mods,nvar", [((PHOS_S,), 95), ((PHOS_S,), 96), ((PHOS_S, OXM), 12), ((PHOS_S, OXM), 13), (SIX, 3),
                                       (SIX + (CAM, VAR_C), 3), (SIX + (OX_W,), 3)],
                         ids=["1-letter-96", "1-letter-97", "2-letters-91", "2-letters-105", "6-letters-84", "6-letters-plus-held-slot",
                              "7-letters"])
def test_expanded_count_vectors(gpu, cpu, mods, nvar):
    """Count vectors over L letters with sum <= nvar: C(nvar + L, L).  96 are accepted, 97 refused; six letters accepted, a
    seventh refused; a letter whose fixed modification holds the variable slot is not a letter."""
    L = len(_expanded_letters(mods))
    vectors = math.comb(nvar + L, L)
    accepted = L <= 6 and vectors <= 96
    assert (L, vectors) in {(1, 96), (1, 97), (2, 91), (2, 105), (6, 84), (7, 120)}
    seqs = _load((gpu, cpu), EXPANDED_PEPTIDES, mods, nvar, EXP)
    pre = _expanded_windows(cpu, seqs, mods, nvar)
    if accepted:
        c = _same_candidates(gpu, cpu, pre)
        assert c["off"][-1] > 0
    else:
        _refused(gpu.candidates, pre)


@pytest.mark.parametrize("n_s", [22, 23])
def test_expanded_placement_cap(gpu, cpu, n_s):
    """S x n K, nvar = 11, window at 11 phospho deltas: C(22, 11) = 705432 placements of one peptide are accepted and equal
    the oracle's; C(23, 11) = 1352078 exceed 2^20 - 1 and are refused."""
    q = "S" * n_s + "K"
    placements = math.comb(n_s, 11)
    accepted = placements <= 2 ** 20 - 1
    assert (placements, accepted) in {(705432, True), (1352078, False)}
    _load((gpu, cpu), [q], (PHOS_S,), 11, EXP)
    w = _wfix(cpu, q, ()) + 11 * PHOS_S.mono_mass_int
    pre = [(2 * w, w, w, 2, 0)]
    if accepted:
        c = _same_candidates(gpu, cpu, pre)
        assert c["off"].tolist() == [0, placements]
        assert len(np.unique(c["var_mask"])) == placements and np.all(c["mod_weight"] == w)
    else:
        _refused(gpu.candidates, pre)


def test_expanded_terminal_and_held_slot(gpu, cpu):
    """Three variable letters (M, Q at the N-terminus, S) and C, whose CAM holds the variable slot: the odometer runs over
    three letters, Q placements exist only on residue 0, and peptides of equal fixed weight come out in index order."""
    mods = (CAM, VAR_C, OXM, PYRO_Q, PHOS_S)
    assert _expanded_letters(mods) == ["M", "Q", "S"]
    prots = _perms("QSMSMQG", 12) + ["CQSMG", "QCSSMMG", "SQMSG"]
    seqs = _load((gpu, cpu), prots, mods, 3, EXP)
    wf = [_wfix(cpu, q, mods) for q in seqs]
    assert max(wf.count(x) for x in wf) >= 12                   # equal fixed weights
    pre = _expanded_windows(cpu, seqs, mods, 3)
    deltas = {"M": OXM.mono_mass_int, "Q": PYRO_Q.mono_mass_int, "S": PHOS_S.mono_mass_int}
    for q in seqs:                                              # single points at placements across the three letters
        for combo in itertools.product(range(3), repeat=3):
            if sum(combo) <= 3:
                x = _wfix(cpu, q, mods) + sum(k * deltas[a] for k, a in zip(combo, "MQS"))
                pre.append((3 * x, x, x, 2, len(pre)))
    c = _same_candidates(gpu, cpu, pre)
    rows = [(seqs[p - 1], m) for p, m in zip(c["peptide_id"].tolist(), c["var_mask"].tolist())]
    assert any({q[i] for i in range(len(q)) if m >> i & 1} == {"M", "Q", "S"} for q, m in rows)
    assert not any(q[i] == "Q" and m >> i & 1 for q, m in rows for i in range(1, len(q)))    # Q only at residue 0
    assert not any(q[i] == "C" and m >> i & 1 for q, m in rows for i in range(len(q)))


# ------------------------------------------------------------------------------------------------------------------
# 6. batch shape: runs of empty windows, one window over the whole index, passes
# ------------------------------------------------------------------------------------------------------------------
def _batch_masses(hits, n):
    """n precursor masses: empty windows (above the index) first, last and between hits."""
    empty = [2_000_000_000 + 1_000_000 * i for i in range(n)]
    if n == 1:
        return [hits[len(hits) // 2]]
    if n == 5:
        return [empty[0], empty[1], hits[3], hits[-1], empty[2]]
    out = empty[: n // 4]
    mid = []
    for i in range(n // 2):
        mid.append(hits[i % len(hits)] if i % 3 == 0 else empty[n // 4 + i])
    return out + mid + empty[len(out) + len(mid): n]


@pytest.mark.parametrize("n", [1, 5, 1200])
@pytest.mark.parametrize("mode,nvar", [(REF, 2), (REF, 0), (EXP, 2)], ids=["reference", "reference-lean", "expanded"])
def test_batch_shape(gpu, cpu, n, mode, nvar, monkeypatch):
    """md_candidates against the oracle for batches of 1, 5 and 1200 precursors with long runs of empty windows, plus
    an absolute window over the whole index; md_identify's n_targets per spectrum equals the md_candidates offsets, in
    one pass and in passes of 3 spectra."""
    mods = (CAM, OXM, PHOS_S)
    prots = ["".join(t) for t in itertools.islice(itertools.product("GASVMC", repeat=4), 500)]
    _load((gpu, cpu), prots, mods, nvar, mode)
    _, kg = gpu.index_export(0, len(prots))
    keys = np.unique(kg)
    assert keys[-1] < 2_000_000_000
    # G/A/V only: no modifiable letter, so W* = wfix and such a window has a candidate in every mode
    plain = sorted({_wstar(cpu, q, mods) for q in prots if not set(q) - set("GAV")})
    sp = _spectra(_batch_masses(plain if n <= 5 else [int(k) for k in keys], n))
    assert len(sp) == n
    pre = [cpu.precursor_window(float(sp.precursor_mz[i]), 2, 10, 10) + (2, i) for i in range(n)]
    assert pre == [gpu.precursor_window(float(sp.precursor_mz[i]), 2, 10, 10) + (2, i) for i in range(n)]
    whole = [(int(keys[-1]) * 3, 1, int(keys[-1]) + 10 ** 9, 2, n)]
    c = _same_candidates(gpu, cpu, pre + whole)
    nt = np.diff(c["off"].astype(np.int64))
    assert nt[-1] > 0 and (n == 1 or np.count_nonzero(nt[:-1] == 0) >= n // 2)
    assert nt[:-1].sum() > 0
    prm = SearchParams(10, 10, n_decoys=1, seed=4, top_k=1)
    pg, st = _identify_equal(gpu, cpu, sp, prm)
    assert np.array_equal(pg[:, 0]["n_targets"], nt[:-1]) and st["n_targets"] == nt[:-1].sum()
    monkeypatch.setenv("MD_MAX_PASS_SPECTRA", "3")
    p3, st3 = gpu.identify(sp, prm)
    assert np.array_equal(p3[:, 0]["n_targets"], nt[:-1]) and st3["n_targets"] == st["n_targets"]
    for k in pg.dtype.names:
        if k != "_pad":
            assert np.array_equal(p3[k], pg[k]), k


# ------------------------------------------------------------------------------------------------------------------
# 7. stored-decoy reuse: only the first n_per accepted store entries of a window are kept
# ------------------------------------------------------------------------------------------------------------------
def test_stored_decoys_beyond_n_per(gpu, cpu):
    """Nine store entries of one key that need both of their phospho-S placed, and five of another that need none; n_per
    from 1 to past both counts.  The generate_decoys tables equal the oracle's and take min(n_per, accepted) stored ones."""
    mods = (CAM, PHOS_S)
    _load((gpu, cpu), ["".join(t) for t in itertools.islice(itertools.product("GAVDE", repeat=5), 200)], mods, 2)
    with_s, without_s = _perms("SSAGVDE", 9), _perms("AGVDNEY", 5)
    w1, w2 = _wstar(cpu, with_s[0], mods), _wstar(cpu, without_s[0], mods)
    assert _wfix(cpu, with_s[0], mods) == w1 - 2 * PHOS_S.mono_mass_int
    pre = [(w1, w1 - 10_000, w1 + 10_000, 2, 0), (w2, w2 - 10_000, w2 + 10_000, 2, 1)]
    assert all(P // _letter_mass(cpu, mods, a) > 2 for P, *_ in pre for a in "CS")     # K_S > count_S, K_C > 0
    accepted = (9, 5)
    try:
        for e in (gpu, cpu):
            e.set_decoy_store(with_s + without_s)
        for n_per in (1, 4, 5, 6, 8, 9, 10):
            dg = gpu.generate_decoys(pre, n_per, maxdecoy.DECOY_REFERENCE_RANDOM, seed=3)
            dc = cpu.generate_decoys(pre, n_per, maxdecoy.DECOY_REFERENCE_RANDOM, seed=3)
            for k in dc:
                assert dg[k].shape == dc[k].shape and np.array_equal(dg[k], dc[k]), (n_per, k)
            for s in range(2):
                a, b = int(dg["off"][s]), int(dg["off"][s + 1])
                stored = dg["attempt"][a:b] == maxdecoy.DECOY_STORED
                assert stored.sum() == min(n_per, accepted[s])
                assert s == 1 or np.all(dg["var_mask"][a:b][stored] != 0)
    finally:
        for e in (gpu, cpu):
            e.set_decoy_store([])
