"""Fragment scoring (K4), GPU against the CPU oracle, bit for bit: raw scores of every candidate and every PSM field.

score.cu picks its code path from the size of each spectrum's table (bin(m/z) = floor(m/z[uDa] / w) + 1, NB = hbin + 76 bins,
nblk = ceil(NB / 64) block-map entries, nact occupied 64-bin blocks, npk binned peaks):
- k_build_tables + k_score_pipe (top_k <= 8): a spectrum with more than 1024 binned peaks, more than 4096 map entries or a
  table record (map + all-zero block + occupied blocks) above the 214-KB ring goes onto a list that k_score works off
  beside the pipe; two records that do not fit the ring together make the loader wait for the ring to drain.
- k_score (MD_SCORE_CLASSIC=1, top_k > 8, the left list): up to 512 peaks and 6144 map entries are staged by the prefetch
  warp, more are built by the whole CTA, and above 6144 entries the block map lives in HBM; up to 719 occupied blocks make
  one tile, more make several, and the running sum enters a later tile through sh.cin.
- 1536-candidate chunks and 2048 length-sorted candidates; top_k <= 8 keeps per-warp lists, larger top_k a block-wide merge;
  fragment charges 1..min(max(z-1, 1), 3, max_fragment_charge) pick one of three scoring templates.

The boundary cases build spectra on a chosen side of each limit.  `geometry` restates how k_build_tables (marks bins
[b-75, b+75]) and k_score (marks [b-75, b+76]) count a spectrum, each case asserts the values it intends, and the engine's
statistics (n_score_left, score_pipelined) show which kernel ran.

The oracle accepts max_fragment_charge 4, tables above 2^26 bins and residue masses of 2^22 bins or more; the CUDA library
refuses all three with MD_ERR_UNSUPPORTED."""
import re

import numpy as np
import pytest

import maxdecoy
from maxdecoy import Modification, SearchParams, synth
from oracle_lib import oracle_engine
import workloads as wl

pytestmark = pytest.mark.gpu

RANDOM = maxdecoy.DECOY_REFERENCE_RANDOM
PROTON, WATER = 1_007_276, 18_010_565                      # uDa
XC, BLK = 75, 64
P_PEAKS, P_MAP, RING, POOL = 1024, 4096, 214 * 1024, 856   # k_build_tables / k_score_pipe
PEAK_CAP, MAP_CAP, TILE = 512, 6144, 719                   # k_score
MAX_BINS = 1 << 26
FIX = {"C": synth.CAM.mono_mass_int}
VAR = {"M": synth.OXM.mono_mass_int}
WAYS = ("default", "classic", "top_k_9")
TRACE_RE = re.compile(r"occupied blocks p10=\d+ p50=\d+ p90=\d+ p99=\d+ max=(\d+)")


@pytest.fixture(scope="module")
def gpu():
    with pytest.MonkeyPatch.context() as mp:       # MD_TRACE is read when the engine is created
        mp.setenv("MD_TRACE", "1")
        e = maxdecoy.Engine()
    assert e.backend == "cuda-sm100a"
    yield e
    e.close()


@pytest.fixture(scope="module")
def cpu():
    e = oracle_engine(8)
    yield e
    e.close()


def _setup(engines, mods=(synth.CAM, synth.OXM), nvar=3):
    for e in engines:
        e.digest(list(wl.proteins(600)), 2, 5, 50)
        e.set_modifications(list(mods), nvar)
        e.index_build()


def _way(way, monkeypatch, top_k=5):
    """The three ways of running a case: the pipelined path, k_score forced, and top_k > 8 (k_score with the block-wide merge)."""
    if way == "classic":
        monkeypatch.setenv("MD_SCORE_CLASSIC", "1")
    return 9 if way == "top_k_9" else top_k


def check(g, cpu, sp, prm, way=None):
    """GPU against the oracle: per-candidate raw scores, every PSM field but _pad, and the same rows without all scores."""
    pg, stg, scg, offg = g.identify(sp, prm, want_all_scores=True)
    pc, stc, scc, offc = cpu.identify(sp, prm, want_all_scores=True)
    assert np.array_equal(offg, offc)
    assert np.array_equal(scg, scc)
    for k in pg.dtype.names:
        if k != "_pad":
            assert np.array_equal(pg[k], pc[k]), k
    assert (stg["n_targets"], stg["n_decoys"]) == (stc["n_targets"], stc["n_decoys"])
    pg2, _ = g.identify(sp, prm)
    assert pg2.tobytes() == pg.tobytes()
    if way is not None:
        assert stg["score_pipelined"] == (1 if way == "default" else 0)
    return pg, stg, scg, offg


# ------------------------------------------------------------------------------------------------ spectra
def mz_of(u):
    """A double m/z whose (int64)(m/z * 1e6) is exactly u uDa (the conversion both sides apply)."""
    m = u / 1e6
    while int(m * 1e6) < u:
        m = np.nextafter(m, np.inf)
    while int(m * 1e6) > u:
        m = np.nextafter(m, -np.inf)
    assert int(m * 1e6) == u
    return float(m)


def bin_mz(b, w):
    """m/z in the middle of bin b (margin w/2 against rounding)."""
    return mz_of((b - 1) * w + w // 2)


def pmz_of(mass, z):
    return (mass / 1e6 + z * synth.PROTON) / z


class Batch:
    def __init__(self):
        self.pmz, self.z, self.peaks = [], [], []

    def add(self, pmz, z, mz, inten):
        mz, inten = np.asarray(mz, dtype=np.float64), np.asarray(inten, dtype=np.float32)
        o = np.argsort(mz, kind="stable")
        self.pmz.append(float(pmz)); self.z.append(int(z)); self.peaks.append((mz[o], inten[o]))
        return len(self.pmz) - 1

    def add_from(self, sp, i, z=None, pmz=None):
        a, b = int(sp.peak_off[i]), int(sp.peak_off[i + 1])
        return self.add(sp.precursor_mz[i] if pmz is None else pmz, sp.charge[i] if z is None else z, sp.peak_mz[a:b], sp.peak_intensity[a:b])

    def spectra(self):
        off = np.concatenate([[0], np.cumsum([len(m) for m, _ in self.peaks])]).astype(np.uint64)
        cat = lambda j, dt: np.concatenate([p[j] for p in self.peaks]).astype(dt) if self.peaks else np.zeros(0, dt)
        return maxdecoy.Spectra(np.array(self.pmz), np.array(self.z, dtype=np.uint8), off, cat(0, np.float64), cat(1, np.float32))


def normal_spectra():
    sp, _ = wl.spectra(600, 40, 2, with_ox=True)
    return sp


def precursor(cpu, pmz, z, sid):
    P, lo, hi = cpu.precursor_window(pmz, z, 10, 10)
    return (P, lo, hi, z, sid)


def fragments(cpu, pre, n_decoys, seed, nch=2, count=4):
    """Fragment m/z (uDa, charges 1..nch) of the spectrum's first decoys: peaks there give those decoys real scores."""
    t = cpu.generate_decoys([pre], n_decoys, RANDOM, seed=seed)
    out = set()
    for seq, mask, modw in list(zip(wl.decoy_strings(t), t["var_mask"].tolist(), t["mod_weight"].tolist()))[:count]:
        res = [cpu.residue_mass(c) + FIX.get(c, 0) + (VAR.get(c, 0) if (mask >> i) & 1 else 0) for i, c in enumerate(seq)]
        assert sum(res) + WATER == modw
        B = np.cumsum(res)[:-1]
        for c in range(1, nch + 1):
            out.update(int((x + c * PROTON) // c) for x in B.tolist() + (modw - B).tolist())
    return sorted(out)


# ------------------------------------------------------------------------------------------------ geometry restated
def binned(sp, i, P, w, min_peaks=10):
    """k_bin_spectra / bin_spectrum: (sorted unique kept bins, hbin over the usable peaks), or None if not scored."""
    a, b = int(sp.peak_off[i]), int(sp.peak_off[i + 1])
    mz, I = sp.peak_mz[a:b], sp.peak_intensity[a:b]
    with np.errstate(invalid="ignore"):
        ok = (I > 0) & (mz > 0) & (mz < 1e7)
        u = np.where(ok, mz, 0.0) * 1e6
    u = u.astype(np.int64)
    ok &= (u > 0) & (u < P + 50_000_000)
    if ok.sum() == 0 or ok.sum() < min_peaks:
        return None
    bins, raw = u[ok] // w + 1, np.sqrt(I[ok].astype(np.float64))
    return np.unique(bins[raw > 0.05 * raw.max()]), int(bins.max())


def _occupied(bins, NB, nblk, reach):
    cov = np.zeros(nblk + 1, dtype=np.int64)
    if len(bins):
        np.add.at(cov, np.maximum(bins - XC, 0) >> 6, 1)
        np.add.at(cov, (np.minimum(bins + reach, NB - 1) >> 6) + 1, -1)
    return np.flatnonzero(np.cumsum(cov)[:nblk] > 0)


def geometry(kept, hbin):
    """How k_build_tables and k_score size the table of one spectrum."""
    NB = hbin + XC + 1
    nblk = -(-NB // BLK)
    occ_pipe = _occupied(kept, NB, nblk, XC)            # k_build_tables: [b-75, b+75]
    occ = _occupied(kept, NB, nblk, XC + 1)             # k_score: [b-75, b+76]
    record = ((nblk + 1) * 2 + 15) // 16 * 16 + (len(occ_pipe) + 1) * 256
    left = len(kept) > P_PEAKS or nblk > P_MAP or len(occ_pipe) + 1 > POOL or record > RING
    return dict(NB=NB, nblk=nblk, npk=len(kept), nact_pipe=len(occ_pipe), nact=len(occ), record=record, left=left,
                tile_x0=[int(occ[c]) * BLK for c in range(TILE, len(occ), TILE)], bins=kept)


def batch_geometry(cpu, sp, w, min_peaks=10):
    out = []
    for i in range(len(sp)):
        P, _, _ = cpu.precursor_window(float(sp.precursor_mz[i]), int(sp.charge[i]), 10, 10)
        r = binned(sp, i, P, w, min_peaks)
        out.append(None if r is None else geometry(*r))
    return out


def comb(n_blocks, frag_bins=()):
    """Peak bins that occupy exactly blocks 0..n_blocks-1 under both markings: an isolated peak at a bin in
    [64k+11, 64k+51] occupies blocks k-1..k+1 (singles at k = 1, 4, 7, ...), two such peaks in blocks k and k+1 occupy
    k-1..k+2 (the pairs after the singles fill the remainder).  A peak sits on a fragment bin where its range has one."""
    pairs = (n_blocks % 3) and (1 if n_blocks % 3 == 1 else 2)
    singles = (n_blocks - 4 * pairs) // 3
    ks = [1 + 3 * j for j in range(singles)]
    for p in range(pairs):
        k = 3 * singles + 4 * p + 1
        ks += [k, k + 1]
    fb = np.asarray(sorted(frag_bins), dtype=np.int64)
    out = []
    for k in ks:
        j = np.searchsorted(fb, 64 * k + 11)
        out.append(int(fb[j]) if j < len(fb) and fb[j] <= 64 * k + 51 else 64 * k + 32)
    return out


def built(pre_mass, z, w, bins, ghost=None):
    """One spectrum: equal-intensity peaks at `bins` (all kept: yq = 50 * 2^16), optionally a peak far below 5 % of the
    others at bin `ghost` (usable, so it sets hbin, but dropped: it occupies no block)."""
    mz = [bin_mz(b, w) for b in bins]
    inten = [100.0] * len(mz)
    if ghost is not None:
        mz.append(bin_mz(ghost, w)); inten.append(0.01)
    return (pmz_of(pre_mass, z), z, mz, inten)


def frag_bins_below(cpu, pre, w, limit, n_decoys=30, seed=5):
    """Charge-1 fragment bins of the spectrum's first decoy below `limit` (few peaks: the table stays small)."""
    return sorted({u // w + 1 for u in fragments(cpu, pre, n_decoys, seed, nch=1, count=1) if u // w + 1 < limit})


# ------------------------------------------------------------------------------------------------ 1. fragment tolerances
TOLS = [0.0001, 0.00015, 0.001, 0.005, 0.01, 0.0200004, 0.05, 0.1, 0.5, 1.0005, 1.007276, 1.5, 2.0]
_SWEEP = {}


def sweep_batch(cpu):
    """40 synthetic spectra (CAM + variable OXM) and two built for heavy precursors (4.3 and 6.4 kDa) whose peaks lie on
    the fragments of their first decoys, all below 6.66 kDa (the 0.0001-Da table stays below 2^26 bins)."""
    if "sp" not in _SWEEP:
        sp = normal_spectra()
        b = Batch()
        for i in range(len(sp)):
            b.add_from(sp, i)
        for mass, z in ((4_300_100_000, 3), (6_400_300_000, 4)):
            sid = len(b.pmz)
            pre = precursor(cpu, pmz_of(mass, z), z, sid)
            us = fragments(cpu, pre, 30, 5, nch=2)
            assert max(us) < 6_660_000_000 and len(us) > 50
            b.add(pmz_of(mass, z), z, [mz_of(u) for u in us], np.full(len(us), 100.0))
        _SWEEP["sp"] = b.spectra()
    return _SWEEP["sp"]


@pytest.mark.parametrize("way", WAYS)
@pytest.mark.parametrize("tol", TOLS)
def test_fragment_tolerance_sweep(gpu, cpu, tol, way, monkeypatch):
    """0.0001 .. 2 Da, incl. 20.0004 mDa (rounds to 20000 uDa), the proton (rp = 0) and 1.5 / 2 Da (qp = 0: K2 wraps)."""
    _setup((gpu, cpu))
    sp = sweep_batch(cpu)
    prm = SearchParams(10, 10, fragment_tolerance=tol, n_decoys=30, seed=5, top_k=_way(way, monkeypatch))
    pg, st, sc, _ = check(gpu, cpu, sp, prm, way)
    assert np.any(pg["rank"] > 0) and np.any(sc > 0)
    geo = batch_geometry(cpu, sp, int(round(tol * 1e6)))
    n_left = sum(1 for g in geo if g is not None and g["left"])
    if way == "default":
        assert st["n_score_left"] == n_left
    if tol == 0.005:                                            # some spectra beyond 4096 map entries: left to k_score
        assert 0 < n_left < len(sp) and any(g["nblk"] > P_MAP for g in geo if g)
    if tol == 0.0001:                                           # every table beyond 6144 entries: k_score with the map in HBM
        assert all(g["nblk"] > MAP_CAP for g in geo if g) and max(g["NB"] for g in geo if g) <= MAX_BINS
        if way == "default":
            assert st["n_score_left"] == sum(1 for g in geo if g)


@pytest.mark.parametrize("tol", [0.000099, 2.000001])
def test_fragment_tolerance_out_of_range(gpu, cpu, tol):
    _setup((gpu, cpu))
    sp = normal_spectra()
    for e in (gpu, cpu):
        with pytest.raises(maxdecoy.MaxDecoyError) as ei:
            e.identify(sp, SearchParams(10, 10, fragment_tolerance=tol, n_decoys=5))
        assert ei.value.status == -1 and "fragment_tolerance" in str(ei.value)


# ------------------------------------------------------------------------------------------------ 2. charges
def charge_batch():
    """Precursor charges 1, 2, 3, 4 and 6 at unchanged precursor masses."""
    sp = normal_spectra()
    b = Batch()
    for i in range(20):
        z0, z = int(sp.charge[i]), (1, 2, 3, 4, 6)[i % 5]
        b.add_from(sp, i, z=z, pmz=(sp.precursor_mz[i] * z0 - synth.PROTON * z0) / z + synth.PROTON)
    return b.spectra()


@pytest.mark.parametrize("way", WAYS)
@pytest.mark.parametrize("mfc", [1, 2, 3, 0])
def test_precursor_and_fragment_charges(gpu, cpu, mfc, way, monkeypatch):
    """max_fragment_charge 1, 2, 3 and 0 (= 3): the one-, two- and three-charge templates of both kernels."""
    _setup((gpu, cpu))
    sp = charge_batch()
    prm = SearchParams(10, 10, n_decoys=30, seed=7, top_k=_way(way, monkeypatch), max_fragment_charge=mfc)
    pg, _, sc, _ = check(gpu, cpu, sp, prm, way)
    assert set(pg["charge"][:, 0].tolist()) == {1, 2, 3, 4, 6} and np.any(sc > 0)


def test_fragment_charge_4_is_refused(gpu, cpu):
    _setup((gpu, cpu))
    sp = charge_batch()
    prm = SearchParams(10, 10, n_decoys=10, seed=7, max_fragment_charge=4)
    with pytest.raises(maxdecoy.MaxDecoyError) as ei:
        gpu.identify(sp, prm)
    assert ei.value.status == -5
    assert np.any(cpu.identify(sp, prm)[0]["rank"] > 0)


# ------------------------------------------------------------------------------------------------ 3. pipelined-path limits
W2 = 20_000       # 0.02 Da


def _heavy(i):
    P, _, _, z, _ = wl.heavy_precursors()[i]
    return P, z


def _ordinary(sp, cpu, lo_mass, hi_mass):
    for i in range(len(sp)):
        P = cpu.precursor_window(float(sp.precursor_mz[i]), int(sp.charge[i]), 10, 10)[0]
        if lo_mass < P < hi_mass:
            return P, int(sp.charge[i])
    raise AssertionError("no precursor in range")


def pipe_case(cpu, kind, n, sid):
    """(spectrum tuple, what its geometry must show) for one side of one limit of the pipelined path."""
    if kind == "peaks":             # n binned peaks, a small table: fragments plus a comb of every other bin from 100 Da
        P, z = _ordinary(normal_spectra(), cpu, 1_500_000_000, 3_000_000_000)
        fb = set(frag_bins_below(cpu, precursor(cpu, pmz_of(P, z), z, sid), W2, P // W2))
        bins, b = sorted(fb)[: n // 2], 5000
        while len(bins) < n:
            if b not in fb:
                bins.append(b)
            b += 2
        return built(P, z, W2, bins), lambda g: g["npk"] == n and g["nblk"] <= P_MAP and g["record"] <= RING
    if kind == "map":               # the highest usable peak at hbin 262068 (4096 entries) / 262069 (4097): the 5.2-kDa precursor
        P, z = _heavy(4)
        hb = 262_068 + (n - P_MAP)
        fb = frag_bins_below(cpu, precursor(cpu, pmz_of(P, z), z, sid), W2, hb)
        return built(P, z, W2, fb, ghost=hb), lambda g: g["nblk"] == n and g["npk"] <= P_PEAKS and g["record"] <= RING
    # "ring": n occupied blocks under a map of 890 entries: 1792 + (848 + 1) * 256 bytes is exactly the ring
    P, z = _ordinary(normal_spectra(), cpu, 1_300_000_000, 3_000_000_000)
    fb = frag_bins_below(cpu, precursor(cpu, pmz_of(P, z), z, sid), W2, 56_000)
    return (built(P, z, W2, comb(n, fb), ghost=56_850),
            lambda g: g["nact_pipe"] == n and g["nblk"] == 890 and g["record"] == RING + (n - 848) * 256 and g["npk"] <= P_PEAKS)


def _with_normal(cases, n_normal=5):
    sp = normal_spectra()
    b = Batch()
    for c in cases:
        b.add(*c)
    for i in range(n_normal):
        b.add_from(sp, i)
    return b.spectra()


PIPE_CASES = [("peaks", 1024), ("peaks", 1025), ("map", 4096), ("map", 4097), ("ring", 848), ("ring", 849)]


@pytest.mark.parametrize("kind,n", PIPE_CASES)
def test_pipelined_limits(gpu, cpu, kind, n, capfd):
    """Each limit of k_build_tables from both sides: 1024 / 1025 binned peaks, 4096 / 4097 block-map entries, a record of
    exactly the ring's 214 KB / one block more.  The spectrum above a limit is left to k_score (n_score_left = 1)."""
    _setup((gpu, cpu))
    spec, want = pipe_case(cpu, kind, n, 0)
    sp = _with_normal([spec])
    geo = batch_geometry(cpu, sp, W2)
    assert want(geo[0]) and all(not g["left"] for g in geo[1:])
    above = geo[0]["left"]
    assert above == (n in (1025, 4097, 849))
    capfd.readouterr()
    pg, st, sc, off = check(gpu, cpu, sp, SearchParams(10, 10, n_decoys=30, seed=5, top_k=5), "default")
    err = capfd.readouterr().err
    assert st["n_score_left"] == (1 if above else 0)
    assert pg["rank"][0, 0] == 1 and np.any(sc[: int(off[1])] > 0)
    if kind == "ring" and not above:      # the engine's own count of occupied blocks agrees with the restatement
        assert [int(x) for x in TRACE_RE.findall(err)][-1] == max(g["nact_pipe"] for g in geo if not g["left"]) == 848


def test_pipelined_and_left_spectra_in_one_batch(gpu, cpu):
    """Spectra above the limits next to ordinary ones: k_score works the left list off beside k_score_pipe."""
    _setup((gpu, cpu))
    cases = [pipe_case(cpu, k, n, i) for i, (k, n) in enumerate(PIPE_CASES)]
    sp = _with_normal([c for c, _ in cases], 10)
    geo = batch_geometry(cpu, sp, W2)
    assert all(want(g) for (_, want), g in zip(cases, geo))
    _, st, _, _ = check(gpu, cpu, sp, SearchParams(10, 10, n_decoys=30, seed=5, top_k=5), "default")
    assert st["n_score_left"] == 3 == sum(g["left"] for g in geo)


def test_ring_full(gpu, cpu):
    """Every record above half the ring: no two spectra are ever resident together, the loader waits for the ring to drain
    before every record (a supported path)."""
    _setup((gpu, cpu))
    P, z = _ordinary(normal_spectra(), cpu, 1_300_000_000, 3_000_000_000)
    b = Batch()
    for i, n in enumerate((430, 500, 600, 700, 800, 848, 450, 760)):
        fb = frag_bins_below(cpu, precursor(cpu, pmz_of(P, z), z, i), W2, 56_000)
        b.add(*built(P, z, W2, comb(n, fb)))
    sp = b.spectra()
    geo = batch_geometry(cpu, sp, W2)
    assert all(RING // 2 < g["record"] <= RING and not g["left"] for g in geo)
    _, st, sc, _ = check(gpu, cpu, sp, SearchParams(10, 10, n_decoys=30, seed=5, top_k=5), "default")
    assert st["n_score_left"] == 0 and np.any(sc > 0)


# ------------------------------------------------------------------------------------------------ 4. k_score limits
W1 = 10_000       # 0.01 Da


def kscore_case(cpu, kind, n, sid):
    if kind == "peaks":             # 512 peaks staged in shared memory by the prefetch warp, 513 built by the whole CTA
        spec, _ = pipe_case(cpu, "peaks", n, sid)
        return spec, W2, lambda g: g["npk"] == n and g["nblk"] <= MAP_CAP
    if kind == "map":               # 6144 map entries in shared memory / 6145 in HBM: hbin 393140 / 393141 at 0.01 Da, 4.3-kDa precursor
        P, z = _heavy(3)
        hb = 393_140 + (n - MAP_CAP)
        fb = frag_bins_below(cpu, precursor(cpu, pmz_of(P, z), z, sid), W1, hb)
        return built(P, z, W1, fb, ghost=hb), W1, lambda g: g["nblk"] == n and g["npk"] <= PEAK_CAP
    # "tiles": n occupied blocks, 719 = one tile; beyond it, peaks whose windows straddle a tile's first bin (sh.cin)
    P, z = _heavy(2)
    fb = frag_bins_below(cpu, precursor(cpu, pmz_of(P, z), z, sid), W2, 64 * n)
    return (built(P, z, W2, comb(n, fb)), W2,
            lambda g: g["nact"] == n and len(g["tile_x0"]) == -(-n // TILE) - 1
            and all(np.any((g["bins"] - XC < x0) & (g["bins"] + XC >= x0)) for x0 in g["tile_x0"][:2]))


@pytest.mark.parametrize("way", ["classic", "top_k_9"])
@pytest.mark.parametrize("kind,n", [("peaks", 512), ("peaks", 513), ("map", 6144), ("map", 6145), ("tiles", 719), ("tiles", 720),
                                    ("tiles", 2200)])
def test_kscore_limits(gpu, cpu, kind, n, way, monkeypatch):
    """k_score's limits from both sides: 512 / 513 staged peaks, 6144 / 6145 block-map entries (shared memory / HBM),
    719 / 720 occupied blocks (one tile / two) and 2200 (four tiles)."""
    _setup((gpu, cpu))
    spec, w, want = kscore_case(cpu, kind, n, 0)
    sp = _with_normal([spec])
    geo = batch_geometry(cpu, sp, w)
    assert want(geo[0])
    pg, _, sc, off = check(gpu, cpu, sp, SearchParams(10, 10, fragment_tolerance=w / 1e6, n_decoys=30, seed=5, top_k=_way(way, monkeypatch)), way)
    assert pg["rank"][0, 0] == 1 and np.any(sc[: int(off[1])] > 0)


# ------------------------------------------------------------------------------------------------ 5. candidate counts
_COUNT = {}


def count_spectra(cpu):
    """Three ordinary spectra with the same number of targets (one each), so that n_decoys = N - 1 gives N candidates."""
    if "sp" not in _COUNT:
        sp = normal_spectra()
        pre = wl.precursors_of(cpu, sp)
        nt = np.diff(cpu.candidates(pre)["off"].astype(np.int64))
        pick = [i for i in range(len(sp)) if nt[i] == 1 and 2_000_000_000 < pre[i][0] < 4_000_000_000][:3]
        assert len(pick) == 3
        b = Batch()
        for i in pick:
            b.add_from(sp, i)
        _COUNT["sp"] = b.spectra()
    return _COUNT["sp"]


COUNTS = [1, 31, 32, 33, 1536, 1537, 2048, 2049, 3072, 3073]


@pytest.mark.parametrize("top_k", [0, 1, 8, 9, 128])
@pytest.mark.parametrize("n", COUNTS)
def test_candidate_counts(gpu, cpu, n, top_k, monkeypatch):
    """Around a warp (32), a chunk (1536), the sorted order (2048) and two chunks (3072) of candidates; top_k 0, within the
    per-warp lists (1, 8), the block-wide merge (9, 128), and beyond N (trailing empty rows)."""
    _setup((gpu, cpu))
    sp = count_spectra(cpu)
    pg, st, _, off = check(gpu, cpu, sp, SearchParams(10, 10, n_decoys=n - 1, seed=3, top_k=top_k))
    assert np.all(np.diff(off.astype(np.int64)) == n)
    if top_k:
        assert np.all(pg["n_targets"] + pg["n_decoys"] == n)
        assert np.array_equal((pg["rank"] > 0).sum(axis=1), np.full(len(sp), min(n, top_k)))


@pytest.mark.parametrize("top_k", [1, 8])
@pytest.mark.parametrize("env", [("MD_SCORE_SPLIT_MIN", "1"), ("MD_SCORE_PARTS", "16")])
def test_candidate_counts_split(gpu, cpu, env, top_k, monkeypatch):
    """3073 candidates per spectrum, each spectrum split into parts over several CTAs."""
    _setup((gpu, cpu))
    monkeypatch.setenv(*env)
    pg, _, _, _ = check(gpu, cpu, count_spectra(cpu), SearchParams(10, 10, n_decoys=3072, seed=3, top_k=top_k), "default")
    assert np.all(pg["n_targets"] + pg["n_decoys"] == 3073)


# ------------------------------------------------------------------------------------------------ 6. ties
def tie_spectra(cpu, kind):
    """zero: peaks only more than 75 bins above every fragment and below P + 50 Da (every score 0);
    comb: equal peaks on every other 0.5-Da bin across the fragment range: T is +75 y on a peak and -76 y between, so a
    score depends on the candidate's length and how many fragments hit a peak (few distinct, mostly negative scores)."""
    src = count_spectra(cpu)
    b = Batch()
    for i in range(len(src)):
        pmz, z = float(src.precursor_mz[i]), int(src.charge[i])
        P = cpu.precursor_window(pmz, z, 10, 10)[0]
        if kind == "zero":
            mz = [mz_of(P + 5_000_000 + 2_000_000 * j) for j in range(20)]
        else:
            mz = [bin_mz(2 * j, 500_000) for j in range(1, (P + 10_000_000) // 1_000_000)]
        b.add(pmz, z, mz, np.full(len(mz), 100.0))
    return b.spectra()


@pytest.mark.parametrize("variant", ["default", "classic", "top_k_9", "split", "split_classic", "parts16"])
@pytest.mark.parametrize("kind", ["zero", "comb"])
def test_score_ties(gpu, cpu, kind, variant, monkeypatch):
    """Ties at the K-th place across warps, units, chunks and parts (3073 candidates): the lower candidate ordinal wins.
    The comb spectra (thousands of peaks) are left to k_score on the pipelined path; split_classic splits them in k_score."""
    _setup((gpu, cpu))
    top_k = _way(variant if variant in WAYS else "default", monkeypatch, 8)
    if variant.startswith("split"):
        monkeypatch.setenv("MD_SCORE_SPLIT_MIN", "1")
    if variant == "split_classic":
        monkeypatch.setenv("MD_SCORE_SPLIT_CLASSIC", "1")
    if variant == "parts16":
        monkeypatch.setenv("MD_SCORE_PARTS", "16")
    sp = tie_spectra(cpu, kind)
    tol = 0.02 if kind == "zero" else 0.5
    pg, _, sc, off = check(gpu, cpu, sp, SearchParams(10, 10, fragment_tolerance=tol, n_decoys=3072, seed=3, top_k=top_k))
    off = off.astype(np.int64)
    kth = [np.sort(sc[a:b])[::-1][top_k - 1] for a, b in zip(off[:-1], off[1:])]
    assert any((sc[a:b] == k).sum() > 1 for a, b, k in zip(off[:-1], off[1:], kth))     # the ordinal decides the K-th row
    if kind == "zero":                  # candidate ordinals 0..K-1: the target, then decoys 0, 1, ...
        assert np.all(sc == 0) and np.all(pg["rank"] > 0)
        assert np.all(pg["is_decoy"][:, 0] == 0) and np.array_equal(pg["candidate"][:, 1:], np.tile(np.arange(top_k - 1), (len(sp), 1)))
    else:
        assert (sc < 0).mean() > 0.5 and len(np.unique(sc)) < len(sc) // 20


# ------------------------------------------------------------------------------------------------ 7. peak input edges
def edge_batch(cpu):
    sp = normal_spectra()
    b = Batch()
    # A: unusable intensities (NaN, -inf, 0, negative, subnormal) and m/z (<= 0, >= 1e7, P + 50 Da), P + 50 Da - 1 uDa,
    #    both sides of a bin edge, one m/z repeated with different intensities
    a0, a1 = int(sp.peak_off[0]), int(sp.peak_off[1])
    P = cpu.precursor_window(float(sp.precursor_mz[0]), int(sp.charge[0]), 10, 10)[0]
    mz, I = list(sp.peak_mz[a0:a1]), list(sp.peak_intensity[a0:a1])
    for j, v in enumerate((np.nan, -np.inf, 0.0, -3.0, 1e-45)):
        mz.append(float(sp.peak_mz[a0 + 3 + j]) + 0.003); I.append(v)
    mz += [-5.0, 0.0, 1e7, 2e7, mz_of(P + 50_000_000 - 1), mz_of(P + 50_000_000), mz_of(40_000 * W2 - 1), mz_of(40_000 * W2), 777.5, 777.5]
    I += [500.0] * 8 + [50.0, 80.0]
    b.add(sp.precursor_mz[0], sp.charge[0], mz, I)
    # B: one +inf intensity among ordinary peaks (its threshold is +inf: no peak is kept); C: every intensity +inf
    a0, a1 = int(sp.peak_off[1]), int(sp.peak_off[2])
    b.add(sp.precursor_mz[1], sp.charge[1], list(sp.peak_mz[a0:a1]) + [900.0], list(sp.peak_intensity[a0:a1]) + [np.inf])
    b.add(sp.precursor_mz[2], sp.charge[2], np.linspace(150.0, 600.0, 12), np.full(12, np.inf))
    # D: exactly 10 usable peaks, 3 of them under 5 %, plus unusable ones
    pre = precursor(cpu, float(sp.precursor_mz[3]), int(sp.charge[3]), 3)
    us = fragments(cpu, pre, 30, 5, nch=1)[:10]
    b.add(sp.precursor_mz[3], sp.charge[3], [mz_of(u) for u in us] + [-1.0, 3e7], [100.0] * 7 + [0.04] * 3 + [100.0, 100.0])
    # E: peaks exactly at the 5 % threshold (sqrt(1) == 0.05 * sqrt(400) in doubles) on fragments: dropped
    assert np.sqrt(1.0) == 0.05 * np.sqrt(400.0)
    pre = precursor(cpu, float(sp.precursor_mz[4]), int(sp.charge[4]), 4)
    us = fragments(cpu, pre, 30, 5, nch=1)[:24]
    b.add(sp.precursor_mz[4], sp.charge[4], [mz_of(u) for u in us], [400.0] * 12 + [1.0] * 12)
    # F: no peaks; G, H: ordinary
    b.add(sp.precursor_mz[5], sp.charge[5], [], [])
    b.add_from(sp, 6)
    b.add_from(sp, 7)
    return b.spectra()


@pytest.mark.parametrize("way", WAYS)
@pytest.mark.parametrize("min_peaks", [0, 1, 10, 1000])
def test_peak_input_edges(gpu, cpu, min_peaks, way, monkeypatch):
    _setup((gpu, cpu))
    sp = edge_batch(cpu)
    pg, _, sc, off = check(gpu, cpu, sp, SearchParams(10, 10, n_decoys=30, seed=5, top_k=_way(way, monkeypatch), min_peaks=min_peaks), way)
    ranked = pg["rank"][:, 0] > 0
    off = off.astype(np.int64)
    if min_peaks == 1000:
        assert not ranked.any()
    else:
        assert ranked[[0, 1, 2, 3, 4, 6, 7]].all() and not ranked[5]
        assert np.all(sc[off[1]:off[3]] == 0)                         # B and C keep no peak
        assert np.any(sc[off[4]:off[5]] != 0)
    geo = batch_geometry(cpu, sp, W2, min_peaks)
    if min_peaks <= 10:                 # D: 10 usable peaks, 7 kept; E: the 12 peaks at the threshold are dropped
        assert geo[3]["npk"] == 7 and geo[4]["npk"] == 12 and geo[5] is None


# ------------------------------------------------------------------------------------------------ 8. range refusals
def test_table_bin_limit_refusal(gpu, cpu, monkeypatch):
    """At 0.0001 Da a usable peak at m/z >= (2^26 - 76) * 100 uDa needs a table beyond 2^26 bins: refused with
    MD_ERR_UNSUPPORTED on every path (the oracle scores it); one uDa lower is scored.  The next call is unaffected."""
    _setup((gpu, cpu))
    P, z = wl.routing_precursors()[4][0], 3                        # 6.9 kDa
    edge = (MAX_BINS - XC - 1) * 100                                # the first uDa of bin 2^26 - 75
    # (alone, the spectrum is the only one the batch scores: nothing else reaches k_score on the pipelined path)
    for (u, ok), n_normal in [(c, n) for c in ((edge - 1, True), (edge, False)) for n in (0, 3)]:
        pre = precursor(cpu, pmz_of(P, z), z, 0)
        us = [x for x in fragments(cpu, pre, 20, 5) if x < 6_600_000_000][:30] + [u]
        sp = _with_normal([(pmz_of(P, z), z, [mz_of(x) for x in us], np.full(len(us), 100.0))], n_normal)
        geo = batch_geometry(cpu, sp, 100)
        assert (geo[0]["NB"] <= MAX_BINS) == ok and geo[0]["NB"] in (MAX_BINS, MAX_BINS + 1)
        for way in WAYS:
            with monkeypatch.context() as mp:
                prm = SearchParams(10, 10, fragment_tolerance=0.0001, n_decoys=20, seed=5, top_k=_way(way, mp))
                if ok:
                    check(gpu, cpu, sp, prm, way)
                    continue
                with pytest.raises(maxdecoy.MaxDecoyError) as ei:
                    gpu.identify(sp, prm)
                assert ei.value.status == -5 and "2^26" in str(ei.value)
                assert cpu.identify(sp, prm)[0]["rank"][0, 0] == 1
                check(gpu, cpu, normal_spectra(), SearchParams(10, 10, n_decoys=20, seed=5, top_k=prm.top_k), way)


def test_residue_mass_limit_refusal(gpu, cpu):
    """Scoring splits residue masses into (q, r) with q < 2^22 bins: at 0.0001 Da a fixed modification that brings W to
    419 430 400 uDa is refused with MD_ERR_UNSUPPORTED (the oracle accepts it); 1 uDa less is scored."""
    sp = normal_spectra()
    prm = SearchParams(10, 10, fragment_tolerance=0.0001, n_decoys=10, seed=5, top_k=5)
    w = 186_079_310                                                 # W
    try:
        for delta, ok in (((1 << 22) * 100 - 1 - w, True), ((1 << 22) * 100 - w, False), (250_000_000, False)):
            heavy_w = Modification("x:9", "Heavy", "A", True, "W", delta / 1e6)
            assert heavy_w.mono_mass_int == delta
            _setup((gpu, cpu), (synth.CAM, heavy_w), 0)
            if ok:
                check(gpu, cpu, sp, prm)
            else:
                with pytest.raises(maxdecoy.MaxDecoyError) as ei:
                    gpu.identify(sp, prm)
                assert ei.value.status == -5 and "fragment_tolerance too small" in str(ei.value)
                assert np.any(cpu.identify(sp, prm)[0]["rank"] > 0)
    finally:
        _setup((gpu, cpu))
    check(gpu, cpu, sp, prm)
