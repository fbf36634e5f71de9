"""Shared seeded workloads for the parity tests (small enough for the oracle to finish in seconds)."""
import functools
import json
import os

import numpy as np

from maxdecoy import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@functools.lru_cache(maxsize=None)
def p77377():
    with open(os.path.join(GOLDEN, "p77377_trypsin.json")) as fh:
        return json.load(fh)


@functools.lru_cache(maxsize=None)
def proteins(n, seed=20260101):
    return tuple(synth.synthetic_proteins(n, seed))


@functools.lru_cache(maxsize=None)
def spectra(n_prot, n_spec, mc, with_ox=False, seed=7):
    mods = (synth.CAM, synth.OXM) if with_ox else (synth.CAM,)
    return synth.synthetic_spectra(list(proteins(n_prot)), n_spec, mc, mods=mods, seed=seed)


def precursors_of(engine, sp, lppm=10, uppm=10):
    out = []
    for i in range(len(sp)):
        P, lo, hi = engine.precursor_window(float(sp.precursor_mz[i]), int(sp.charge[i]), lppm, uppm)
        out.append((P, lo, hi, int(sp.charge[i]), i))
    return out


def heavy_precursors():
    """Heavy precursors (1.7-6.4 kDa, 10 ppm): decoy attempts grow past 32 residues, some past 60."""
    return [(m, m - m // 100_000, m + m // 100_000, 2 + i % 3, 500 + i)
            for i, m in enumerate((1_700_800_000, 2_900_400_000, 3_600_700_000, 4_300_100_000, 5_200_900_000, 6_400_300_000))]


def routing_precursors():
    """Precursors whose decoys include sequences of exactly 32, 33 and 60 residues (the repair passes' routing edges)."""
    return [(m, m - m // 100_000, m + m // 100_000, 2 + i % 3, 900 + i)
            for i, m in enumerate((3_550_000_000, 3_700_000_000, 3_850_000_000, 6_700_000_000, 6_900_000_000, 7_050_000_000))]


def degenerate_mod_sets():
    """Modification sets that make letters collide: G+14.01565 equals A to the micro-dalton (an equal-mass run: ties go to
    the lower alphabet index), S+12.03637 lands 10 uDa under V and T+27.04728 lands 1 uDa above K (near-ties on either side of
    a midpoint), plus two variable letters, one of them also fixed (the generic variable-modification path)."""
    from maxdecoy import Modification
    fix_g = Modification("x:1", "GtoA", "A", True, "G", 14.015650)
    fix_s = Modification("x:2", "StoV", "A", True, "S", 12.036370)
    fix_t = Modification("x:3", "TtoK", "A", True, "T", 27.047280)
    var_m = Modification("unimod:35", "Oxidation", "A", False, "M", 15.994915)
    var_g = Modification("x:4", "Gvar", "A", False, "G", 0.984016)
    return [((synth.CAM, fix_g, fix_s, fix_t), 0), ((synth.CAM, fix_g, fix_s, var_m, var_g), 2)]


def decoy_strings(table):
    raw = table["seq"].tobytes()
    so = table["seq_off"]
    return [raw[int(so[i]):int(so[i + 1])].decode() for i in range(len(so) - 1)]
