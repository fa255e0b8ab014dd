"""CPU test of the equivalence the fused align-and-predict path (`Predictor.submit_pairs`, `nw_trace_frame_kernel`) relies on: the
contact map the reference builds from the gapped strings `insert_gaps(q, t, ops)` (`build_align_contact_map`,
bio_utils.py:348-385) equals the map built from a query-frame table that a walk over the alignment string fills directly - diagonal
column: target residue over query residue (nothing when the structure has no such row), D column: query residue unmapped and
spawning generated contacts, I column: nothing - without any gapped string."""
import numpy as np
import pytest

import cmap_oracle as co
import nw_oracle as nw
from metagenomic_deepfri_b200 import synth

THRESHOLDS = (6.0, 10.0)
GENS = (0, 1, 2, 3)


def frame_contact_map(query: str, target: str, ops: str, coords: np.ndarray, threshold: float, generated_contacts: int) -> np.ndarray:
    """The frame walk restated: ops + coordinates -> int32 [Lq, Lq] map, the way the device builds it (query frame, then the
    distance test on query index pairs, diagonal and generated contacts)."""
    Lq, Lt = len(query), len(target)
    t_of_q = np.full(Lq, -1, np.int64)               # target residue over each query residue, -1 = none
    gap = np.zeros(Lq, bool)                         # query residue over a target gap (spawns generated contacts)
    i = j = 0
    for o in ops:
        if o in "MX":
            t_of_q[i] = j
            i += 1
            j += 1
        elif o == "D":
            gap[i] = True
            i += 1
        elif o == "I":
            j += 1
        else:
            raise AssertionError(o)
    assert i == Lq and j == Lt
    out = np.zeros((Lq, Lq), np.int32)
    np.fill_diagonal(out, 1)
    for g in np.flatnonzero(gap):
        for k in range(1, generated_contacts + 1):
            for a in (g - k, g + k):
                if 0 <= a < Lq:
                    out[a, g] = out[g, a] = 1
    rows = coords.shape[0]
    mapped = np.flatnonzero((t_of_q >= 0) & (t_of_q < rows))
    if mapped.size:
        target_map = co.calculate_contact_map(coords, threshold=threshold)
        ti = t_of_q[mapped]
        out[np.ix_(mapped, mapped)] |= target_map[np.ix_(ti, ti)]
    return out


def walk(rng, n):
    steps = rng.normal(size=(n, 3))
    steps *= 3.8 / np.linalg.norm(steps, axis=1, keepdims=True)
    return np.round(np.cumsum(steps, axis=0), 3).astype(np.float32)


def edge_cases():
    """(query, target, coordinates): empty target (all D), leading / trailing gaps of both kinds, structures with fewer and with
    more rows than the target, one-residue queries."""
    rng = np.random.default_rng(11)
    core = "MKTAYIAKQRQISFVKSHFSRQ"
    return [
        ("ACDEFG", "", walk(rng, 4)),                        # empty target: every column is D
        (core, "WWWW" + core, walk(rng, 26)),                # leading I columns
        (core, core + "WWWW", walk(rng, 26)),                # trailing I columns
        ("WWWW" + core, core, walk(rng, 22)),                # leading D columns
        (core + "WWWW", core, walk(rng, 22)),                # trailing D columns
        (core, core, walk(rng, 10)),                         # fewer structure rows than target residues
        (core, core[:15], walk(rng, 40)),                    # more structure rows than target residues
        ("A", core, walk(rng, 22)),                          # one-residue query against a longer target
        ("W", "W", walk(rng, 1)),
        ("W", "A", walk(rng, 3)),
    ]


def cases():
    wl = synth.keyed_workload(np.arange(2048), 3)
    out = [(q, gt.replace("-", ""), c) for q, gt, c in zip(wl.query_seqs, wl.gapped_target, wl.coords)]
    return out + edge_cases()


@pytest.fixture(scope="module")
def aligned():
    res = []
    for q, t, c in cases():
        _, ops = nw.align(q, t)
        res.append((q, t, ops, c))
    return res


def test_edge_cases_cover_what_they_claim(aligned):
    ops = {q + "|" + t: o for q, t, o, _ in aligned}
    assert set(ops["ACDEFG|"]) == {"D"}
    assert ops["MKTAYIAKQRQISFVKSHFSRQ|WWWWMKTAYIAKQRQISFVKSHFSRQ"].startswith("IIII")
    assert ops["MKTAYIAKQRQISFVKSHFSRQ|MKTAYIAKQRQISFVKSHFSRQWWWW"].endswith("IIII")
    assert ops["WWWWMKTAYIAKQRQISFVKSHFSRQ|MKTAYIAKQRQISFVKSHFSRQ"].startswith("DDDD")
    assert ops["MKTAYIAKQRQISFVKSHFSRQWWWW|MKTAYIAKQRQISFVKSHFSRQ"].endswith("DDDD")


@pytest.mark.parametrize("threshold", THRESHOLDS)
def test_frame_walk_equals_gapped_strings(aligned, threshold):
    for q, t, ops, c in aligned:
        gq, gt = co.insert_gaps(q, t, ops)
        for gen in GENS:
            want = co.build_align_contact_map(gq, gt, c, threshold, gen)
            got = frame_contact_map(q, t, ops, c, threshold, gen)
            assert np.array_equal(got, want), (len(q), len(t), c.shape[0], threshold, gen)
