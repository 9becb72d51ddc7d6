"""CPU model of the candidate-set logic of the tensor-core kNN epilogue (csrc/knn_tc.cu) -- the part the GPU tests can only probe
through final lists: several sets per row (column halves, CTAs) scan disjoint column ranges in streaming order, each keeps the 32
smallest stored values it has seen, prunes against its own maximum and against what the other sets have published, and the merged
lists feed the exact re-rank.  Stored values have five low mantissa bits cleared, so VALUE TIES ARE COMMON, and the entry a full
set drops among tied maxima is picked by slot, not by column index.  What the completeness proof of knn_rerank needs is a statement
about VALUES, checked here on data that ties heavily:
  1. every column that is not among the merged 32 candidates has a stored value >= the 32nd candidate's, whatever the publication
     schedule and whichever form of the shared bound is used;
  2. k > 33: the second round admits every column whose stored value is >= the first round's 32nd value except that entry itself;
     after dropping the first-round members that come back, every column outside both rounds has a stored value >= the second
     round's 32nd.  (The former rule, "key beyond the first round's 32nd KEY", can lose a column that ties with the 32nd value,
     has the smaller index and was dropped from its set: a set's slots are not in index order once entries have been replaced.)
"""
import numpy as np
import pytest

KC = 32


def clear5(v: np.ndarray) -> np.ndarray:
    return (np.ascontiguousarray(v, dtype=np.float32).view(np.uint32) & np.uint32(0xFFFFFFE0)).view(np.float32)


def next_bucket(t: np.float32) -> np.float32:
    """start of the five-bit bucket after the one t lies in (positive floats)"""
    b = np.array([t], dtype=np.float32).view(np.uint32)
    return ((b | np.uint32(31)) + np.uint32(1)).view(np.float32)[0]


def run_row(values: np.ndarray, nsets: int, chunk: int, publish_every: int, rule: str, excl=None):
    """values: the row's shifted approximate values v' > 0 (float32), one per column.  Columns are dealt to `nsets` sets in
    contiguous ranges; all sets advance in lockstep `chunk` columns at a time; every `publish_every` chunks each full set publishes
    its maximum and reads the minimum over what the OTHERS have published.  Returns the union of the sets as (stored value, index)."""
    n = len(values)
    bounds = np.linspace(0, n, nsets + 1).astype(int)
    sets = [[] for _ in range(nsets)]            # lists of (stored value, index), at most KC
    tlim = [np.float32(np.inf)] * nsets
    published = [np.float32(np.inf)] * nsets
    pos = [int(b) for b in bounds[:-1]]
    step = 0
    while any(pos[s] < bounds[s + 1] for s in range(nsets)):
        for s in range(nsets):
            for j in range(pos[s], min(pos[s] + chunk, int(bounds[s + 1]))):
                v = values[j]
                stored = clear5(np.array([v]))[0]
                if excl is not None and (stored, j) <= excl:
                    continue                        # second round: the first round's list holds it
                smax = max(x[0] for x in sets[s]) if len(sets[s]) == KC else np.float32(np.inf)
                thr = min(smax, tlim[s])
                if not (v < thr):
                    continue
                if len(sets[s]) < KC:
                    sets[s].append((stored, j))
                else:                               # replace the largest stored value (ties: any of them -- later column wins the slot)
                    k = max(range(KC), key=lambda q: (sets[s][q][0], q))
                    sets[s][k] = (stored, j)
            pos[s] = min(pos[s] + chunk, int(bounds[s + 1]))
        step += 1
        if step % publish_every == 0:
            for s in range(nsets):
                if len(sets[s]) == KC:
                    published[s] = min(published[s], max(x[0] for x in sets[s]))
            for s in range(nsets):
                others = [published[o] for o in range(nsets) if o != s and np.isfinite(published[o])]
                if others:
                    t = min(others)
                    tlim[s] = min(tlim[s], next_bucket(t) if rule == "next_bucket" else t)
    return sorted(x for st in sets for x in st)


def tied_values(rng, n, levels):
    """positive float32 values with many exact ties after clearing: a few hundred distinct levels plus sub-bucket noise"""
    base = rng.choice(np.linspace(1.0, 3.0, levels), size=n).astype(np.float32)
    noise = (rng.integers(0, 32, size=n).astype(np.uint32))           # differences inside one five-bit bucket
    return (clear5(base).view(np.uint32) | noise).view(np.float32)


def first_round(v, nsets, chunk, publish_every, rule):
    return run_row(v, nsets, chunk, publish_every, rule)[:KC]


@pytest.mark.parametrize("rule", ["next_bucket", "plain"])
@pytest.mark.parametrize("nsets,chunk,publish_every", [(2, 32, 4), (4, 32, 8), (6, 16, 3), (2, 32, 1)])
@pytest.mark.parametrize("levels", [40, 400])
def test_every_non_candidate_is_at_least_the_32nd_value(nsets, chunk, publish_every, levels, rule):
    rng = np.random.default_rng(100 * nsets + chunk + publish_every + levels)
    for trial in range(6):
        v = tied_values(rng, 1500, levels)
        stored = clear5(v)
        r1 = first_round(v, nsets, chunk, publish_every, rule)
        assert len(r1) == KC
        members = {j for _, j in r1}
        u32 = r1[-1][0]
        assert all(stored[j] >= u32 for j in range(len(v)) if j not in members), (trial, nsets, levels)
        assert sorted(s for s, _ in r1) == sorted(stored)[:KC]      # the 32 smallest VALUES, whichever tied columns carry them


def second_round_rule(rule2, first):
    last = first[-1]
    if rule2 == "value":   # knn_tc.cu: value >= the 32nd value, except the 32nd entry itself
        return lambda key: key != last and key[0] >= last[0]
    return lambda key: key > last   # the former rule


def run_two_rounds(v, rule2):
    r1 = first_round(v, 4, 32, 4, "next_bucket")
    admit = second_round_rule(rule2, r1)
    stored = clear5(v)
    # second round: the same machinery over the admitted columns only (their own thresholds)
    idx = [j for j in range(len(v)) if admit((stored[j], j))]
    sub = run_row(v[idx], 4, 32, 4, "next_bucket")[:KC]
    r2 = [(s, idx[j]) for s, j in sub]
    first_members = {j for _, j in r1}
    r2_new = [x for x in r2 if x[1] not in first_members]          # the k > 33 re-rank drops the first round's members by index
    return r1, r2, r2_new


@pytest.mark.parametrize("levels", [40, 400])
def test_second_round_leaves_nothing_below_its_32nd_value(levels):
    rng = np.random.default_rng(11 + levels)
    for trial in range(6):
        v = tied_values(rng, 2000, levels)
        stored = clear5(v)
        r1, r2, r2_new = run_two_rounds(v, "value")
        cand = {j for _, j in r1} | {j for _, j in r2_new}
        lower = r2[-1][0]
        assert all(stored[j] >= lower for j in range(len(v)) if j not in cand), trial
        assert len(cand) >= 2 * KC - 1 - sum(1 for s_, _ in r1 if s_ == r1[-1][0])   # only value ties with the 32nd come back
