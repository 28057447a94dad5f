"""Row F1 (SURVEY section 8f): proximity edge selection.  oracle.proximity_edges against the edge lists the UNMODIFIED reference method
`FactorGraph.add_proximity_factors` (factor_graph.py:346-412) emitted on the same inputs (tests/golden/make_proximity_golden.py);
bit-exact, order included."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle.proximity as prox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_proximity_golden as mk  # noqa: E402

@pytest.fixture(scope="module")
def gold():
    return torch.load(os.path.join(ROOT, "tests", "golden", "proximity.pt"))


def oracle_case(case):
    name, kw, t, stereo, max_factors, seed, n_exist, nan = case
    d = mk.distance_matrix(kw["t0"], kw["t1"], t, seed, nan=nan)
    e = mk.existing_edges(t, n_exist, seed + 100)
    ii1 = torch.cat([e[0], e[2], e[4]])
    jj1 = torch.cat([e[1], e[3], e[5]])
    es, _ = prox.proximity_edges(d.numpy(), kw["t0"], kw["t1"], t, ii1.numpy(), jj1.numpy(), rad=kw["rad"], nms=kw["nms"],
                                 thresh=kw["thresh"], max_factors=max_factors, stereo=stereo)
    return es


@pytest.mark.parametrize("name", [c[0] for c in mk.cases()])
def test_oracle_matches_the_reference_method(gold, name):
    case = [c for c in mk.cases() if c[0] == name][0]
    es = oracle_case(case)
    g = gold[name + "_es"].numpy()
    assert es.shape == g.shape, (es.shape, g.shape)
    assert np.array_equal(es, g)


def test_cases_exercise_every_branch(gold):
    by = {c[0]: c for c in mk.cases()}
    # proximity edges beyond the temporal neighbours were selected, the cap stopped one case early, NaNs were taken
    for name in ("init_12", "frontend_30", "backend_90", "stereo_20", "with_nan"):
        _, kw, t, stereo, mf, *_ = by[name]
        n_base = sum((1 if stereo else 0) + 2 * (i - max(i - kw["rad"] - 1, 0)) for i in range(kw["t0"], t))
        assert gold[name + "_es"].shape[0] > n_base, name
    assert gold["backend_cap_es"].shape[0] in (382, 383, 384)     # first length above the cap of 380, in steps of 2
    full = oracle_case(by["backend_cap"][:4] + (-1,) + by["backend_cap"][5:])
    assert full.shape[0] > gold["backend_cap_es"].shape[0]
