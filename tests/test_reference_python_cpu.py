"""The reference's own Python call sites, imported unmodified (tests/golden/make_reference_python_golden.py), against the oracle:
  * pops.projective_transform (geom/projective_ops.py:165-198, called by DepthVideo.reproject depth_video.py:171-179) pins
    oracle.reproject -- row A5;
  * CorrBlock / AltCorrBlock (modules/corr.py:23-117) pin oracle.corr_pyramid / corr_block_lookup / altcorr_block_lookup.
The reference's outputs are the stored vectors of tests/golden/reference_python.pt."""
import os
import sys

import pytest
import torch

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_reference_python_golden as mk  # noqa: E402

@pytest.fixture(scope="module")
def gold():
    return torch.load(os.path.join(ROOT, "tests", "golden", "reference_python.pt"))


@pytest.mark.parametrize("case", [c[0] for c in mk.reproject_cases()])
def test_oracle_reproject_matches_reference_projective_transform(gold, case):
    name, poses, disps, intr, ii, jj = [c for c in mk.reproject_cases() if c[0] == case][0]
    coords, valid = oracle.reproject(poses, disps, intr, ii, jj)
    gc, gv = gold["reproject_%s_coords" % name][0], gold["reproject_%s_valid" % name][0]
    assert coords.shape == gc.shape and valid.shape == gv.shape
    assert torch.equal(valid, gv)
    rel = ((coords - gc).abs() / gc.abs().clamp(min=1.0)).max()          # pixel coordinates: 1e-4 relative, floor 1 px
    assert float(rel) < 1e-4, float(rel)                                  # observed 5e-6 (lietorch normalises quaternions, the oracle does not)


def test_oracle_corr_classes_match_reference_classes(gold):
    (f1, f2, coords), (fm, ca, ii, jj) = mk.corr_cases()
    pyr = oracle.corr_pyramid(f1, f2, 3)
    for l, v in enumerate(pyr):
        assert torch.equal(v, gold["corrblock_pyr%d" % l])
    assert torch.equal(oracle.corr_block_lookup(pyr, coords, 3), gold["corrblock_lookup"])
    assert torch.equal(oracle.altcorr_block_lookup(oracle.fmap_pyramid(fm, 3), ca, ii, jj, 3), gold["altcorrblock_lookup"])
