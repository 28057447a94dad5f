"""A process that drives a second GPU gets the same results there as on the first.  Kernel attributes (the dynamic shared-memory
opt-in) and the cached device facts (SM count, shared-memory limit, Cholesky cluster size) belong to one device, so device 1 after
device 0 exercises the setup of a device the process has not launched on yet."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle
import oracle.proximity as prox
from droid_slam_b200 import synth
from droid_slam_b200.update import UpdateModule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_proximity_golden as mk  # noqa: E402

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two visible CUDA devices")]


def test_proximity_and_update_operator_on_a_second_device():
    from droid_slam_b200 import install
    be = install()
    # 700 x 700 pairs: a 61 KB "still alive" bitmap, which fits shared memory only with the opt-in beyond 48 KB
    t = 700
    d = mk.distance_matrix(0, 0, t, 7, nan=3)
    e = mk.existing_edges(t, 500, 107)
    ii1, jj1 = torch.cat([e[0], e[2], e[4]]), torch.cat([e[1], e[3], e[5]])
    want, _ = prox.proximity_edges(d.numpy(), 0, 0, t, ii1.numpy(), jj1.numpy(), rad=2, nms=2, thresh=22.0, max_factors=-1, stereo=False)
    w = synth.make_update_weights(0)
    net, inp, corr, flow, ii = synth.make_update_inputs(E=4, ht=48, wd=64, seed=4, n_src=2)
    ref = oracle.update_module_forward(w, net.half().float(), inp.half().float(), corr.half().float(), flow, ii)
    tol = dict(net=1e-2, delta=2e-2, weight=1e-2, eta=2e-4, upmask=2e-2)
    for dev in ("cuda:0", "cuda:1"):
        es = be.proximity_edges(d.to(dev), 0, 0, t, ii1.to(dev), jj1.to(dev), 2, 2, 22.0, -1, False)
        assert np.array_equal(es.cpu().numpy(), want), dev
        mod = UpdateModule().to(dev)
        mod.load_state_dict(w)
        with torch.no_grad():
            got = mod(net.half().to(dev), inp.half().to(dev), corr.half().to(dev), flow.to(dev), ii.to(dev))
        torch.cuda.synchronize(dev)
        for k, a, b in zip(tol, got, ref):
            err = float((a.float().cpu() - b).abs().max())
            assert err < tol[k], (dev, k, err)
