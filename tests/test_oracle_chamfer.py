"""Pins the chamfer oracle (oracle/chamfer.py): bit-exact against the golden vectors the COMPILED reference wrote
(tests/golden/chamfer_*.npz, oracle/make_golden_chamfer.py; tests/golden/ref_chamfer_random.npz,
oracle/make_golden_ref.py on the inputs of tests/ref_inputs.py).  CPU only."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import chamfer as oc
from tests import ref_inputs as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = sorted(glob.glob(os.path.join(ROOT, 'tests', 'golden', 'chamfer_*.npz')))


def test_golden_present():
    assert len(GOLDEN) >= 5


@pytest.mark.parametrize('path', GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_port_matches_golden_bit_exact(path):
    g = np.load(path)
    d1, d2, i1, i2 = oc.chamfer_forward(g['xyz1'], g['xyz2'])
    assert np.array_equal(i1, g['idx1']) and np.array_equal(i2, g['idx2'])
    assert np.array_equal(d1.view(np.uint32), g['dist1'].view(np.uint32))
    assert np.array_equal(d2.view(np.uint32), g['dist2'].view(np.uint32))
    g1, g2 = oc.chamfer_backward(g['xyz1'], g['xyz2'], g['grad_dist1'], g['grad_dist2'], g['idx1'], g['idx2'])
    assert np.array_equal(g1.view(np.uint32), g['grad_xyz1'].view(np.uint32))
    assert np.array_equal(g2.view(np.uint32), g['grad_xyz2'].view(np.uint32))
    h1, h2 = oc.chamfer_backward(g['xyz1'], g['xyz2'], g['grad_dist1'], np.zeros_like(g['grad_dist2']), g['idx1'], g['idx2'])
    assert np.array_equal(h1.view(np.uint32), g['grad_xyz1_oneway'].view(np.uint32))
    assert np.array_equal(h2.view(np.uint32), g['grad_xyz2_oneway'].view(np.uint32))


def test_ties_take_first_minimum():
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'chamfer_ties.npz'))
    a, c = g['xyz1'], g['xyz2']
    D = ((c[:, None, :, :] - a[:, :, None, :]) ** 2).sum(-1)
    ntie = ((D == D.min(-1, keepdims=True)).sum(-1) > 1).sum()
    assert ntie > 20                                   # the fixture really exercises ties
    assert np.array_equal(g['idx1'], D.argmin(-1))     # numpy argmin = first minimum = the reference's `d < best`


def test_port_matches_live_reference():
    """Bit-exact against the compiled reference module's forward / backward on random clouds of several shapes, stored by
    oracle/make_golden_ref.py (the name dates from when the module was called inside the test)."""
    ref = R.fixture('ref_chamfer_random')
    for b, n, m, a, c, gd1, gd2 in R.chamfer_random_cases():
        r = {k.split(':')[1]: v for k, v in ref.items() if k.startswith('%d_%d_%d:' % (b, n, m))}
        p1, p2, q1, q2 = oc.chamfer_forward(a, c)
        assert np.array_equal(q1, r['idx1']) and np.array_equal(q2, r['idx2'])
        assert np.array_equal(p1, r['dist1']) and np.array_equal(p2, r['dist2'])
        o1, o2 = oc.chamfer_backward(a, c, gd1, gd2, q1, q2)
        assert np.array_equal(o1, r['grad_xyz1']) and np.array_equal(o2, r['grad_xyz2'])


def test_empty_target_cloud():
    d, i = oc.nn_search(np.zeros((2, 4, 3), np.float32), np.zeros((2, 0, 3), np.float32))
    assert d.shape == (2, 4) and not d.any() and not i.any()


def test_points3d_loss_gradient_is_the_chamfer_scatter():
    """autograd through the gathered pairs == 0.5 * w * chamfer_backward(grad_dist1 = 1) on the predicted cloud."""
    rng = np.random.default_rng(3)
    B, T, No, Nv = 2, 3, 40, 70
    obs = torch.from_numpy(rng.normal(size=(B, T, No, 3)).astype(np.float32))
    pred = torch.from_numpy(rng.normal(size=(B, T, Nv, 3)).astype(np.float32)).requires_grad_(True)
    loss = oc.points3d_loss(obs, pred, robust_loss='none')
    loss.backward()
    o = obs.reshape(B * T, No, 3).numpy()
    p = pred.detach().reshape(B * T, Nv, 3).numpy()
    d1, i1 = oc.nn_search(o, p)
    assert abs(float(loss) - 0.5 * float(d1.astype(np.float64).sum())) < 1e-4 * float(loss)
    _, g2 = oc.chamfer_backward(o, p, np.full((B * T, No), 0.5, np.float32), None, i1, None)
    assert np.allclose(pred.grad.reshape(B * T, Nv, 3).numpy(), g2, rtol=1e-5, atol=1e-6)


def test_bisquare_weights_reject_outliers():
    res = torch.cat([torch.rand(1, 200) * 0.01, torch.tensor([[5.0, 9.0]])], 1)
    w = oc.bisquare_robust_weights(res)
    assert float(w[0, -1]) == 0.0 and float(w[0, -2]) == 0.0 and float(w[0, :200].min()) > 0.0
