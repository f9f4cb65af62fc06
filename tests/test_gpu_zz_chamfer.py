"""GPU parity of the chamfer nearest-neighbour kernels (csrc/chamfer.cu through the C-ABI) and of the points3d
energy built on them.  Bit-exact against (1) the golden vectors written by the reference's own compiled C++
(tests/golden/chamfer_*.npz), (2) the CPU oracle port on ragged sizes, (3) the compiled reference's forward on larger
random clouds (tests/golden/ref_chamfer_gpu.npz); closure-level parity against the PROX-RGBD golden case of the
unmodified reference (stage3_proxd) and the oracle port; size-independent properties at the full PROX size
(4096 observed points against 6890 vertices).

(The file sorts last among the GPU tests on purpose: it is the newest row of the scope table.)"""
import glob
import os

import numpy as np
import pytest
import torch

from humor_b200 import synth
from oracle import chamfer as oc
from tests import util_stage3 as U

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = sorted(glob.glob(os.path.join(ROOT, 'tests', 'golden', 'chamfer_*.npz')))


def bits(x):
    return np.ascontiguousarray(x).view(np.uint32)


def dev(a, grad=False):
    return torch.as_tensor(a).cuda().requires_grad_(grad)


@pytest.mark.parametrize('path', GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_kernels_match_reference_golden_bit_exact(path):
    from humor_b200.chamfer import chamfer_nn
    g = np.load(path)
    a, c = dev(g['xyz1'], True), dev(g['xyz2'], True)
    d1, d2, i1, i2 = chamfer_nn(a, c)
    assert np.array_equal(i1.cpu().numpy(), g['idx1']) and np.array_equal(i2.cpu().numpy(), g['idx2'])
    assert np.array_equal(bits(d1.detach().cpu().numpy()), bits(g['dist1']))
    assert np.array_equal(bits(d2.detach().cpu().numpy()), bits(g['dist2']))
    torch.autograd.backward([d1, d2], [dev(g['grad_dist1']), dev(g['grad_dist2'])])
    assert np.array_equal(bits(a.grad.cpu().numpy()), bits(g['grad_xyz1']))
    assert np.array_equal(bits(c.grad.cpu().numpy()), bits(g['grad_xyz2']))
    # one-way search (what points3d_loss uses): same dist1/idx1, gradient of the reference with a zero dist2 gradient
    a2, c2 = dev(g['xyz1'], True), dev(g['xyz2'], True)
    e1, e2, j1, j2 = chamfer_nn(a2, c2, one_way=True)
    assert e2 is None and j2 is None and torch.equal(e1, d1) and torch.equal(j1, i1)
    e1.backward(dev(g['grad_dist1']))
    assert np.array_equal(bits(a2.grad.cpu().numpy()), bits(g['grad_xyz1_oneway']))
    assert np.array_equal(bits(c2.grad.cpu().numpy()), bits(g['grad_xyz2_oneway']))


@pytest.mark.parametrize('b,n,m', [(1, 1, 1), (2, 1023, 1025), (1, 1025, 3), (3, 5, 2049), (2, 2050, 1024), (1, 0, 7), (2, 6, 0)])
def test_kernels_match_port_on_ragged_sizes(b, n, m):
    from humor_b200.chamfer import ChamferDistance
    rng = np.random.default_rng(n * 7 + m)
    a = rng.normal(size=(b, n, 3)).astype(np.float32)
    c = rng.normal(size=(b, m, 3)).astype(np.float32)
    ta, tc = dev(a, True), dev(c, True)
    d1, d2 = ChamferDistance()(ta, tc)                       # the reference's module surface (chamfer_distance.py:58-60)
    e1, e2, j1, j2 = oc.chamfer_forward(a, c)
    assert np.array_equal(bits(d1.detach().cpu().numpy()), bits(e1)) and np.array_equal(bits(d2.detach().cpu().numpy()), bits(e2))
    gd1 = rng.normal(size=(b, n)).astype(np.float32)
    gd2 = rng.normal(size=(b, m)).astype(np.float32)
    torch.autograd.backward([d1, d2], [dev(gd1), dev(gd2)])
    o1, o2 = oc.chamfer_backward(a, c, gd1 if m > 0 else None, gd2 if n > 0 else None, j1, j2)
    assert np.array_equal(bits(ta.grad.cpu().numpy()), bits(o1)) and np.array_equal(bits(tc.grad.cpu().numpy()), bits(o2))


def test_matches_compiled_reference_when_present():
    """Bit-exact against the compiled reference module's forward on 4 x 600 against 4 x 1500 random points, stored by
    oracle/make_golden_ref.py; always runs (the name dates from when the module itself had to be present)."""
    from humor_b200.chamfer import chamfer_nn
    from tests import ref_inputs as R
    ref = R.fixture('ref_chamfer_gpu')
    a, c = R.chamfer_gpu_case()
    e1, e2, j1, j2 = chamfer_nn(dev(a), dev(c))
    assert np.array_equal(bits(e1.cpu().numpy()), bits(ref['dist1'])) and np.array_equal(bits(e2.cpu().numpy()), bits(ref['dist2']))
    assert np.array_equal(j1.cpu().numpy(), ref['idx1']) and np.array_equal(j2.cpu().numpy(), ref['idx2'])


def test_full_size_properties():
    """PROX size: 4096 observed points against 6890 vertices, 64 frames (the oracle needs ~a minute for this on CPU, so:
    properties + an oracle check of 2 frames).  (1) every reported distance is the distance to the reported index;
    (2) no sampled target is closer; (3) a cloud searched against itself finds itself at distance 0;
    (4) two runs agree bit for bit (forward and reverse)."""
    from humor_b200.chamfer import chamfer_nn
    g = torch.Generator(device='cuda').manual_seed(0)
    b, n, m = 64, 4096, 6890
    pred = torch.randn(b, m, 3, device='cuda', generator=g) * torch.tensor([0.25, 0.9, 0.15], device='cuda') + 1.5
    obs = pred[:, torch.randint(0, m, (n,), device='cuda', generator=g)] + 0.01 * torch.randn(b, n, 3, device='cuda', generator=g)
    pred.requires_grad_(True)
    d1, _, i1, _ = chamfer_nn(obs, pred, one_way=True)
    near = torch.gather(pred.detach(), 1, i1.long()[:, :, None].expand(-1, -1, 3))
    diff = near - obs
    sq = diff * diff
    assert torch.equal(d1.detach(), (sq[..., 0] + sq[..., 1]) + sq[..., 2])
    probe = torch.randint(0, m, (256,), device='cuda', generator=g)
    dp = ((pred.detach()[:, probe][:, None] - obs[:, :, None]) ** 2).sum(-1).min(-1)[0]
    assert bool((d1.detach() <= dp * (1 + 1e-6) + 1e-12).all())
    d_self, _, i_self, _ = chamfer_nn(pred.detach(), pred.detach(), one_way=True)
    assert float(d_self.max()) == 0.0
    gd = torch.rand(b, n, device='cuda', generator=g)
    d1.backward(gd)
    g_first = pred.grad.clone()
    pred.grad = None
    d1b, _, i1b, _ = chamfer_nn(obs, pred, one_way=True)
    d1b.backward(gd)
    assert torch.equal(d1b, d1) and torch.equal(i1b, i1) and torch.equal(pred.grad, g_first)
    e, j = oc.nn_search(obs[:2].cpu().numpy(), pred[:2].detach().cpu().numpy())
    assert np.array_equal(j, i1[:2].cpu().numpy()) and np.array_equal(bits(e), bits(d1[:2].detach().cpu().numpy()))
    _, o2 = oc.chamfer_backward(obs[:2].cpu().numpy(), pred[:2].detach().cpu().numpy(), gd[:2].cpu().numpy(), None, j, None)
    assert np.array_equal(bits(o2), bits(g_first[:2].cpu().numpy()))


def test_points3d_loss_matches_oracle():
    from humor_b200.fitting_loss import FittingLoss
    rng = np.random.RandomState(5)
    B, T, V, No = 3, 4, 700, 256
    verts = (rng.randn(B, T, V, 3) * np.array([0.25, 0.9, 0.15]) + 1.5).astype(np.float32)
    obs = synth.sample_point_cloud(verts, No, seed=1)
    for robust in ('bisquare', 'none'):
        fl = FittingLoss([dict(synth.PROXD_STAGE3_WEIGHTS)] * 3, robust_loss=robust, use_chamfer=True)
        vp = dev(verts, True)
        loss = fl.points3d_loss(dev(obs), vp)
        loss.backward()
        vc = torch.tensor(verts, requires_grad=True)
        ref = oc.points3d_loss(torch.tensor(obs), vc, robust)
        ref.backward()
        assert abs(float(loss) - float(ref)) <= 1e-5 * max(1.0, abs(float(ref))), (robust, float(loss), float(ref))
        assert float((vp.grad.cpu() - vc.grad).abs().max()) <= 1e-5 * float(vc.grad.abs().max()), robust


@pytest.mark.parametrize('precision', ['exact', 'tensor'])
def test_closure_matches_reference_golden_proxd(precision):
    """Stage-III closure with the point-cloud energy (configs/fit_proxd.cfg weights) against the fixture the
    UNMODIFIED reference produced with its own compiled chamfer module."""
    from tests.golden_util import load_case, check_against_golden
    g, prob, c = load_case('stage3_proxd')
    mo = U.build_product(c['B'], c['T'], c['W'], c['optim_floor'], prob)
    mo.set_precision(precision)
    loss, grads, aux = U.closure_product(mo, prob, c['nsteps'], c['scale'])
    assert 'points3d' in aux['stats']
    check_against_golden(g, loss, aux['stats'], grads, loss_tol=1e-5, stat_tol=1e-4, grad_tol=1e-4 if precision == 'exact' else 1e-2)


def test_proxd_graph_step_matches_eager():
    """The points3d closure through stage3_step (CUDA graph when capturable, eager otherwise): same loss/gradients."""
    from tests.golden_util import load_case
    g, prob, c = load_case('stage3_proxd')
    mo = U.build_product(c['B'], c['T'], c['W'], c['optim_floor'], prob)
    mo.set_precision('exact')
    l_e, g_e, _ = U.closure_product(mo, prob)
    names = mo.set_stage3_state(prob['params'])
    obs = {k: torch.as_tensor(v).cuda() for k, v in prob['obs'].items() if k in U.obs_keys(True, prob)}
    params = [getattr(mo, n) for n in names]
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        loss = mo.stage3_step(obs, None, 1.0, params)
    assert abs(float(loss) - l_e) <= 1e-5 * max(1.0, abs(l_e))
    for n, p in zip(names, params):
        assert float((p.grad - g_e[n]).abs().max()) <= 1e-5 * (float(g_e[n].abs().max()) + 1e-8), n
