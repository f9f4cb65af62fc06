"""CPU tests that pin the oracle: (1) the torch port against the committed fixtures produced by the REAL reference
(oracle/make_golden.py, oracle/make_golden_ref.py); (2) analytic known answers for the restated smplx LBS (no runnable
third-party source exists: LBS parity is pinned only here)."""
import numpy as np
import pytest
import torch

from humor_b200 import synth
from tests import ref_inputs as R
from tests import util_stage3 as U
from tests.golden_util import CASES, load_case, check_against_golden


@pytest.mark.parametrize('name', CASES)
def test_port_matches_reference_golden(name):
    g, prob, c = load_case(name)
    port = U.build_port(c['B'], c['T'], c['W'], c['optim_floor'], prob)
    loss, grads, aux = U.closure_port(port, prob, c['optim_floor'], c['nsteps'], c['scale'])
    check_against_golden(g, loss, aux['stats'], grads, loss_tol=2e-6, stat_tol=2e-5, grad_tol=1e-4)
    inter = aux['inter']
    assert np.abs(inter['cam_pred']['verts3d'].detach().numpy() - g['cam_verts3d']).max() < 1e-5
    assert np.abs(inter['rollout']['trans'].detach().numpy() - g['rollout_trans']).max() < 1e-5
    assert np.abs(inter['rollout']['cond_prior'][0].detach().numpy() - g['cond_prior_mean']).max() < 1e-5


@pytest.mark.parametrize('name', ['stage1_rgb', 'stage2_rgb', 'stage2_amass', 'stage2_proxd'])
def test_port_stage12_matches_reference_golden(name):
    """Stage-I (root_fit) / Stage-II (smpl_fit) closures of the port against fixtures of the unmodified reference."""
    from tests.golden_util import load_case12
    g, c = load_case12(name)
    port = U.build_port(c['B'], c['T'], c['W3'], c['optim_floor'], {'cam_mat': c['cam_mat']})
    names = ['trans', 'root_orient'] + (['betas', 'latent_pose'] if c['stage'] == 1 else [])
    p = {k: torch.as_tensor(v).clone().requires_grad_(k in names) for k, v in c['params'].items()}
    obs = {k: torch.as_tensor(v).clone() for k, v in c['obs'].items()}
    loss, stats, inter = port.closure12(p, obs, c['stage'], c['W12'])
    loss.backward()
    st = {k: float(v.detach()) if torch.is_tensor(v) else float(v) for k, v in stats.items()}
    check_against_golden(g, float(loss.detach()), st, {k: p[k].grad for k in names}, loss_tol=2e-6, stat_tol=2e-5, grad_tol=1e-4)
    assert np.abs(inter['pred']['verts3d'].detach().numpy() - g['pred_verts3d']).max() < 1e-5


@pytest.mark.parametrize('optim_floor,nsteps,scale', R.STAGE3_SEED31)
def test_port_matches_live_reference(optim_floor, nsteps, scale):
    """Loss, every energy term and every gradient of the port against the reference's Stage-III closure on the seeded
    synthetic problem as generated (observations included), stored by oracle/make_golden_ref.py (the name dates from when
    the reference was executed inside the test)."""
    g = R.fixture(R.stage3_name(optim_floor, nsteps, scale))
    B, T, W, prob = R.stage3_case(optim_floor)
    port = U.build_port(B, T, W, optim_floor, prob)
    l2, g2, aux = U.closure_port(port, prob, optim_floor, nsteps, scale)
    assert sorted(k[5:] for k in g if k.startswith('grad_')) == sorted(g2)
    check_against_golden(g, l2, aux['stats'], g2, loss_tol=2e-6, stat_tol=2e-5, grad_tol=1e-4)


def test_reference_rotation_helpers_match_port():
    """Port rotation helpers against the reference's batch_rodrigues / rotation_matrix_to_angle_axis /
    compute_world2aligned_mat on 500 seeded axis-angle vectors (stored by oracle/make_golden_ref.py)."""
    from oracle.stage3_port import mat2aa, world2aligned
    from oracle.smplh_lbs import rodrigues
    g = R.fixture('ref_rotations')
    aa = R.rotation_inputs()
    assert torch.equal(aa, torch.from_numpy(g['aa']))         # the fixture was made from these inputs
    rot = torch.from_numpy(g['rodrigues'])
    assert torch.allclose(rodrigues(aa), rot, atol=1e-6)
    assert torch.allclose(mat2aa(rot), torch.from_numpy(g['mat2aa']), atol=1e-6)
    assert torch.allclose(world2aligned(rot), torch.from_numpy(g['world2aligned']), atol=1e-6)


# ------------------------------------------------------------------------------------------------ LBS known answers
@pytest.fixture(scope='module')
def smpl():
    from oracle.smplh_lbs import SMPLHOracle
    asset = synth.make_smplh_asset()
    return asset, SMPLHOracle(asset, dtype=torch.float64)


def test_lbs_zero_pose_is_template(smpl):
    asset, m = smpl
    tr = torch.tensor([[0.3, -0.1, 2.0]], dtype=torch.float64)
    v, J, _ = m.forward(torch.zeros(1, 16, dtype=torch.float64), torch.zeros(1, 3, dtype=torch.float64),
                        torch.zeros(1, 63, dtype=torch.float64), tr)
    vt = torch.tensor(asset['v_template'], dtype=torch.float64)
    assert (v[0] - (vt + tr)).abs().max() < 3e-7     # rodrigues(0) == I; skinning rows sum to 1 only to fp32 rounding
    Jr = torch.tensor(asset['J_regressor'], dtype=torch.float64) @ vt
    assert (J[0, :52] - (Jr + tr)).abs().max() < 1e-9
    assert J.shape == (1, 73, 3)


def test_lbs_root_rotation_is_rigid_about_root_joint(smpl):
    asset, m = smpl
    from oracle.smplh_lbs import rodrigues
    beta = torch.randn(1, 16, dtype=torch.float64) * 0.5
    aa = torch.tensor([[0.3, -1.1, 0.7]], dtype=torch.float64)
    z63, z3 = torch.zeros(1, 63, dtype=torch.float64), torch.zeros(1, 3, dtype=torch.float64)
    v0, J0, _ = m.forward(beta, z3, z63, z3)
    v1, J1, _ = m.forward(beta, aa, z63, z3)
    R = rodrigues(aa)[0]
    root = J0[0, 0]
    assert ((v0[0] - root) @ R.T + root - v1[0]).abs().max() < 1e-6    # weights sum to 1 to fp32 rounding
    assert ((J0[0] - root) @ R.T + root - J1[0]).abs().max() < 1e-6


def test_lbs_hand_columns_of_posedirs_are_dead(smpl):
    asset, _ = smpl
    from oracle.smplh_lbs import SMPLHOracle
    a2 = dict(asset)
    pd = asset['posedirs'].copy()
    pd[:, :, 189:] = 123.0
    a2['posedirs'] = pd
    m1, m2 = SMPLHOracle(asset, dtype=torch.float64), SMPLHOracle(a2, dtype=torch.float64)
    g = torch.Generator().manual_seed(0)
    args = (torch.randn(2, 16, generator=g, dtype=torch.float64), torch.randn(2, 3, generator=g, dtype=torch.float64),
            torch.randn(2, 63, generator=g, dtype=torch.float64) * 0.4, torch.randn(2, 3, generator=g, dtype=torch.float64))
    assert (m1.forward(*args)[0] - m2.forward(*args)[0]).abs().max() < 1e-6


def test_pack_smplh_reproduces_dense_operators():
    """host packing logic (ELL skinning weights, fused blend matrix, joint regressor folding)."""
    from humor_b200.body_model import pack_smplh
    asset = synth.make_smplh_asset()
    p = pack_smplh(asset)
    V = 6890
    W = np.zeros((V, 52), np.float32)
    np.add.at(W, (np.repeat(np.arange(V), p['wk']), p['w_idx'].reshape(-1)), p['w_val'].reshape(-1))
    assert np.abs(W - asset['weights']).max() == 0.0 and p['wk'] <= 4
    assert np.abs(p['blend'][:16, :3 * V].T.reshape(V, 3, 16) - asset['shapedirs']).max() == 0.0
    assert np.abs(p['blend'][16:205, :3 * V].T.reshape(V, 3, 189) - asset['posedirs'][:, :, :189]).max() == 0.0
    assert (p['blend'][205:] == 0).all() and (p['blend_t'] == p['blend'].T).all()
    beta = np.random.RandomState(0).randn(16).astype(np.float32)
    J = asset['J_regressor'] @ (asset['v_template'] + asset['shapedirs'] @ beta)
    assert np.abs(p['j_template'].reshape(52, 3) + (p['j_dirs'] @ beta).reshape(52, 3) - J).max() < 2e-6
    assert p['parents'][0] == -1 and (p['parents'][1:] < np.arange(1, 52)).all()
