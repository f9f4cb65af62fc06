"""The inputs of the tests that compare with tests/golden/ref_*.npz, in one place: oracle/make_golden_ref.py runs the
reference on exactly these, and the tests run the port / the product on them.  Change an input here and regenerate the
fixtures (python oracle/build_ref.py && python -m oracle.make_golden_ref)."""
import functools
import json
import os

import numpy as np
import torch

from humor_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@functools.lru_cache(maxsize=None)
def fixture(name):
    """tests/golden/<name>.npz as a dict (loaded when a test first asks for it)."""
    return dict(np.load(os.path.join(GOLDEN, name + '.npz')))


# ------------------------------------------------------------------------------- Stage-III closure (tests/test_oracle.py)
STAGE3_SEED31 = [(True, None, 1.0), (True, 5, 1.0), (False, None, 2.4)]     # (optim_floor, nsteps, scale)


def stage3_name(optim_floor, nsteps, scale):
    return 'ref_stage3_seed31_%s%s%s' % ('rgb' if optim_floor else 'amass', '_n%d' % nsteps if nsteps else '',
                                         '_s%g' % scale if scale != 1.0 else '')


def stage3_case(optim_floor):
    """(B, T, weights, problem): the seeded synthetic problem as generated, observations included.  B = 4, not 3: see
    oracle/make_golden.py (torch.cross default-dim quirk of the reference)."""
    B, T = 4, 9
    W = synth.RGB_STAGE3_WEIGHTS if optim_floor else synth.AMASS_STAGE3_WEIGHTS
    return B, T, W, synth.make_stage3_problem(B, T, seed=31, overlap=3, cam=optim_floor)


# --------------------------------------------------------------------------- rotation helpers (tests/test_oracle.py)
def rotation_inputs():
    return torch.randn(500, 3, generator=torch.Generator().manual_seed(0)) * 1.3


# ------------------------------------------------------------------------------ on-disk formats (tests/test_io_formats.py)
KEYPOINT_FRAMES = 6
SPLITS = [(300, 60, 10), (301, 60, 10), (125, 60, 10), (1000, 60, 10), (77, 30, 5), (61, 60, 10)]
SAVE_CASES = [('RGB', False), ('AMASS', True), ('PROX-RGBD', True)]
STITCHED_FILES = ('gt_results.npz', 'observations.npz', 'stage3_results.npz')


def write_openpose_dir(path, T, seed=0, empty=(3,)):
    rng = np.random.RandomState(seed)
    os.makedirs(path, exist_ok=True)
    frames = []
    for t in range(T):
        kp = np.concatenate([rng.rand(25, 2) * 1000, rng.rand(25, 1)], 1)
        people = [] if t in empty else [{'pose_keypoints_2d': kp.reshape(-1).tolist()},
                                        {'pose_keypoints_2d': (kp * 0.5).reshape(-1).tolist()}]    # 2nd person ignored
        with open(os.path.join(path, 'frame_%06d_keypoints.json' % t), 'w') as f:
            json.dump({'version': 1.3, 'people': people}, f)
        frames.append(np.zeros((25, 3)) if t in empty else kp)
    return np.stack(frames, 0)


def fake_results(B, T, rng):
    t = lambda *s: torch.tensor(rng.randn(*s).astype(np.float32))
    optim = {'betas': t(B, 16), 'trans': t(B, T, 3), 'root_orient': t(B, T, 3), 'pose_body': t(B, T, 63),
             'latent_pose': t(B, T, 32), 'latent_motion': t(B, T - 1, 48), 'contacts': (t(B, T, 22) > 0).float(),
             'floor_plane': t(B, 4)}
    stages = {'stage3': {'prior_trans': t(B, T, 3), 'prior_root_orient': t(B, T, 3)}}
    obs = {'joints2d': t(B, T, 25, 3), 'floor_plane': t(B, 4), 'seq_interval': torch.tensor([[i * (T - 3), i * (T - 3) + T] for i in range(B)], dtype=torch.int)}
    gt = {'cam_matx': t(B, 3, 3), 'name': ['v_%04d' % i for i in range(B)]}
    return optim, stages, obs, gt


def image_paths(B, T):
    return [tuple('f%d_b%d.png' % (t, b) for b in range(B)) for t in range(T)]


def save_case(data_type, with_smpl_gt):
    """(optim, stages, gt, obs, img, B) handed to save_optim_result(..., data_type, optim_floor=True, obs_img_paths=img)."""
    rng = np.random.RandomState(0)
    B, T = 3, 7
    optim, stages, obs, gt = fake_results(B, T, rng)
    if with_smpl_gt:
        g = lambda *s: torch.tensor(rng.randn(*s).astype(np.float32))
        gt.update(betas=g(B, 16) if data_type.startswith('PROX') else g(B, T, 16), trans=g(B, T, 3), root_orient=g(B, T, 3),
                  pose_body=g(B, T, 63), contacts=g(B, T, 22))
    return optim, stages, gt, obs, image_paths(B, T), B


def stitched_case():
    """(optim, stages, gt, obs, img, B): per-sequence results whose stitched final_results/ the test compares."""
    rng = np.random.RandomState(1)
    B, T = 3, 8
    optim, stages, obs, gt = fake_results(B, T, rng)
    optim['floor_plane'] = torch.tensor([[0.0, -1.0, 0.05, -0.6]] * B)
    optim['trans'][..., 2] += 3.0
    return optim, stages, gt, obs, image_paths(B, T), B


def ref_digests(prefix):
    """The digests (tests/golden_util.npz_digests) stored in ref_io_formats.npz under `prefix`, with the prefix removed."""
    lines = fixture('ref_io_formats')['digests'].item().decode().splitlines()
    return {k[len(prefix):]: v for k, v in (line.split('\t') for line in lines) if k.startswith(prefix)}


# ------------------------------------------------------------------------ chamfer module (CPU and GPU chamfer tests)
CHAMFER_RANDOM = [(1, 1, 1), (2, 5, 3), (3, 129, 1025), (1, 700, 2)]


def chamfer_random_cases():
    """(b, n, m, xyz1, xyz2, grad_dist1, grad_dist2) for every shape of CHAMFER_RANDOM, drawn from one seeded stream."""
    rng = np.random.default_rng(7)
    for b, n, m in CHAMFER_RANDOM:
        a = rng.normal(size=(b, n, 3)).astype(np.float32)
        c = rng.normal(size=(b, m, 3)).astype(np.float32)
        gd1 = rng.normal(size=(b, n)).astype(np.float32)
        gd2 = rng.normal(size=(b, m)).astype(np.float32)
        yield b, n, m, a, c, gd1, gd2


def chamfer_gpu_case():
    """(xyz1, xyz2) of the GPU test against the reference's forward: larger clouds than the CPU cases."""
    rng = np.random.default_rng(11)
    return rng.normal(size=(4, 600, 3)).astype(np.float32), rng.normal(size=(4, 1500, 3)).astype(np.float32)
