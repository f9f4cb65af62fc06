"""On-disk formats (humor_b200/io_formats.py) against what the reference's own readers/writers produced on the same
inputs (tests/golden/ref_io_formats.npz, written by oracle/make_golden_ref.py from the inputs of tests/ref_inputs.py) and
against known answers.  CPU only."""
import os

import numpy as np
import pytest
import torch

from humor_b200 import io_formats as F
from tests import ref_inputs as R
from tests.golden_util import npz_digests
from tests.ref_inputs import write_openpose_dir


def test_read_keypoints_known_answer(tmp_path):
    kp = write_openpose_dir(str(tmp_path), 5)
    for t, p in enumerate(F.keypoint_paths(str(tmp_path))):
        got = F.read_keypoints(p)
        assert got.shape == (25, 3) and got.dtype == np.float64
        assert np.array_equal(got, kp[t])


def test_read_keypoints_matches_reference(tmp_path):
    """fitting_utils.read_keypoints's arrays for the same OpenPose files (one frame without a person)."""
    want = R.fixture('ref_io_formats')['read_keypoints']
    write_openpose_dir(str(tmp_path), R.KEYPOINT_FRAMES)
    got = np.stack([F.read_keypoints(p) for p in F.keypoint_paths(str(tmp_path))])
    assert got.dtype == want.dtype and np.array_equal(got, want)


@pytest.mark.parametrize('F_,L,o', R.SPLITS)
def test_split_intervals_matches_reference(F_, L, o):
    """The windows and overlap of the reference's RGB-video split (rgb_dataset.py:74-99)."""
    ref = R.fixture('ref_io_formats')
    got, ov = F.split_intervals(F_, L, o)
    want = [tuple(int(x) for x in r) for r in ref['split:%d:%d:%d' % (F_, L, o)]]
    assert got == want and ov == int(ref['split_overlap:%d:%d:%d' % (F_, L, o)])


def test_split_intervals_properties():
    for Fr, L, o in [(300, 60, 10), (301, 60, 10), (999, 60, 10), (125, 60, 10)]:
        iv, ov = F.split_intervals(Fr, L, o)
        assert iv[0][0] == 0 and all(e - s == L for s, e in iv)
        assert iv[-1][1] >= Fr and iv[-1][0] < Fr                         # covers the video, last window not empty
        assert all(iv[i][1] - iv[i + 1][0] >= o for i in range(len(iv) - 1))   # at least the requested overlap
    assert F.split_intervals(50, None, None)[0] == [(0, 50)]


def test_load_rgb_video(tmp_path):
    kp = write_openpose_dir(str(tmp_path / 'op'), 40)
    cam = np.array([[1060.5, 0, 951.3], [0, 1060.4, 536.8], [0, 0, 1]])
    obs, gt = F.load_rgb_video(str(tmp_path / 'op'), cam, seq_len=16, overlap_len=4)
    iv = obs['seq_interval']
    assert obs['joints2d'].dtype == np.float32 and obs['joints2d'].shape == (len(iv), 16, 25, 3)
    for b, (s, e) in enumerate(iv):
        assert np.allclose(obs['joints2d'][b], kp[s:e].astype(np.float32))
    assert np.array_equal(obs['floor_plane'][0], np.array(F.DEFAULT_GROUND)) and gt['cam_matx'].shape == (len(iv), 3, 3)
    assert gt['name'][1] == 'rgb_video_0001'


@pytest.mark.parametrize('data_type,with_smpl_gt', R.SAVE_CASES)
def test_save_optim_result_matches_reference(tmp_path, data_type, with_smpl_gt):
    """Every file fitting_utils.save_optim_result writes for these inputs: same files, keys, dtypes and bytes."""
    optim, stages, gt, obs, img, B = R.save_case(data_type, with_smpl_gt)
    dirs = [str(tmp_path / ('s%d' % b)) for b in range(B)]
    for d in dirs:
        os.makedirs(d)
    F.save_optim_result(dirs, optim, stages, gt, obs, data_type, optim_floor=True, obs_img_paths=img)
    want = R.ref_digests('save:%s:' % data_type)
    got = npz_digests(str(tmp_path))
    assert sorted(got) == sorted(want)
    for k in want:
        assert got[k] == want[k], k


def test_stitched_result_matches_reference(tmp_path):
    """final_results/ against what the reference's save_rgb_stitched_result wrote from the same per-sequence files (run with
    its own BodyModel, restated smplx behind it, for the prior-frame copy); the files that do not depend on SMPL must be
    identical."""
    from oracle.ref_closure import asset_npz
    optim, stages, gt, obs, img, B = R.stitched_case()
    dirs = [str(tmp_path / ('s%d' % b)) for b in range(B)]
    for d in dirs:
        os.makedirs(d)
    F.save_optim_result(dirs, optim, stages, gt, obs, 'RGB', obs_img_paths=img)
    F.write_meta(dirs, asset_npz())
    iv = [tuple(int(x) for x in r) for r in obs['seq_interval']]
    F.save_rgb_stitched_result(iv, dirs, str(tmp_path))
    final = str(tmp_path / 'final_results')
    want = R.ref_digests('stitched:')
    got = npz_digests(final, R.STITCHED_FILES)
    assert sorted(got) == sorted(want)
    for k in want:
        assert got[k] == want[k], k
    assert open(os.path.join(final, 'meta.txt')).read() == R.fixture('ref_io_formats')['stitched_meta'].item().replace('<asset>', asset_npz())
    st = F.stitch_subsequences(iv, dirs)
    assert st['trans'].shape[0] == iv[-1][1] and st['joints2d'].shape[0] == iv[-1][1] and len(st['img_paths']) == iv[-1][1]


def test_gmm_and_checkpoint_loaders(tmp_path):
    rng = np.random.RandomState(2)
    np.savez(str(tmp_path / 'prior_gmm.npz'), weights=rng.rand(12), means=rng.randn(12, 138), covariances=rng.randn(12, 138, 138))
    w, m, c = F.load_gmm(str(tmp_path))
    assert w.dtype == np.float32 and m.shape == (12, 138) and c.shape == (12, 138, 138)
    with pytest.raises(FileNotFoundError):
        F.load_gmm(str(tmp_path / 'nope'))
    net = torch.nn.Linear(3, 2)
    sd = {'module.' + k: v + 1 for k, v in net.state_dict().items()}          # saved under DataParallel
    torch.save({'model': sd, 'optim': {}, 'epoch': 7, 'min_val_loss': 0.5}, str(tmp_path / 'ck.pth'))
    ep, mv, mt = F.load_state(str(tmp_path / 'ck.pth'), net, map_location='cpu')
    assert ep == 7 and mv == 0.5 and mt == float('Inf')
    assert torch.equal(net.weight, sd['module.weight'])
