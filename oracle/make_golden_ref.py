"""ORACLE (test infrastructure) — writes the tests/golden/ref_*.npz fixtures by running the UNMODIFIED reference
(/root/reference, build container only; the chamfer part needs oracle/_ref/cd_ref.so from oracle/build_ref.py) on the
inputs of tests/ref_inputs.py, which the tests that compare with the fixtures use as well:

    ref_stage3_seed31_*.npz   Stage-III closure (loss, energy terms, gradients)   tests/test_oracle.py
    ref_rotations.npz         rotation helpers of utils/transforms.py             tests/test_oracle.py
    ref_io_formats.npz        readers / writers of fitting_utils.py (written files as digests, see
                              tests/golden_util.npz_digests), rgb_dataset.py interval split      tests/test_io_formats.py
    ref_chamfer_random.npz    compiled chamfer module, CPU tests' random clouds   tests/test_oracle_chamfer.py
    ref_chamfer_gpu.npz       compiled chamfer module, GPU test's random clouds   tests/test_gpu_zz_chamfer.py

    python oracle/build_ref.py && python -m oracle.make_golden_ref
"""
import contextlib
import io
import os
import sys
import tempfile
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402
from tests import ref_inputs as R  # noqa: E402
from tests.golden_util import npz_digests  # noqa: E402

OUT = R.GOLDEN


def stage3_seed31():
    from oracle import ref_closure
    from tests import util_stage3 as U
    for optim_floor, nsteps, scale in R.STAGE3_SEED31:
        B, T, W, prob = R.stage3_case(optim_floor)
        ref, mo, _, _ = ref_closure.build(B, T, W, optim_floor, prob['cam_mat'] if optim_floor else None)
        names = ref_closure.set_params(mo, prob['params'])
        obs = {k: torch.as_tensor(prob['obs'][k]) for k in U.obs_keys(optim_floor)}
        loss, stats, _ = ref_closure.stage3_closure(ref, mo, {k: v.clone() for k, v in obs.items()}, nsteps, scale)
        out = {'loss': np.float64(loss.item())}
        out.update({'stat_' + k: np.float64(float(v)) for k, v in stats.items()})
        out.update({'grad_' + n: getattr(mo, n).grad.numpy() for n in names})
        np.savez_compressed(os.path.join(OUT, R.stage3_name(optim_floor, nsteps, scale) + '.npz'), **out)


def rotations():
    ref = ref_import.load()
    aa = R.rotation_inputs()
    rot = ref.transforms.batch_rodrigues(aa)
    np.savez_compressed(os.path.join(OUT, 'ref_rotations.npz'), aa=aa.numpy(), rodrigues=rot.numpy(),
                        mat2aa=ref.transforms.rotation_matrix_to_angle_axis(rot).numpy(),
                        world2aligned=ref.transforms.compute_world2aligned_mat(rot).numpy())


def ref_mods():
    ref = ref_import.load()
    np.float = float                     # the reference predates numpy 1.24 (fitting_utils.py:30,33-34)
    return ref


def reference_intervals(num_frames, seq_len, overlap_len):
    """rgb_dataset.py:74-99 executed literally (the module itself needs cv2, which this image lacks)."""
    import math
    src = open(os.path.join(ref_import.REF_ROOT, 'datasets', 'rgb_dataset.py')).read().splitlines()
    a = next(i for i, l in enumerate(src) if l.strip() == 'seq_intervals = []')
    b = next(i for i, l in enumerate(src) if l.strip() == 'seq_intervals = [(0, self.seq_len)]')
    body = '\n'.join(l[8:] for l in src[a:b + 1])          # rgb_dataset.py:74-99
    ns = types.SimpleNamespace(seq_len=seq_len, overlap_len=overlap_len)
    env = {'self': ns, 'num_frames': num_frames, 'math': math, 'print': lambda *a, **k: None}
    exec(body, env)
    return [tuple(x) for x in env['seq_intervals']], ns.overlap_len


def seq_dirs(root, B):
    dirs = [os.path.join(root, 's%d' % b) for b in range(B)]
    for d in dirs:
        os.makedirs(d)
    return dirs


def io_formats():
    from humor_b200 import io_formats as F
    ref = ref_mods()
    out, digests = {}, {}
    with tempfile.TemporaryDirectory() as tmp:
        R.write_openpose_dir(os.path.join(tmp, 'op'), R.KEYPOINT_FRAMES)
        out['read_keypoints'] = np.stack([ref.fitting_utils.read_keypoints(p) for p in F.keypoint_paths(os.path.join(tmp, 'op'))])
    for F_, L, o in R.SPLITS:
        iv, ov = reference_intervals(F_, L, o)
        out['split:%d:%d:%d' % (F_, L, o)] = np.array(iv, np.int64)
        out['split_overlap:%d:%d:%d' % (F_, L, o)] = np.int64(ov)
    for data_type, with_smpl_gt in R.SAVE_CASES:
        optim, stages, gt, obs, img, B = R.save_case(data_type, with_smpl_gt)
        with tempfile.TemporaryDirectory() as tmp:
            ref.fitting_utils.save_optim_result(seq_dirs(tmp, B), optim, stages, gt, obs, data_type, optim_floor=True, obs_img_paths=img)
            for k, v in npz_digests(tmp).items():
                digests['save:%s:%s' % (data_type, k)] = v
    sys.modules.setdefault('cv2', types.ModuleType('cv2'))       # imported, never used, by the reference function
    from oracle.ref_closure import asset_npz
    optim, stages, gt, obs, img, B = R.stitched_case()
    with tempfile.TemporaryDirectory() as tmp:
        dirs = seq_dirs(tmp, B)
        F.save_optim_result(dirs, optim, stages, gt, obs, 'RGB', obs_img_paths=img)
        F.write_meta(dirs, asset_npz())
        iv = [tuple(int(x) for x in r) for r in obs['seq_interval']]
        with contextlib.redirect_stdout(io.StringIO()):
            ref.fitting_utils.save_rgb_stitched_result(iv, dirs, tmp, torch.device('cpu'), asset_npz(), 16, True)
        final = os.path.join(tmp, 'final_results')
        for k, v in npz_digests(final, R.STITCHED_FILES).items():
            digests['stitched:' + k] = v
        # the body-model path written into meta.txt is a temporary file of the machine that runs the test
        out['stitched_meta'] = np.array(open(os.path.join(final, 'meta.txt')).read().replace(asset_npz(), '<asset>'))
    out['digests'] = np.bytes_(''.join('%s\t%s\n' % kv for kv in sorted(digests.items())))
    np.savez_compressed(os.path.join(OUT, 'ref_io_formats.npz'), **out)


def _chamfer(cd, a, c, gd1=None, gd2=None):
    b, n, m = a.shape[0], a.shape[1], c.shape[1]
    d1, d2 = torch.zeros(b, n), torch.zeros(b, m)
    i1, i2 = torch.zeros(b, n, dtype=torch.int), torch.zeros(b, m, dtype=torch.int)
    cd.forward(torch.from_numpy(a), torch.from_numpy(c), d1, d2, i1, i2)
    res = {'dist1': d1.numpy(), 'dist2': d2.numpy(), 'idx1': i1.numpy(), 'idx2': i2.numpy()}
    if gd1 is not None:
        g1, g2 = torch.zeros(b, n, 3), torch.zeros(b, m, 3)
        cd.backward(torch.from_numpy(a), torch.from_numpy(c), g1, g2, torch.from_numpy(gd1), torch.from_numpy(gd2), i1, i2)
        res.update(grad_xyz1=g1.numpy(), grad_xyz2=g2.numpy())
    return res


def chamfer():
    from oracle.build_ref import load_cd_ref
    cd = load_cd_ref()
    if cd is None:
        raise SystemExit('oracle/_ref/cd_ref.so missing: run python oracle/build_ref.py first')
    out = {}
    for b, n, m, a, c, gd1, gd2 in R.chamfer_random_cases():
        for k, v in _chamfer(cd, a, c, gd1, gd2).items():
            out['%d_%d_%d:%s' % (b, n, m, k)] = v
    np.savez_compressed(os.path.join(OUT, 'ref_chamfer_random.npz'), **out)
    np.savez_compressed(os.path.join(OUT, 'ref_chamfer_gpu.npz'), **_chamfer(cd, *R.chamfer_gpu_case()))


def main():
    torch.set_num_threads(8)
    stage3_seed31()
    rotations()
    io_formats()
    chamfer()


if __name__ == '__main__':
    main()
