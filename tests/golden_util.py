import hashlib
import os
import numpy as np
from humor_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def npz_digests(root, names=None):
    """{'<dir relative to root>:<file>:<key>': 'dtype shape sha256'} of every array in the npz files under `root` (or of the
    files `names` in `root`): two trees have equal digests exactly when they hold the same files, keys, dtypes and bytes."""
    out = {}
    for d, _, files in os.walk(root):
        for fn in sorted(files):
            if fn.endswith('.npz') and (names is None or (d == root and fn in names)):
                z = np.load(os.path.join(d, fn))
                for k in z.files:
                    a = np.ascontiguousarray(z[k])
                    key = ':'.join(([] if names is not None else [os.path.relpath(d, root)]) + [fn, k])
                    out[key] = '%s %s %s' % (a.dtype.str, a.shape, hashlib.sha256(a.tobytes()).hexdigest())
    return out
CASES = ['stage3_rgb', 'stage3_rgb_phase1', 'stage3_rgb_refine', 'stage3_amass', 'stage3_proxd', 'stage3_rgb_xbatch']


def load_case(name):
    g = dict(np.load(os.path.join(GOLDEN, name + '.npz')))
    B, T, seed, overlap, nsteps, of = [int(x) for x in g['meta']]
    optim_floor = bool(of)
    prob = synth.make_stage3_problem(B, T, seed=seed, overlap=overlap, cam=optim_floor)
    for k in g:
        if k.startswith('obs_prevres_'):          # observed_data['prev_batch_overlap_res'] (run_fitting.py:428-435)
            prob['obs'].setdefault('prev_batch_overlap_res', {})[k[12:]] = g[k]
        elif k.startswith('obs_'):
            prob['obs'][k[4:]] = g[k]
    W = synth.RGB_STAGE3_WEIGHTS if optim_floor else synth.AMASS_STAGE3_WEIGHTS
    if 'wset' in g:
        W = synth.WEIGHT_SETS[str(g['wset'])]
    return g, prob, dict(B=B, T=T, optim_floor=optim_floor, nsteps=None if nsteps < 0 else nsteps, scale=float(g['scale']), W=W)


def check_against_golden(g, loss, stats, grads, loss_tol=2e-5, stat_tol=2e-4, grad_tol=2e-3):
    assert abs(loss - float(g['loss'])) <= loss_tol * max(1.0, abs(float(g['loss']))), (loss, float(g['loss']))
    for k in g:
        if k.startswith('stat_'):
            v = float(g[k])
            assert k[5:] in stats, k
            assert abs(stats[k[5:]] - v) <= stat_tol * max(1.0, abs(v)), (k, stats[k[5:]], v)
        if k.startswith('grad_'):
            ref = g[k]
            got = np.asarray(grads[k[5:]].cpu() if hasattr(grads[k[5:]], 'cpu') else grads[k[5:]])
            err = np.abs(got - ref).max() / (np.abs(ref).max() + 1e-8)
            assert err < grad_tol, (k, err)


CASES12 = ['stage1_rgb', 'stage2_rgb', 'stage2_amass', 'stage2_proxd']


def load_case12(name):
    """Stage-I/II fixtures of oracle/make_golden.py (run_case12): observations from the file, variables from the seed."""
    g = dict(np.load(os.path.join(GOLDEN, name + '.npz')))
    B, T, seed, overlap, stage, of = [int(x) for x in g['meta']]
    prob = synth.make_stage3_problem(B, T, seed=seed, overlap=overlap, cam=bool(of))
    obs = {k[4:]: g[k] for k in g if k.startswith('obs_')}
    wset = str(g['wset'])
    return g, dict(B=B, T=T, stage=stage, optim_floor=bool(of), wset=wset, W12=synth.stage12_weights(wset),
                   W3=synth.WEIGHT_SETS[wset], obs=obs, params=synth.make_stage12_params(B, T, seed=seed + 1), cam_mat=prob['cam_mat'])


STAGE_FILES = ('stage1_results', 'stage2_results', 'stage3_init_results', 'stage3_init_results_prior', 'stage2_results_prior')


def make_stage_dirs(root, B):
    """One output directory per sub-sequence, as run_fitting.py hands them to MotionOptimizer.run(stages_res_out=...)."""
    import os
    dirs = [os.path.join(str(root), str(i)) for i in range(B)]
    for d in dirs:
        os.makedirs(d, exist_ok=True)
    return dirs


def collect_stage_files(dirs):
    """The per-stage npz dumps of run() as {'file_<name>_<key>': (B, ...)} - the layout oracle/make_golden_run.py stores."""
    import os
    import numpy as np
    out = {}
    for f in STAGE_FILES:
        per = [np.load(os.path.join(d, f + '.npz')) for d in dirs]
        for k in per[0].files:
            out['file_%s_%s' % (f, k)] = np.stack([q[k] for q in per], 0)
    return out
