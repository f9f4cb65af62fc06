#!/usr/bin/env python
"""Benchmark of the HuMoR Stage-III optimiser step (BASELINE.json metric: frames/sec = B*T / t_closure).

One *step* = one full-T Stage-III closure: forward (VPoser decode -> cam2prior -> CVAE rollout -> SMPL+H LBS ->
fitting energies) + backward to every optimisation variable (reference: humor/fitting/motion_optimizer.py:514-608).
Workload at N=1: the configuration the target is quoted on, B x T = 256 x 60, RGB config (optim_floor,
stage-3 weights of configs/fit_rgb_demo_use_split.cfg), synthetic seeded inputs (no licensed assets exist offline).

    python bench.py --gpus N --steps K --warmup W            # this repo's arm
    python bench.py --impl reference ...                     # the reference algorithm on the host CPUs (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step returned, as DIR/*.npy
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from humor_b200 import synth  # noqa: E402

LBS_BYTES_FWD = 83896          # SURVEY.md §8(d): per frame, fwd (inputs + v + Jtr)
LBS_BYTES_BWD = 84236
METRIC = 'stage3_optimizer_step_frames_per_sec'
DUMP_LIMIT_BYTES = 64_000_000
NPY_HEADER_BYTES = 128          # np.save's header for arrays of up to four dimensions


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d['hbm_gbs'], d.get('bf16_tflops', 1590.0), 'measured'
    return 6650.0, 1590.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self, first_row=0, timed_rows=None):
        """Statistics over the rows sampled from `first_row` on (the caller passes the row count at the start of the timed region)."""
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.05)
        self.proc.terminate()
        rows = self.rows[first_row:]
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith('active') for r in rows)]
        out = {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons, 'samples': len(sm)}
        if timed_rows is not None:
            out['samples_in_timed_region'] = timed_rows
        return out


CONFIGS = {
    # BASELINE.json configs[2] / [3]: fit_rgb_demo_use_split stage-3 weights, optim_floor, 2-D keypoints + overlap consistency
    'rgb': dict(optim_floor=True, weights='RGB_STAGE3_WEIGHTS', obs=('joints2d', 'floor_plane', 'seq_interval'),
                what='RGB config (optim_floor, fit_rgb_demo_use_split stage-3 weights, rgb_overlap_consist 200, overlap 10)'),
    # BASELINE.json configs[4]: fit_amass_keypts - 3-D key vertices with occlusions (inf), no floor optimisation
    'amass': dict(optim_floor=False, weights='AMASS_STAGE3_WEIGHTS', obs=('verts3d',),
                  what='AMASS key-vertex config (fit_amass_keypts stage-3 weights, verts3d observations with inf-masked occlusions, no floor)'),
}


def build_problem(B, T, seed=4, config='rgb'):
    return synth.make_stage3_problem(B, T, seed=seed, overlap=10, cam=CONFIGS[config]['optim_floor'])


def workload_config(args, world):
    """The `config` object both arms print: what is computed, not how."""
    c = CONFIGS[args.config]
    return {'workload': f'Stage-III full-T closure fwd+bwd, B={args.batch} sub-sequences/GPU x T={args.seq_len}, {c["what"]}',
            'config_name': args.config, 'batch_per_gpu': args.batch, 'seq_len': args.seq_len,
            'parallelism': f'dp{world} over sub-sequences',
            'l2': 'working set per step (rollout tape + dense vertices, > 1 GB at B=256) exceeds the 126 MB L2'}


def make_optimizer(B, T, prob, dev, config='rgb'):
    from humor_b200.body_model import BodyModel
    from humor_b200.humor_model import HumorModel
    from humor_b200.motion_optimizer import MotionOptimizer
    cfg = CONFIGS[config]
    of = cfg['optim_floor']
    bm = BodyModel(synth.make_smplh_asset(), num_betas=16, batch_size=B * T, use_vtx_selector=of).to(dev)
    humor = HumorModel(in_rot_rep='mat', out_rot_rep='aa', latent_size=48, model_data_config='smpl+joints+contacts', steps_in=1)
    humor.load_state_dict(synth.make_humor_state_dict())
    humor.to(dev).eval()
    gmm = tuple(g.to(dev) for g in synth.make_gmm())
    w = dict(getattr(synth, cfg['weights']))
    mo = MotionOptimizer(dev, bm, 16, B, T, list(cfg['obs']), [dict(w), dict(w), dict(w)],
                         synth.FakeVPoser().to(dev), humor, {'gmm': gmm}, of, torch.as_tensor(prob['cam_mat']).to(dev) if of else None,
                         'bisquare', 4.6851, 100.0)
    mo.fitting_loss.assume_unit_grad = True
    return mo


OBS_KEYS = ('joints2d', 'floor_plane', 'seq_interval')


def project_obs(prob, config='rgb'):
    """Informative observations: the prediction at the seeded initial state + seeded noise (2-D keypoints for the RGB config,
    key vertices with the synthetic occlusion mask for the AMASS config).  The prediction is the oracle port's forward (plain
    PyTorch on the host, float64, rounded once to float32), not the code being measured: the observations depend on the seeds,
    numpy and torch only, so every build benchmarked with the same arguments receives the same bytes (inputs_sha256 in the
    result line), and a build whose forward pass is wrong leaves residuals that show in its loss and gradients."""
    from tests import util_stage3 as U
    cfg = CONFIGS[config]
    of = cfg['optim_floor']
    B, T = prob['obs']['joints2d'].shape[:2]
    port = U.build_port(B, T, getattr(synth, cfg['weights']), of, prob, dtype=torch.float64)
    params = {k: torch.as_tensor(prob['params'][k], dtype=torch.float64) for k in U.PARAM_NAMES + (['floor_plane'] if of else [])}
    obs = {k: U.obs_to(prob['obs'][k], 'cpu') for k in U.obs_keys(of)}
    with torch.no_grad():
        _, _, inter = port.closure(params, obs)
    cam = inter['cam_pred']
    if config == 'amass':
        v = cam['verts3d'].numpy()
        rng = np.random.RandomState(5)
        occl = np.isinf(prob['obs']['verts3d'])
        prob['obs']['verts3d'] = np.where(occl, np.inf, v + rng.randn(*v.shape) * 0.01).astype(np.float32)
        return prob
    return U.project_joints2d(prob, torch.cat([cam['joints3d'], cam['joints3d_extra']], 2).numpy(), seed=5, noise=2.0)


def inputs_sha256(prob, obs_keys):
    """SHA-256 of every array the timed step reads (variables and observations, in a fixed order)."""
    h = hashlib.sha256()
    for part in (prob['params'], prob['obs']):
        keys = sorted(part) if part is prob['params'] else obs_keys
        for k in keys:
            a = np.ascontiguousarray(part[k])
            h.update(f'{k} {a.dtype.str} {a.shape}'.encode() + a.tobytes())
    return h.hexdigest()


def run_product(args):
    from humor_b200 import _ext
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl')
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    _ext.check(_ext.lib().humor_lbs_configure(args.lbs_skin, args.lbs_blend, args.lbs_slab), 'humor_lbs_configure')
    B, T = args.batch, args.seq_len
    OBS_KEYS = CONFIGS[args.config]['obs']
    prob = project_obs(build_problem(B, T, seed=4 + rank, config=args.config), args.config)
    mo = make_optimizer(B, T, prob, dev, args.config)
    # global frame intervals of this rank's block of sub-sequences (one video split across the ranks)
    prob['obs']['seq_interval'] = prob['obs']['seq_interval'] + rank * B * (T - 10)
    inputs_digest = inputs_sha256(prob, OBS_KEYS)
    if world > 1 and 'seq_interval' in OBS_KEYS and not args.no_halo:
        from humor_b200.parallel import Shard
        mo.shard = Shard.from_env(ov_max=16)
    names = mo.set_stage3_state(prob['params'])
    obs = {k: torch.as_tensor(prob['obs'][k]).to(dev) for k in OBS_KEYS}
    params = [getattr(mo, n) for n in names]
    if world > 1 and mo.shard is not None:
        mo.shard.prepare(obs['seq_interval'])
    mo.use_cuda_graph = not args.no_graph
    mo.set_precision(args.precision)

    def step():
        return mo.stage3_step(obs, params=params)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    # the sampler (nvidia-smi -lms 100) is started before the warm-up: its first row takes ~0.2 s, longer than a 10-step timed region
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    # ---- device-resident timing (value)
    barrier()
    row0 = len(sampler.rows)
    l0 = _ext.LaunchCounter.total
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]     # per-step stamps inside the ONE timed region
    e0.record()
    marks[0].record()
    for i in range(args.steps):
        loss = step()
        marks[i + 1].record()
    e1.record()
    barrier()
    # what the last timed step returned, copied on the device; written to disk once the clock sampling has ended
    last = (loss.detach().clone(), {n: getattr(mo, n).grad.detach().clone() for n in names}) if args.dump_outputs and rank == 0 else None
    ms = e0.elapsed_time(e1)
    per = torch.tensor([marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)], device=dev)
    per_all = per[None]
    if world > 1:
        import torch.distributed as dist
        buf = [torch.empty_like(per) for _ in range(world)]
        dist.all_gather(buf, per)
        per_all = torch.stack(buf, 0)
    per_step = {'median': float(per_all.median()), 'p95': float(torch.quantile(per_all.flatten(), 0.95)), 'max': float(per_all.max()),
                'by_rank_median': [float(x) for x in per_all.median(1).values], 'by_rank_max': [float(x) for x in per_all.max(1).values]}
    launches = _ext.LaunchCounter.total - l0
    # clocks under THIS load: the rows sampled inside the timed region and, when that region was shorter than three sampling periods,
    # rows of untimed steps of the same closure run right after it (every rank runs the same number: the step holds the halo exchange)
    timed_rows = len(sampler.rows) - row0
    extra = max(0, int(450.0 / max(ms / args.steps, 1e-3)) - args.steps) if (rank == 0 and timed_rows < 3) else 0
    if world > 1:
        import torch.distributed as dist
        ex = torch.tensor([extra], device=dev)
        dist.broadcast(ex, 0)
        extra = int(ex.item())
    for _ in range(extra):
        step()
    torch.cuda.synchronize()
    clocks = sampler.stop(row0, timed_rows) if rank == 0 else None
    if clocks is not None:
        clocks['untimed_steps_under_sampling'] = extra
    if last is not None:
        dump_outputs(args.dump_outputs, *last)
        last = None
    # ---- end-to-end timing: host params/observations in pinned memory in, loss + gradients out, every step
    host_in = {n: torch.as_tensor(prob['params'][n]).pin_memory() for n in names}
    host_obs = {k: torch.as_tensor(prob['obs'][k]).pin_memory() for k in OBS_KEYS}
    host_out = {n: torch.empty_like(host_in[n]).pin_memory() for n in names}
    host_loss = torch.empty(1).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in host_in.values()) + sum(t.numel() * t.element_size() for t in host_obs.values())
    d2h = sum(t.numel() * t.element_size() for t in host_out.values()) + 4

    def step_e2e():
        with torch.no_grad():
            for n in names:
                getattr(mo, n).copy_(host_in[n], non_blocking=True)
            for k in OBS_KEYS:
                obs[k].copy_(host_obs[k], non_blocking=True)
        loss = step()
        host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
        for n in names:
            host_out[n].copy_(getattr(mo, n).grad, non_blocking=True)
        torch.cuda.current_stream().synchronize()        # the caller (L-BFGS) reads the loss on the host

    step_e2e()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        step_e2e()
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    times = torch.tensor([ms, ms_e2e], device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(times[0]), float(times[1])
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        mo.shard = None                 # the rank-0-only diagnostics below must not enter collectives
    if rank != 0:
        return
    frames = B * T * world * args.steps
    value = frames / (ms * 1e-3)
    e2e = frames / (ms_e2e * 1e-3)
    hbm_peak, _, peak_kind = load_peaks()
    graphed = bool(mo.use_cuda_graph)
    mo_shard_off = 'seq_interval' not in OBS_KEYS or args.no_halo
    roof = lbs_roofline(mo, B, T, dev, hbm_peak, peak_kind)
    roof['forms'] = {'skin': args.lbs_skin or int(os.environ.get('HB_LBS_SKIN', 3)), 'blend': args.lbs_blend or int(os.environ.get('HB_LBS_BLEND', 5)),
                     'slab_frames': args.lbs_slab or int(os.environ.get('HB_LBS_SLAB', 512))}
    shares = kernel_shares(mo, obs, params, dev)
    cpu = torch_cuda = None
    try:        # what the last end-to-end step returned to the host: lets runs of the same seeded problem be compared across modes
        result_check = {'loss': float(host_loss[0]),
                        'grad_l2': float(torch.sqrt(sum((host_out[n].double() ** 2).sum() for n in names)))}
    except Exception:  # noqa: BLE001
        result_check = None
    out = {
        'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic (seeded SMPL+H-shaped asset, random-init HuMoR weights, projected 2-D keypoints)',
        'config': workload_config(args, world),
        'impl_details': {'cuda_graph': graphed, 'precision': args.precision, 'decoder_chain': 'launch-per-layer' if os.environ.get('HB_CHAIN') == '0' else 'persistent kernel (csrc/chain_persist.cuh)',
                         'collectives_per_step': 0 if (world == 1 or mo_shard_off) else 'halo exchange of the overlap pack fwd + its gradient bwd'},
        'e2e': {'value': e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'ms_per_step': ms_e2e / args.steps},
        'gpu_launches': int(launches), 'gpu_launches_per_step': launches / args.steps, 'per_step_ms': per_step,
        'clocks': clocks, 'roofline': roof, 'step_breakdown_ms': shares, 'cpu_baseline': cpu,
        'torch_cuda_port': torch_cuda, 'result_check': result_check, 'inputs_sha256': inputs_digest,
        'lbs_bytes_roofline_frac_of_step': value * (2.0 + 3.0 / T) * (LBS_BYTES_FWD + LBS_BYTES_BWD) / (hbm_peak * 1e9),
    }
    # The two context numbers run in bounded child processes AFTER the measurement, inside what is left of the run's time
    # limit: the result line must never be lost to them (the watchdog prints `out` as it stands if they overrun anyway).
    global _PARTIAL
    _PARTIAL = out
    if not args.no_cpu_baseline and world == 1:          # context numbers: rank 0 at N = 1 only
        left = _time_left() - 20.0
        if left - 45.0 >= 30.0:
            args.cpu_steps, args.cpu_warmup, args.cpu_budget = 3, 1, min(args.cpu_budget, 25.0)
            out['cpu_baseline'] = cpu_baseline(args, limit_s=min(150.0, left - 45.0))
        else:
            out['cpu_baseline'] = {'value': None, 'unit': 'frames/s', 'cores': cpu_threads(), 'kind': 'port',
                                   'sample': 'skipped: the run\'s time limit was nearly spent'}
        # the same algorithm as eager PyTorch on this GPU (context for the '>= 20x the reference PyTorch-CUDA step' target)
        left = _time_left() - 20.0
        out['torch_cuda_port'] = port_cuda_child(args, batch=B, limit_s=min(150.0, left)) if left >= 40.0 else \
            {'batch': B, 'error': 'skipped: the run\'s time limit was nearly spent'}
        if out['torch_cuda_port'].get('frames_per_s'):
            out['vs_torch_cuda_port'] = {'ratio': value / out['torch_cuda_port']['frames_per_s'], 'e2e_ratio': e2e / out['torch_cuda_port']['frames_per_s'],
                                         'same_batch': out['torch_cuda_port'].get('batch') == B, 'target': 20.0}
        # the kernel forms of the dense LBS forward (default 3/5, its 3xTF32 sibling 3/1, the round-1 two-kernel form 1/1), verified
        # against form 1/1 and timed stand-alone on this GPU (separate child processes: a fault must not take the measurement down)
        out['roofline_candidates'] = lbs_candidates(B, T, hbm_peak)
        # opt-in modes of the STEP (never the default), each a complete child run of this script on the same seeded problem;
        # `verified` = its loss and gradient norm agree with the run above
        out['step_candidates'] = step_candidates(args, result_check)
    _PARTIAL = None
    print(json.dumps(out))


def dump_outputs(path, loss, grads):
    """What the last timed step returned to its caller: loss.npy (1,) and grad_<variable>.npy for every stage-3 variable, all
    float32 (2 961 floats per sub-sequence in the RGB config: 3.0 MB at B = 256).  Every variable leads with the sub-sequence
    axis; when the files would exceed DUMP_LIMIT_BYTES, the same seeded sample of sub-sequences is kept of each and
    sample_rows.npy (float64) lists it, the sample sized so that all files, headers included, stay within the limit."""
    os.makedirs(path, exist_ok=True)
    out = {'grad_' + n: g.detach().float().cpu().numpy() for n, g in grads.items()}
    B = next(iter(out.values())).shape[0]
    row_bytes = sum(a.nbytes for a in out.values()) // B
    headers = NPY_HEADER_BYTES * (len(out) + 2)                  # the gradients, loss.npy and sample_rows.npy
    if B * row_bytes + 4 + headers > DUMP_LIMIT_BYTES:
        keep = (DUMP_LIMIT_BYTES - 4 - headers) // (row_bytes + 8)
        rows = np.sort(np.random.RandomState(0).choice(B, keep, replace=False))
        out = {k: a[rows] for k, a in out.items()}
        out['sample_rows'] = rows.astype(np.float64)
    out['loss'] = loss.detach().float().reshape(1).cpu().numpy()
    for k, a in out.items():
        np.save(os.path.join(path, k + '.npy'), a)


def lbs_roofline(mo, B, T, dev, hbm_peak, peak_kind):
    """Dominant-bytes kernel named by BASELINE: the dense LBS forward timed alone with CUDA
    events on the launching stream; algorithmic bytes = 83 896 B/frame (SURVEY.md §8d) x frames per launch."""
    from humor_b200.body_model import lbs
    N = B * T
    g = torch.Generator(device='cpu').manual_seed(0)
    ro = (torch.randn(N, 3, generator=g) * 0.5).to(dev)
    pb = (torch.randn(N, 63, generator=g) * 0.3).to(dev)
    be = (torch.randn(B, 16, generator=g) * 0.5).to(dev)
    tr = torch.randn(N, 3, generator=g).to(dev)
    m = mo.body_model.lbs_model
    with torch.no_grad():
        for _ in range(3):
            lbs(m, ro, pb, be, tr, T, None, True, False, 73)
        torch.cuda.synchronize()
        import ctypes as C
        from humor_b200 import _ext
        L = _ext.lib()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        # the dominant kernel (lbs_fuseg_kernel) between its own event pair, recorded by the library on the launching stream
        # (humor_lbs_fuseg_timing); the whole call (pose kernel, fp16 planes, shaped templates, joint gather, wrapper) around it
        L.humor_lbs_fuseg_timing(1, None, None)
        e0.record()
        for _ in range(reps):
            lbs(m, ro, pb, be, tr, T, None, True, False, 73)
        e1.record()
        torch.cuda.synchronize()
        kms, kn = C.c_float(0.0), C.c_int(0)
        L.humor_lbs_fuseg_timing(0, C.byref(kms), C.byref(kn))
    ms_call = e0.elapsed_time(e1) / reps
    us, ub = C.c_int(0), C.c_int(0)
    L.humor_lbs_forms_used(C.byref(us), C.byref(ub))
    fused_timed = us.value == 3 and kn.value == reps
    ms = kms.value / kn.value if fused_timed else ms_call       # forms without the fused kernel: the whole call
    achieved = N * LBS_BYTES_FWD / (ms * 1e-3) / 1e9
    if (us.value, ub.value) != (1, 1):          # the fused kernel (humor_lbs_configure skin form 3)
        name = ('lbs_fuseg_kernel, the dominant kernel of the dense LBS forward (persistent tcgen05 blend + group skinning' +
                (', fp16 hi/lo planes' if ub.value == 5 else ', 3xTF32 planes') + '; all vertices of every frame out)')
        traffic, tsrc = None, None
        if (us.value, ub.value) == (3, 5):
            # dram__bytes_read.sum + dram__bytes_write.sum of lbs_fuseg_kernel, ncu --set full of one 15 360-frame launch
            # (306.0 MB read + 1 262.5 MB written = 1.22 x the algorithmic 1 288.6 MB, which are 94 % output vertices)
            traffic, tsrc = 1568.6e6 * N / 15360.0, 'profiles/r03g_fuseg35_set_full_details.txt (gpurun_out/r03g_fuseg35_set_full.ncu-rep)'
        return {'kernel': name, 'bound': 'hbm', 'achieved': achieved, 'peak': hbm_peak, 'peak_source': peak_kind, 'unit': 'GB/s',
                'frac': achieved / hbm_peak, 'traffic': traffic, 'traffic_source': tsrc, 'ms_per_launch': ms,
                'timed': ('CUDA event pair around the kernel on its launching stream (humor_lbs_fuseg_timing), ' + str(kn.value) + ' launches'
                          if fused_timed else 'CUDA events around the whole humor_lbs_fwd call'),
                'ms_dense_forward_call': ms_call, 'frac_dense_forward_call': N * LBS_BYTES_FWD / (ms_call * 1e-3) / 1e9 / hbm_peak,
                'frames_per_launch': N, 'algorithmic_bytes_per_frame': LBS_BYTES_FWD, 'forms_used': [us.value, ub.value]}
    return {'kernel': 'dense LBS forward: lbs_pose_kernel + per 512-frame slab umma_gemm3_kernel<128,BIAS> (tcgen05 blend) + '
                      'lbs_skin_apply_kernel', 'bound': 'hbm', 'achieved': achieved,
            'peak': hbm_peak, 'peak_source': peak_kind, 'unit': 'GB/s', 'frac': achieved / hbm_peak,
            # dram__bytes_read.sum + dram__bytes_write.sum of the two slab kernels in profiles/r01g_lbs_slab_kernels_set_full.ncu-rep
            # (ncu --set full, cold L2: 41.4 MB blend GEMM + 46.7 MB skin pass per 512-frame slab) x slabs per launch.  Cold-cache
            # replay: the blend planes (37 MB) are re-read from DRAM for every slab and v_posed makes a DRAM round trip, while the
            # final write-back of the vertices is only partly inside the kernel's window.
            'traffic': (41.36e6 + 46.68e6) * ((N + 511) // 512), 'traffic_source': 'profiles/r01g_lbs_slab_kernels_set_full.ncu-rep',
            'ms_per_launch': ms, 'frames_per_launch': N, 'algorithmic_bytes_per_frame': LBS_BYTES_FWD}


def kernel_shares(mo, obs, params, dev):
    """Coarse split of one step (CUDA events around phases of an extra, untimed step)."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    for p in params:
        p.grad = None
    mo.use_cuda_graph = False
    mo.stage3_step(obs, params=params)          # eager warm-up (the timed region replayed a graph)
    for p in params:
        p.grad = None
    torch.cuda.synchronize()
    ev[0].record()
    loss, _, _, _, _ = mo.stage3_forward(obs)
    ev[1].record()
    loss.backward()
    ev[2].record()
    torch.cuda.synchronize()
    return {'forward': ev[0].elapsed_time(ev[1]), 'backward': ev[1].elapsed_time(ev[2])}


def cpu_baseline_inproc(args, threads):
    """The oracle port (plain-torch restatement of the reference closure) on the host cores.  One step = one full-T closure
    (fwd+bwd) of the SAME configuration at a bounded sample batch: the largest power of two <= --batch for which warm-up + steps
    fit the time budget, calibrated on one closure at B=8 (the port's cost is ~linear in B beyond B=8: 590 frames/s at B=8,
    755 frames/s at B=64 on 8 threads, so frames/s of the sample stands for the full batch)."""
    from tests import util_stage3 as U
    torch.set_num_threads(max(1, threads))
    T = args.seq_len
    cfg = CONFIGS[args.config]
    W = getattr(synth, cfg['weights'])
    of = cfg['optim_floor']

    def one(Bc, n_warm, n_steps):
        prob = build_problem(Bc, T, seed=4, config=args.config)
        port = U.build_port(Bc, T, W, of, prob)
        for _ in range(n_warm):
            U.closure_port(port, prob, of)
        ts = []
        for _ in range(n_steps):
            t0 = time.perf_counter()
            U.closure_port(port, prob, of)
            ts.append(time.perf_counter() - t0)
        return ts

    Bc = args.cpu_batch
    calib = None
    if Bc <= 0:
        calib = one(8, 1, 1)[0]
        Bc = 8
        while Bc * 2 <= args.batch and (args.cpu_warmup + args.cpu_steps) * calib * (Bc * 2 / 8.0) <= args.cpu_budget:
            Bc *= 2
    ts = one(Bc, args.cpu_warmup, args.cpu_steps)
    med = float(np.median(ts))
    return {'value': Bc * T / med, 'unit': 'frames/s', 'cores': threads, 'kind': 'port',
            'sample': f'{args.cpu_steps} full-T closures (fwd+bwd) after {args.cpu_warmup} warm-up at B={Bc} of the B={args.batch} workload, T={T}, '
                      f'config {args.config}, median; sample batch chosen for a {args.cpu_budget:.0f} s budget'
                      + (f' from a {calib:.2f} s calibration closure at B=8' if calib is not None else ''),
            's_per_step': med, 'sample_batch': Bc, 'steps': args.cpu_steps, 'warmup': args.cpu_warmup}


def port_on_cuda(args):
    """Context number for SURVEY.md 8(d): the reference ALGORITHM as eager PyTorch on the same B200 (the oracle port on
    device='cuda' - the reference itself cannot travel to the GPU box).  Launch/dispatch-bound, so its time per closure
    barely depends on B; the largest batch that fits is the fairest frames/s.  Not part of the default run."""
    from tests import util_stage3 as U
    import warnings
    warnings.filterwarnings('ignore')
    T = args.seq_len
    res = []
    for Bc in [int(b) for b in args.port_cuda.split(',')]:
        try:
            cfg = CONFIGS[args.config]
            of = cfg['optim_floor']
            prob = build_problem(Bc, T, seed=4, config=args.config)
            port = U.build_port(Bc, T, getattr(synth, cfg['weights']), of, prob, device='cuda')
            U.closure_port(port, prob, of, device='cuda')
            torch.cuda.synchronize()
            ts = []
            for _ in range(args.cpu_steps):
                t0 = time.perf_counter()
                U.closure_port(port, prob, of, device='cuda')
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            med = float(np.median(ts))
            res.append({'batch': Bc, 's_per_step': med, 'frames_per_s': Bc * T / med,
                        'peak_mem_gb': torch.cuda.max_memory_allocated() / 2**30})
        except torch.OutOfMemoryError:
            res.append({'batch': Bc, 'oom': True})
        except Exception as e:  # noqa: BLE001  (a context number must never take the bench down)
            res.append({'batch': Bc, 'error': f'{type(e).__name__}: {str(e)[:200]}'})
        finally:
            port = None
            torch.cuda.empty_cache()
    print(json.dumps({'impl': 'port-cuda', 'metric': METRIC, 'unit': 'frames/s', 'kind': 'oracle port of the reference closure, eager PyTorch (fp32) on cuda:0',
                      'config_name': args.config, 'steps': args.cpu_steps, 'results': res}))


def port_cuda_child(args, batch=64, limit_s=150):
    """SURVEY.md 8(d) / BASELINE.md section 3 - the denominator of the '>= 20x the reference PyTorch-CUDA step' target: the
    reference ALGORITHM as eager PyTorch on the same B200 (the oracle port on device='cuda'; the reference itself cannot travel
    to the GPU box), same configuration and batch as this run, in a child process with a hard limit."""
    cmd = [sys.executable, os.path.abspath(__file__), '--port-cuda', str(batch), '--cpu-steps', '3', '--seq-len', str(args.seq_len),
           '--config', args.config]
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT'):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=limit_s, env=env)
        d = json.loads(r.stdout.strip().splitlines()[-1])
        res = d['results'][0]
        res['kind'] = d['kind']
        return res
    except Exception as e:  # noqa: BLE001
        return {'batch': batch, 'error': f'{type(e).__name__}: {str(e)[:200]}'}


def lbs_candidates(B, T, hbm_peak):
    """tools/lbs_forms_time.py in bounded children: per opt-in form {used, ms, GBps, frac, max |dv| vs forms 1/1, deterministic,
    verified}.  One child per form, so a fault in one keeps the records of the others."""
    tool = os.path.join(ROOT, 'tools', 'lbs_forms_time.py')
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT', 'HB_LBS_SKIN', 'HB_LBS_BLEND'):
        env.pop(k, None)
    recs = []
    for forms in ('1,1', '3,1', '3,5'):
        left = _time_left() - 20.0
        if left < 40.0:
            recs.append({'forms': forms, 'error': 'skipped: the run\'s time limit was nearly spent'})
            continue
        cmd = [sys.executable, tool, '--forms', forms, '--seqs', str(B), '--frames-per-seq', str(T), '--reps', '5', '--peak-gbs', str(hbm_peak)]
        got, err = [], None
        try:
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=min(90.0, left), env=env)
            text, rc, tail = r.stdout, r.returncode, r.stderr[-300:]
        except subprocess.TimeoutExpired as e:
            text = e.stdout.decode() if isinstance(e.stdout, bytes) else (e.stdout or '')
            rc, tail = 'timeout', ''
        except Exception as e:  # noqa: BLE001
            text, rc, tail = '', type(e).__name__, str(e)[:300]
        for line in text.splitlines():
            if line.startswith('{'):
                try:
                    got.append(json.loads(line))
                except ValueError:
                    pass
        recs.extend(got)
        if rc != 0:
            done = {(g['skin'], g['blend']) for g in got}
            missing = [f for f in forms.split(';') if tuple(int(x) for x in f.split(',')) not in done]
            recs.append({'forms': ';'.join(missing), 'error': f'child ended with {rc}', 'stderr_tail': tail})
    return recs


def step_candidates(args, ref_check):
    """Child runs of bench.py with an opt-in mode switched on: {what, ms_per_step, value, e2e, loss / grad-norm difference to this
    run, verified}.  Last in line: whatever does not fit into the run's time limit is reported as skipped."""
    cands = [('precision tensor16 (forward decoder chain + prior on fp16 hi/lo operand planes)', ['--precision', 'tensor16'], {}),
             ('HB_UMMA_PREFETCH_B=1 (weight tiles requested before the dependent-launch wait)', [], {'HB_UMMA_PREFETCH_B': '1'})]
    recs = []
    for what, flags, extra in cands:
        left = _time_left() - 15.0
        if left < 60.0 or args.precision != 'tensor':
            recs.append({'what': what, 'error': 'skipped: the run\'s time limit was nearly spent'})
            continue
        cmd = [sys.executable, os.path.abspath(__file__), '--steps', str(args.steps), '--warmup', str(args.warmup), '--batch', str(args.batch),
               '--seq-len', str(args.seq_len), '--no-cpu-baseline'] + flags
        env = dict(os.environ, **extra)
        for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT'):
            env.pop(k, None)
        env['HB_BENCH_LIMIT_S'] = str(int(min(100.0, left)))
        try:
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=min(100.0, left), env=env)
            d = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])
            rec = {'what': what, 'ms_per_step': d['ms_per_step'], 'value': d['value'], 'e2e': d['e2e']['value'],
                   'result_check': d.get('result_check')}
            if ref_check and d.get('result_check'):
                dl = abs(d['result_check']['loss'] - ref_check['loss']) / max(1.0, abs(ref_check['loss']))
                dg = abs(d['result_check']['grad_l2'] - ref_check['grad_l2']) / max(1e-30, abs(ref_check['grad_l2']))
                rec.update(loss_rel_diff=dl, grad_l2_rel_diff=dg, verified=bool(dl < 1e-5 and dg < 1e-2))
            recs.append(rec)
        except Exception as e:  # noqa: BLE001
            recs.append({'what': what, 'error': f'{type(e).__name__}: {str(e)[:200]}'})
    return recs


def cpu_threads():
    # the closure is ~10^5 small torch ops: beyond ~16 intra-op threads the fork/join cost dominates
    return min(os.cpu_count() or 1, int(os.environ.get('HB_CPU_THREADS', 16)))


def cpu_baseline(args, threads=None, limit_s=150):
    """Runs cpu_baseline_inproc in a child process with a hard time limit so the bench always finishes."""
    threads = threads or cpu_threads()
    cmd = [sys.executable, os.path.abspath(__file__), '--_cpu-child', '--cpu-batch', str(args.cpu_batch), '--batch', str(args.batch),
           '--cpu-steps', str(args.cpu_steps), '--cpu-warmup', str(args.cpu_warmup), '--cpu-budget', str(args.cpu_budget),
           '--seq-len', str(args.seq_len), '--cpu-threads', str(threads), '--config', args.config]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='', OMP_NUM_THREADS=str(threads), MKL_NUM_THREADS=str(threads))
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT'):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=limit_s, env=env)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001
        return {'value': None, 'unit': 'frames/s', 'cores': threads, 'kind': 'port',
                'sample': f'did not finish within {limit_s} s ({type(e).__name__})'}


def run_reference(args):
    """Reference arm: the reference ALGORITHM (oracle port; the reference itself is Python + smplx, absent from the box) on the
    host cores, on THIS arm's configuration, metric and unit, with the driver's --steps / --warmup: every step is one full-T
    closure at a calibrated sample batch of the B = --batch workload (frames/s is intensive; see cpu_baseline_inproc)."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    world = int(os.environ.get('WORLD_SIZE', 1))
    args.cpu_steps, args.cpu_warmup = args.steps, args.warmup
    args.cpu_budget = max(args.cpu_budget, 170.0)
    cb = cpu_baseline(args, limit_s=330)
    out = {'impl': 'reference', 'metric': METRIC, 'value': cb['value'], 'unit': 'frames/s', 'n_gpus': world,
           'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': (cb.get('s_per_step') or 0.0) * 1e3,
           'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
           'data': 'synthetic (same seeded generator as the humor_b200 arm)',
           'config': workload_config(args, world), 'cpu_baseline': cb,
           'e2e': {'value': cb['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(out))


_T0 = time.monotonic()
_LIMIT_S = float(os.environ.get('HB_BENCH_LIMIT_S', 420))
_PARTIAL = None          # the finished measurement while the optional context children run


def _time_left():
    return _LIMIT_S - (time.monotonic() - _T0)


def _watchdog(limit_s):
    """A hung collective must not hold a GPU box: hard-exit after limit_s.  A finished measurement is printed first."""
    def run():
        time.sleep(limit_s)
        part = _PARTIAL
        if part is not None:
            sys.stderr.write(f'bench.py watchdog: context baselines still running after {limit_s} s, reporting without them\n')
            print(json.dumps(part), flush=True)
            os._exit(0)
        sys.stderr.write(f'bench.py watchdog: no result after {limit_s} s, aborting\n')
        os._exit(3)
    threading.Thread(target=run, daemon=True).start()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='humor_b200', choices=['humor_b200', 'reference'])
    ap.add_argument('--batch', type=int, default=256, help='sub-sequences per GPU')
    ap.add_argument('--seq-len', type=int, default=60)
    ap.add_argument('--config', default='rgb', choices=sorted(CONFIGS), help='rgb: fit_rgb_demo_use_split (BASELINE configs 2-3); amass: fit_amass_keypts (config 4)')
    ap.add_argument('--cpu-batch', type=int, default=0, help='sample batch of the host-CPU baseline (0: calibrated to --cpu-budget)')
    ap.add_argument('--cpu-steps', type=int, default=3)
    ap.add_argument('--cpu-warmup', type=int, default=1)
    ap.add_argument('--cpu-budget', type=float, default=25.0, help='seconds of host-CPU work the baseline may use')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--precision', default='tensor', choices=['tensor', 'exact', 'tensor16'],
                    help="'tensor': GEMMs on tcgen05 (3xTF32); 'exact': fp32 FFMA kernels (gradient-exact parity mode); "
                         "'tensor16': 'tensor' with the forward decoder chain on fp16 hi/lo operand planes (opt-in)")
    ap.add_argument('--lbs-skin', type=int, default=0, help='dense LBS form (humor_lbs_configure): 3 (default) fused blend + lane=frame group skinning in one persistent kernel, 1 blend GEMM + lane=vertex skin pass')
    ap.add_argument('--lbs-blend', type=int, default=0, help='dense LBS blend operand form: 5 (default, skin 3) fp16 hi/lo planes for every column (fp32-level), 1 three TF32 passes on fp32 hi/lo planes')
    ap.add_argument('--lbs-slab', type=int, default=0, help='frames per v_posed slab (128..512)')
    ap.add_argument('--no-halo', action='store_true', help='diagnostic: N independent replicas (no overlap coupling between ranks, no collective)')
    ap.add_argument('--no-graph', action='store_true', help='evaluate the closure eagerly instead of replaying a CUDA graph')
    ap.add_argument('--port-cuda', default='', help='comma list of batch sizes: time the oracle port as eager PyTorch on cuda:0')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='after the timed steps, write the loss and gradients the last of them returned as DIR/<name>.npy '
                         '(float32, at most 64 MB; with several GPUs, those of rank 0). The inputs do not depend on the '
                         'build, so dumps of two builds run with the same arguments can be compared output for output')
    ap.add_argument('--_cpu-child', dest='cpu_child', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--cpu-threads', type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'humor_b200' or args.port_cuda):
        ap.error('--dump-outputs writes what the timed humor_b200 step returned: not with --impl reference or --port-cuda')
    if args.cpu_child:
        import warnings
        warnings.filterwarnings('ignore')
        print(json.dumps(cpu_baseline_inproc(args, args.cpu_threads or cpu_threads())))
        return
    args.warmup = max(args.warmup, 3) if args.impl == 'humor_b200' else args.warmup
    _watchdog(_LIMIT_S)
    if args.port_cuda:
        port_on_cuda(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_product(args)


if __name__ == '__main__':
    main()
