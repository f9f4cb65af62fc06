"""bench.py --dump-outputs on the host: every file is written in float32 / float64, the whole dump stays within
bench.DUMP_LIMIT_BYTES, and a sampled dump keeps the same seeded sub-sequences of every variable.  CPU only."""
import os

import numpy as np
import pytest
import torch

import bench


def grads(B, T, seed=0):
    g = torch.Generator().manual_seed(seed)
    return {'trans': torch.randn(B, 1, 3, generator=g), 'betas': torch.randn(B, 16, generator=g),
            'latent_motion': torch.randn(B, T - 1, 48, generator=g)}


def dump_bytes(path):
    return sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))


def test_dump_small_is_complete(tmp_path):
    g = grads(8, 10)
    bench.dump_outputs(str(tmp_path), torch.tensor(2.5), g)
    assert sorted(os.listdir(tmp_path)) == ['grad_betas.npy', 'grad_latent_motion.npy', 'grad_trans.npy', 'loss.npy']
    assert np.load(tmp_path / 'loss.npy').tolist() == [2.5]
    for n, v in g.items():
        a = np.load(tmp_path / f'grad_{n}.npy')
        assert a.dtype == np.float32 and np.array_equal(a, v.numpy())


@pytest.mark.parametrize('limit', [200_000, 1_000_000])
def test_dump_large_is_a_seeded_sample_within_the_limit(tmp_path, monkeypatch, limit):
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', limit)
    B, T = 2000, 60
    g = grads(B, T)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), torch.tensor(1.0), g)
        assert dump_bytes(tmp_path / d) <= limit
    rows = np.load(tmp_path / 'a' / 'sample_rows.npy')
    assert rows.dtype == np.float64 and np.array_equal(rows, np.load(tmp_path / 'b' / 'sample_rows.npy'))
    assert len(rows) > 0 and (np.diff(rows) > 0).all()
    idx = rows.astype(np.int64)
    for n, v in g.items():
        assert np.array_equal(np.load(tmp_path / 'a' / f'grad_{n}.npy'), v.numpy()[idx])
    row = 4 * (3 + 16 + (T - 1) * 48) + 8                    # float32 gradients of one sub-sequence + its sample_rows entry
    assert dump_bytes(tmp_path / 'a') > limit - row           # the sample is as large as the limit allows
