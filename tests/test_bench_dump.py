"""bench.py --dump-outputs on the host: names, dtypes, the seeded sample of large arrays, the size limit."""
import numpy as np
import pytest
import torch

import bench


def test_dump_outputs(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, 'DUMP_MAX_ELEMS', 64)
    g = torch.Generator().manual_seed(0)
    out = {'depth': torch.rand(1, 4, 5, 1, generator=g),
           'depth_up': torch.rand(1, 16, 20, 1, generator=g),
           'prob_volume_agg': torch.randn(1, 3, 4, 5, generator=g, dtype=torch.float64),
           'cost_volume_agg': torch.randn(1, 3, 4, 5, 8, generator=g).half(),
           'depth_views': [torch.rand(1, 4, 5, 1, generator=g) for _ in range(2)]}
    for run in ('a', 'b'):
        bench.dump_outputs(out, str(tmp_path / run))
    got = {n: np.load(str(tmp_path / 'a' / (n + '.npy'))) for n in out}
    assert np.array_equal(got['depth'], out['depth'].numpy())
    assert np.array_equal(got['depth_views'], torch.stack(out['depth_views']).numpy())
    assert got['prob_volume_agg'].dtype == np.float64
    assert np.array_equal(got['prob_volume_agg'], out['prob_volume_agg'].numpy())
    for n in ('depth_up', 'cost_volume_agg'):          # above DUMP_MAX_ELEMS: the seeded sample
        full = out[n].float().numpy().ravel()
        idx = np.sort(np.random.default_rng(0).choice(full.size, 64, replace=False))
        assert got[n].dtype == np.float32 and np.array_equal(got[n], full[idx])
        assert np.array_equal(got[n], np.load(str(tmp_path / 'b' / (n + '.npy'))))

    # a step without the reverse passes returns depth_views = [None, ...]: nothing is written for it
    bench.dump_outputs(dict(out, depth_views=[None, None]), str(tmp_path / 'd'))
    assert sorted(p.name for p in (tmp_path / 'd').iterdir()) == sorted(n + '.npy' for n in out if n != 'depth_views')

    monkeypatch.setattr(bench, 'DUMP_MAX_BYTES', 1000)
    with pytest.raises(RuntimeError):
        bench.dump_outputs(out, str(tmp_path / 'c'))
    assert not (tmp_path / 'c').exists()
