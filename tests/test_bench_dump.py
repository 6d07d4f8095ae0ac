"""bench.py --dump-outputs on the host: file names and dtypes, the fixed sample of a large output, the size bound."""
import os

import numpy as np
import pytest
import torch

import bench


def test_dump_outputs_dtypes_and_fixed_sample(tmp_path):
    g = torch.Generator().manual_seed(1)
    big = torch.rand(3 * bench.DUMP_SAMPLE + 5, generator=g)
    arrays = {'loss': torch.tensor(0.25), 'big': big, 'f64': torch.rand(2, 3, dtype=torch.float64, generator=g),
              'half': torch.rand(4, generator=g).half()}
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {k: np.load(str(tmp_path / 'a' / (k + '.npy'))) for k in arrays}
    assert sorted(os.listdir(str(tmp_path / 'a'))) == sorted(k + '.npy' for k in arrays)
    assert got['loss'].dtype == np.float32 and got['loss'].shape == () and float(got['loss']) == 0.25
    assert got['f64'].dtype == np.float64 and np.array_equal(got['f64'], arrays['f64'].numpy())
    assert got['half'].dtype == np.float32 and np.array_equal(got['half'], arrays['half'].float().numpy())
    # one element from each stride of 3, at the same positions on every run
    s = got['big']
    assert s.dtype == np.float32 and s.shape == (bench.DUMP_SAMPLE,)
    strata = big[:3 * bench.DUMP_SAMPLE].numpy().reshape(-1, 3)
    assert ((strata == s[:, None]).sum(axis=1) >= 1).all()
    assert np.array_equal(s, np.load(str(tmp_path / 'b' / 'big.npy')))


def test_dump_outputs_refuses_more_than_the_limit(tmp_path):
    arrays = {'o%d' % i: torch.zeros(bench.DUMP_SAMPLE) for i in range(bench.DUMP_LIMIT // (4 * bench.DUMP_SAMPLE) + 1)}
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path), arrays)
