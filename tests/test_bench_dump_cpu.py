"""bench.py --dump-outputs, host side: per config the documented file names and dtypes, a larger output reduced to the same fixed,
seeded sample on every run, and the files of one run within 64 MB.  Stand-ins replace the trained model (the step itself needs the GPU)."""
import os
import types

import numpy as np
import pytest
import torch

import bench


class _Trainer:
    loss_value = staticmethod(lambda terms: sum(float(t) * w for t, w in terms))

    def __init__(self):
        g = torch.Generator().manual_seed(0)
        self.d_arena = self.arena = types.SimpleNamespace(theta=torch.randn(bench.DUMP_MAX_ELEMS + 12345, generator=g))
        self.g_arena = types.SimpleNamespace(theta=torch.randn(1000, generator=g))


def _dump(cfg, out, d, tr):
    bench.dump_outputs(types.SimpleNamespace(cfg=cfg, trainer=tr), out, str(d))
    return {n[:-4]: np.load(os.path.join(d, n)) for n in os.listdir(d)}


def test_dump_outputs_names_dtypes_sample_and_size(tmp_path):
    tr = _Trainer()
    d_terms, g_terms = [(torch.tensor(2.0), 1.0), (torch.tensor(0.5), 0.3)], [(torch.tensor(3.0), 1.0)]
    cases = {1: (torch.randn(2, 256, 256, 5), {"logits"}),
             2: ((torch.tensor(1.5), torch.tensor(0.25)), {"wce_loss", "dice_loss", "params"}),
             3: (d_terms, {"dis_loss", "dis_params"}),
             4: ((d_terms, g_terms), {"dis_loss", "gen_loss", "dis_params", "gen_params"})}
    for cfg, (out, names) in cases.items():
        d = tmp_path / str(cfg)
        got = _dump(cfg, out, d, tr)
        assert set(got) == names
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        assert sum(os.path.getsize(d / (n + ".npy")) for n in got) <= 64 * 2 ** 20
    assert np.array_equal(_dump(1, cases[1][0], tmp_path / "1b", tr)["logits"], cases[1][0].numpy())
    got = _dump(4, cases[4][0], tmp_path / "4b", tr)
    assert float(got["dis_loss"]) == pytest.approx(2.15) and float(got["gen_loss"]) == 3.0
    assert np.array_equal(got["gen_params"], tr.g_arena.theta.numpy())
    # the arena above DUMP_MAX_ELEMS: the same sample of its values on every run
    assert got["dis_params"].shape == (bench.DUMP_MAX_ELEMS,)
    assert np.array_equal(got["dis_params"], _dump(3, d_terms, tmp_path / "3b", tr)["dis_params"])
    assert np.isin(got["dis_params"][:1000], tr.d_arena.theta.numpy()).all()
