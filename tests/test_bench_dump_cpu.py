"""bench.py --dump-outputs: arrays are written as float32 / float64, and an output too large to keep whole is cut to the
same seeded sample on every run, so that two builds' dumps line up element for element."""
import numpy as np
import torch

import bench


def test_dump_sample_is_a_fixed_subset_in_index_order():
    t = torch.arange(2 * bench.DUMP_SAMPLE + 7)
    a, b = bench.dump_sample(t), bench.dump_sample(t.clone())
    assert a.numel() == bench.DUMP_SAMPLE and torch.equal(a, b)
    assert bool((a[1:] > a[:-1]).all())                      # distinct elements, in index order
    small = torch.randn(5, 7)
    assert torch.equal(bench.dump_sample(small), small.reshape(-1))


def test_dump_outputs_writes_float32_or_float64(tmp_path):
    bench.dump_outputs(str(tmp_path), {"counts": torch.tensor([3, 2**40 + 1]), "mask": torch.tensor([0, 1], dtype=torch.uint8),
                                       "act": torch.tensor([1.5, -2.0], dtype=torch.bfloat16), "loss": torch.tensor(0.25)})
    got = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert {k: v.dtype for k, v in got.items()} == {"counts": np.float64, "mask": np.float32, "act": np.float32, "loss": np.float32}
    assert got["counts"].tolist() == [3, 2**40 + 1] and got["mask"].tolist() == [0, 1] and got["act"].tolist() == [1.5, -2.0]
