"""CPU: bench.py --dump-outputs, the maps of the last timed step written as .npy files."""
import importlib.util
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _maps(n, ins_num):
    """Per-ray maps whose every entry names its ray, so a row of any map shows which ray it came from."""
    idx = torch.arange(n, dtype=torch.float32)
    return {"rgb_fine": idx[:, None] + torch.tensor([0.0, 0.25, 0.5]), "depth_fine": idx, "acc_fine": idx + 0.5,
            "ins_fine": idx[:, None].repeat(1, ins_num)}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_writes_every_map_and_samples_the_same_rays(tmp_path):
    bench = _bench()
    small = _maps(1000, 13)
    bench.dump_outputs(small, 1000, 13, str(tmp_path / "small"))
    got = _load(tmp_path / "small")
    assert set(got) == set(small)
    for k, v in small.items():
        assert got[k].dtype == np.float32
        np.testing.assert_array_equal(got[k], v.numpy())

    n, ins_num = 307200, 59                                   # a 640x480 frame with 59 objects: 78.6 MB of maps
    big = _maps(n, ins_num)
    packed = torch.cat([big["rgb_fine"], big["depth_fine"][:, None], big["acc_fine"][:, None], big["ins_fine"]], -1)
    bench.dump_outputs(big, n, ins_num, str(tmp_path / "one_rank"))
    bench.dump_outputs(torch.cat([packed, torch.zeros(64, packed.shape[1])]).reshape(2, -1, packed.shape[1]), n, ins_num,
                       str(tmp_path / "two_ranks"))             # all-gathered slab, padded rows at the end
    one, two = _load(tmp_path / "one_rank"), _load(tmp_path / "two_ranks")
    assert sum(os.path.getsize(tmp_path / "one_rank" / (k + ".npy")) for k in one) <= 64e6
    rays = one["depth_fine"]
    assert n // 2 < len(rays) < n and np.all(np.diff(rays) > 0)
    np.testing.assert_array_equal(one["acc_fine"], rays + 0.5)
    np.testing.assert_array_equal(one["rgb_fine"][:, 0], rays)
    np.testing.assert_array_equal(one["ins_fine"][:, -1], rays)
    for k in one:
        np.testing.assert_array_equal(one[k], two[k])
    bench.dump_outputs(big, n, ins_num, str(tmp_path / "again"))
    np.testing.assert_array_equal(_load(tmp_path / "again")["depth_fine"], rays)
