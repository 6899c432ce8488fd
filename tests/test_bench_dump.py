"""bench.py --dump-outputs: the files written for one step's output dict (CPU tensors stand in for the device ones)."""
import os

import numpy as np
import torch

import bench


def step_outputs(B, frames=1000, Tp=125):
    """The dict one headline step returns: framewise / clipwise / embedding (cla) of Cnn_9layers_Gru_FrameAtt."""
    g = torch.Generator().manual_seed(0)
    return {"framewise_output": torch.rand(B, frames, 25, generator=g),
            "clipwise_output": torch.rand(B, 25, generator=g),
            "embedding": torch.rand(B, 25, Tp, generator=g)}


def read(d, names):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in names}


def test_headline_outputs_are_dumped_as_one_seeded_sample_of_clips_within_64_mb(tmp_path):
    out = step_outputs(1024)
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    names = bench.dump_outputs(out, a)
    assert names == ["clipwise_output", "embedding", "framewise_output", "sampled_clips"]
    assert sum(os.path.getsize(os.path.join(a, n + ".npy")) for n in names) <= 64 * 10 ** 6
    got = read(a, names)
    idx = got["sampled_clips"]
    assert idx.dtype == np.float64 and 100 < len(idx) < 1024
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < 1024
    rows = idx.astype(np.int64)
    for k, v in out.items():
        assert got[k].dtype == np.float32
        assert np.array_equal(got[k], v.numpy()[rows]), k
    # same outputs -> the same files
    assert bench.dump_outputs(out, b) == names
    again = read(b, names)
    assert all(np.array_equal(got[n], again[n]) for n in names)


def test_small_outputs_are_dumped_whole_in_float32(tmp_path):
    out = step_outputs(6, frames=200, Tp=25)
    out["clipwise_output"] = out["clipwise_output"].half()
    out["embedding"] = None  # models without that entry
    names = bench.dump_outputs(out, str(tmp_path))
    assert names == ["clipwise_output", "framewise_output"]
    got = read(str(tmp_path), names)
    for k in names:
        assert got[k].dtype == np.float32
        assert np.array_equal(got[k], out[k].float().numpy()), k
