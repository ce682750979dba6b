"""bench.py host logic: --dump-outputs writes float32 .npy files, --steps must name at least one timed step."""
import sys

import numpy as np
import pytest
import torch

import bench


def test_dump_outputs_writes_exact_float32(tmp_path):
    g = torch.Generator().manual_seed(0)
    images = torch.randint(0, 256, (2, 8, 8, 3), dtype=torch.uint8, generator=g)
    latents = torch.randn(2, 4, 1, 1, generator=g).to(torch.bfloat16)
    out = tmp_path / "dump"
    bench.dump_outputs(str(out), {"images": images, "latents": latents})
    assert sorted(p.name for p in out.iterdir()) == ["images.npy", "latents.npy"]
    got_i, got_l = np.load(out / "images.npy"), np.load(out / "latents.npy")
    assert got_i.dtype == np.float32 and got_l.dtype == np.float32
    np.testing.assert_array_equal(got_i, images.numpy().astype(np.float32))
    np.testing.assert_array_equal(got_l, latents.float().numpy())


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_rejected_arguments(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
