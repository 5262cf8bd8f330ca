"""bench.py --dump-outputs: float32 files of the step's outputs, bounded in size by a seeded sample of the batch."""
import numpy as np
import torch

import bench


def _outputs(n):
    g = torch.Generator().manual_seed(0)
    return {"images": torch.randn(n, 3, 8, 8, generator=g).bfloat16(), "latents": torch.randn(n, 4, 2, 2, generator=g)}


def test_dump_outputs_writes_every_output_as_float32(tmp_path):
    out = _outputs(6)
    bench.dump_outputs(str(tmp_path / "d"), out)
    for k, v in out.items():
        a = np.load(tmp_path / "d" / f"{k}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, v.float().numpy())


def test_dump_outputs_samples_the_same_rows_of_every_output_within_the_limit(tmp_path, monkeypatch):
    n, keep = 10, 4
    out = _outputs(n)
    row_bytes = 4 * (3 * 8 * 8 + 4 * 2 * 2)
    monkeypatch.setattr(bench, "DUMP_BYTES", keep * row_bytes + row_bytes // 2)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    total = sum(f.stat().st_size - 128 for f in (tmp_path / "a").iterdir())   # 128-byte .npy headers
    assert total <= bench.DUMP_BYTES
    imgs = np.load(tmp_path / "a" / "images.npy")
    assert imgs.shape == (keep, 3, 8, 8)
    for name in ("images", "latents"):   # the same sample from run to run
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))
    full = out["images"].float().numpy()
    rows = [i for i in range(n) if any(np.array_equal(full[i], img) for img in imgs)]
    assert len(rows) == keep
    assert np.array_equal(np.load(tmp_path / "a" / "latents.npy"), out["latents"][rows].numpy())
