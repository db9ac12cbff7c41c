"""not gpu: bench.py --dump-outputs writes the faces of the last timed step as float32, and above the size cap a fixed
sample of whole shapes."""
import numpy as np
import torch

import bench


def test_dump_faces_full_and_capped(tmp_path, monkeypatch):
    faces = torch.randn(6, 4, 3, 3, generator=torch.Generator().manual_seed(0))
    faces[1, 2] = float("nan")                      # a face that was not generated
    bench.dump_faces(str(tmp_path / "full"), faces)
    full = np.load(tmp_path / "full" / "faces.npy")
    assert full.dtype == np.float32 and np.array_equal(full, faces.numpy(), equal_nan=True)

    limit = 3 * faces[0].numel() * 4 + 100          # room for three shapes
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", limit)
    bench.dump_faces(str(tmp_path / "a"), faces)
    bench.dump_faces(str(tmp_path / "b"), faces)
    a, b = np.load(tmp_path / "a" / "faces.npy"), np.load(tmp_path / "b" / "faces.npy")
    assert a.shape == (3, 4, 3, 3) and a.nbytes <= limit
    assert np.array_equal(a, b, equal_nan=True)     # the sample does not change from run to run
    rows = [next(i for i in range(6) if np.array_equal(r, faces[i].numpy(), equal_nan=True)) for r in a]
    assert rows == sorted(set(rows))                # distinct shapes, in their original order
