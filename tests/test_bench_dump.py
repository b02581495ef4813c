"""bench.py --dump-outputs: field elements survive the float64 files exactly, a long output is sampled at the same
positions on every run, commitments are written as affine points, and several ranks share the size budget"""
import numpy as np
import torch

import bench


def test_dump_outputs_exact_and_repeatable(orc, tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_ROWS", 64)
    g = torch.Generator().manual_seed(3)
    long = torch.randint(-(1 << 63), (1 << 63) - 1, (1000, 4), dtype=torch.int64, generator=g)
    short = long[:10].clone()
    bases = orc.gen_bases(1, 40, 40, True)
    points = [orc.msm(bases, orc.gen_fr(2, 40, False)), orc.msm(bases, np.zeros((40, 4), dtype=np.uint64))]
    com = [torch.from_numpy(p.view(np.int64).copy()) for p in points]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"long": long, "short": short}, com)

    files = sorted(f.name for f in (tmp_path / "a").iterdir())
    assert files == ["commitments.npy", "long.npy", "short.npy"]
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b)

    def limbs(name):
        return np.load(tmp_path / "a" / name).astype(np.uint32).view(np.int64)

    assert np.array_equal(limbs("short.npy"), short.numpy())
    pos = {r.tobytes(): i for i, r in enumerate(long.numpy())}
    picked = [pos[r.tobytes()] for r in limbs("long.npy")]
    assert len(picked) == 64 and picked == sorted(set(picked))

    cm = np.load(tmp_path / "a" / "commitments.npy")
    assert cm.shape == (2, 25)
    assert np.array_equal(cm[0, :24].astype(np.uint32).view(np.uint8), orc.normalize(points[0])[:96]) and cm[0, 24] == 0
    assert cm[1, 24] == 1

    bench.dump_outputs(str(tmp_path / "r"), {"long": long}, com, rank=1, world=2)
    assert sorted(f.name for f in (tmp_path / "r").iterdir()) == ["commitments_rank1.npy", "long_rank1.npy"]
    assert np.load(tmp_path / "r" / "long_rank1.npy").shape == (32, 8)
