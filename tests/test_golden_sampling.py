"""The sampled golden fixtures (tests/golden/sampled.py): positions and the round trip shrink -> Golden.pick."""
import numpy as np
import torch

from tests.golden import sampled


def test_positions_are_distinct_sorted_and_spread():
    for n_total, n in ((10, 3), (1000, 1000), (1000, 5000), (8 * 128 * 160, 4096), (2 * 90 * 160, 512)):
        p = sampled.positions(n_total, n)
        assert len(p) == min(n, n_total) and len(np.unique(p)) == len(p)
        assert (np.diff(p) > 0).all() and p[0] >= 0 and p[-1] < n_total
        if 100 <= n < n_total:   # no large gap: every tenth of the range holds about a tenth of the positions
            counts = np.bincount(p * 10 // n_total, minlength=10)
            assert counts.min() >= 0.8 * n / 10, counts


def test_shrink_and_pick_round_trip(tmp_path):
    g = torch.Generator().manual_seed(0)
    flow = torch.randn(1, 7, 2, 32, 40, generator=g)
    frames = torch.randint(0, 256, (7, 32, 40, 3), generator=g, dtype=torch.uint8).numpy()
    mask = (torch.rand(7, 32, 40, generator=g) > 0.8).numpy()
    store = sampled.shrink({"flow": flow, "frames": frames, "mask": mask}, {"flow": (2, 100), "frames": (-1, 200)})
    np.savez_compressed(tmp_path / "f.npz", **store)
    G = sampled.Golden(str(tmp_path / "f.npz"))
    assert G["flow"].shape == (100, 2) and G["frames"].shape == (200, 3)
    assert G.shape("flow") == (1, 7, 2, 32, 40) and G.shape("mask") == (7, 32, 40)
    assert np.array_equal(G.pick("flow", flow), G["flow"]) and np.array_equal(G.pick("frames", frames), G["frames"])
    assert np.array_equal(G.pick("mask", mask), mask)
    # each sample is the channel vector of one pixel, and a per-pixel array picks the same pixels
    rows = frames.reshape(-1, 3)
    hit = [int(np.flatnonzero((rows == v).all(1))[0]) for v in G["frames"][:5]]
    assert all((rows[i] == v).all() for i, v in zip(hit, G["frames"][:5]))
    idx = G.pick("frames", np.arange(7 * 32 * 40).reshape(7, 32, 40))
    assert np.array_equal(rows[idx], G["frames"])
    assert np.array_equal(G.pick("frames", mask), mask.reshape(-1)[idx])
    # a full output of another shape is refused
    try:
        G.pick("flow", flow[:, :6])
    except AssertionError:
        pass
    else:
        raise AssertionError("shape mismatch not detected")
