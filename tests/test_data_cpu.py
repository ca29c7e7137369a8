"""Host logic of the token data pipeline (open_musiclm_b200/data.py): the sqlite format of the reference
(preprocess.py:200,279; data.py:33-47), the crop arithmetic of PreprocessedDataset (data.py:334-434) and the
checkpoint file helpers (scripts/train_utils.py:19-46).  The device gather itself is covered in tests/test_data_gpu.py."""
import os
import random
import sqlite3

import numpy as np
import pytest
import torch

from open_musiclm_b200 import data as D


def synth_items(n, seconds=(14, 23), seed=0, sw=10, sps=50, aps=75):
    rng = np.random.default_rng(seed)
    items = []
    for i in range(n):
        L = int(rng.integers(seconds[0], seconds[1]))
        items.append(dict(clap=rng.integers(0, 1024, (L - sw + 1, 12)).astype(np.uint16),
                          semantic=rng.integers(0, 1024, (1, L * sps - 1)).astype(np.uint16),
                          coarse=rng.integers(0, 1024, (1, L * aps, 3)).astype(np.uint16),
                          fine=rng.integers(0, 1024, (1, L * aps, 5)).astype(np.uint16)))
    return items


def test_sqlite_round_trip_in_reference_format(tmp_path):
    items = synth_items(3)
    path = D.write_sqlite(str(tmp_path), items)
    conn = sqlite3.connect(path)
    cols = [r[1] for r in conn.execute("PRAGMA table_info(tokens)")]
    assert cols == ["idx", "path", "clap", "semantic", "coarse", "fine"]
    blob = conn.execute("SELECT coarse FROM tokens WHERE idx = 1").fetchone()[0]
    assert np.array_equal(D._unblob(blob), items[1]["coarse"])          # numpy .npy serialisation, as the reference's adapter
    conn.close()


class HostStore(D.TokenStore):
    """TokenStore with the flat arrays kept on the host (the crop logic under test never touches the device)."""

    def sample_batch(self, batch_size, rng=None, items=None):
        plans = [self.crop_plan(i, rng) for i in items]
        out = []
        for name in D.STAGE_COLUMNS[self.stage]:
            flat = self.flat[name].numpy().view(np.uint16).astype(np.int64)
            rows = [flat[int(self.offset[name][i]) + p[name][0]:int(self.offset[name][i]) + p[name][0] + p[name][1]] for i, p in zip(items, plans)]
            t = torch.from_numpy(np.stack(rows))
            out.append(t[:, 0] if name == "clap" else t)
        return out


def host_store(stage, items):
    return HostStore.from_items(stage, [{c: it[c] for c in D.STAGE_COLUMNS[stage]} for it in items], device="cpu")


@pytest.mark.parametrize("stage", ["semantic", "coarse", "fine"])
def test_crops_match_reference_dataset(stage):
    """Same items, same random draws -> the same token crops as the reference's PreprocessedDataset.__getitem__ over a
    database of these items (its crops with random.seed(100 + idx) are stored in tests/golden/reference_checks.pt)."""
    ds = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_checks.pt"), weights_only=False)["crops"][stage]
    items = synth_items(5, seed=3)
    store = host_store(stage, items)
    assert store.n_items == len(ds)
    for idx in range(len(ds)):
        theirs = ds[idx]
        mine = store.sample_batch(1, rng=random.Random(100 + idx), items=[idx])
        assert len(theirs) == len(mine)
        for a, b in zip(theirs, mine):
            assert a.numel() == b.numel(), (a.shape, b.shape)
            assert torch.equal(a.reshape(-1).long(), b.reshape(-1)), stage


def test_crop_lengths_are_the_training_shapes():
    items = synth_items(4, seed=1)
    for stage, exp in [("semantic", {"semantic": 499}), ("coarse", {"semantic": 199, "coarse": 300}), ("fine", {"coarse": 150, "fine": 150})]:
        store = host_store(stage, items)
        rng = random.Random(0)
        for i in range(4):
            plan = store.crop_plan(i, rng)
            assert plan["clap"][1] == 1
            for k, n in exp.items():
                assert plan[k][1] == n                 # 10 s of semantic tokens; 4 s windows for coarse; 2 s for fine
                assert 0 <= plan[k][0] and plan[k][0] + n <= np.asarray(items[i][k]).shape[1]


def test_latest_checkpoints(tmp_path):
    for step in (100, 200, 300):
        for kind in ("transformer", "optimizer", "scheduler"):
            open(tmp_path / f"coarse.{kind}.{step}.pt", "w").close()
    paths, step = D.latest_checkpoints(str(tmp_path))
    assert step == 300 and all("300" in p for p in paths)
    assert tuple(paths) == D.checkpoint_paths(str(tmp_path), "coarse", 300)
    paths, step = D.latest_checkpoints(str(tmp_path), max_step=250)
    assert step == 200
    os.remove(tmp_path / "coarse.optimizer.300.pt")
    with pytest.raises(AssertionError):
        D.latest_checkpoints(str(tmp_path))
