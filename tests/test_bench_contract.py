"""CPU test of the bench contract that does not need a GPU: `bench.py --impl reference` (the reference's CPU path,
timed through the oracle port) prints exactly ONE JSON line on stdout with the keys the driver reads, and ranks other
than 0 print nothing."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                           "--warmup", "0"], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    p = _run()
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "postproc_tiles_per_s" and d["unit"] == "tiles/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["config"]["workload"] == "slide" and d["config"]["masks"] == "paste"    # the reference's own mask path
    # nothing is extrapolated: ms_per_step is the measured time of one sample pass, value follows from it
    assert abs(d["value"] - d["tiles_per_step"] / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"] + 1e-9
    assert d["steps"] == d["steps_requested"] == 1 and d["other_mask_variant"]["masks"] == "proto"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    p = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def _bench_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_cpu_merge_scaling_leg():
    """The slide bench's CPU merge baseline (SURVEY 8d): sub-slides are cut by tile index, every size is an exact
    Ensemble.merge of its boxes, the exponent is fitted over the sizes that fit the budget."""
    import torch
    import torchvision

    bench = _bench_module()
    g = torch.Generator().manual_seed(0)
    n_cols, per = 5, 300
    boxes, scores, tile = [], [], []
    for t in range(n_cols * n_cols):
        r, cc = divmod(t, n_cols)
        c = torch.rand((per, 2), generator=g) * 1024 + torch.tensor([cc * 960., r * 960.])
        s = 12 + 24 * torch.rand((per, 2), generator=g)
        boxes.append(torch.cat([c - s / 2, c + s / 2], 1))
        scores.append(0.2 + 0.7 * torch.rand(per, generator=g))
        tile.append(torch.full((per,), t))
    boxes, scores, tile = torch.cat(boxes), torch.cat(scores), torch.cat(tile)
    out = bench.cpu_merge_scaling(boxes, scores, tile, n_cols, 0.25, 0.45, grids=(2, 3, 4))
    assert out["tiles"] == [4, 9, 16] and out["boxes"] == [4 * per, 9 * per, 16 * per] and "exponent" in out
    sel = ((tile // n_cols) < 2) & ((tile % n_cols) < 2)
    b, sc = boxes[sel], scores[sel]
    keep = sc > 0.25
    assert out["kept"][0] == len(torchvision.ops.nms(b[keep], sc[keep], 0.45))


def test_dump_outputs_writes_samples_and_mask_pixels(tmp_path, monkeypatch):
    """--dump-outputs: float32/float64 arrays only, a seeded sample (the same positions on every run) above DUMP_ROWS
    detections, and the packed masks of the sampled detections unpacked to exactly their pixels."""
    import numpy as np
    import torch

    from hd_yolo_b200.masks import PackedMasks

    bench = _bench_module()
    rng = np.random.default_rng(1)
    n = 40
    dense, geom, offsets, words = [], [], [0], []
    for _ in range(n):                       # windows up to 3 words wide, some empty
        w, h = int(rng.integers(0, 80)), int(rng.integers(0, 9))
        m = rng.random((h, w)) < 0.5
        dense.append(m)
        geom.append((int(rng.integers(0, 500)), int(rng.integers(0, 500)), w, h))
        wpr = (w + 31) // 32
        padded = np.zeros((h, wpr * 32), dtype=np.uint8)
        padded[:, :w] = m
        words.append(np.packbits(padded.reshape(-1), bitorder="little").view(np.uint32))
        offsets.append(offsets[-1] + wpr * h)
    bits = torch.from_numpy(np.concatenate(words).view(np.int32).copy())
    pm = PackedMasks(torch.tensor(geom, dtype=torch.int32), torch.tensor(offsets), bits, 600, 600,
                     torch.zeros((1,), dtype=torch.int32))
    K = 25
    boxes, scores = torch.rand((K, 4)), torch.rand((K,))
    labels = torch.randint(1, 5, (K,))
    mask_rows = torch.from_numpy(rng.permutation(n)[:K])

    def load(d):
        out = {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
        assert all(a.dtype in (np.float32, np.float64) for a in out.values())
        return out

    bench.dump_outputs(str(tmp_path / "all"), boxes, scores, labels, mask_rows, pm, {"counts": np.array([n, K], float)})
    a = load(tmp_path / "all")
    assert np.array_equal(a["sample"], np.arange(K)) and np.array_equal(a["boxes"], boxes.numpy())
    assert np.array_equal(a["labels"], labels.numpy()) and np.array_equal(a["counts"], [n, K])
    want = [dense[r] for r in mask_rows.tolist()]
    assert np.array_equal(a["mask_windows"], np.array([geom[r] for r in mask_rows.tolist()], dtype=np.float32))
    assert np.array_equal(a["mask_pixels"], np.concatenate([m.reshape(-1) for m in want]).astype(np.float32))

    monkeypatch.setattr(bench, "DUMP_ROWS", 10)
    monkeypatch.setattr(bench, "DUMP_MASKS", 4)
    bench.dump_outputs(str(tmp_path / "s1"), boxes, scores, labels, mask_rows, pm, {})
    bench.dump_outputs(str(tmp_path / "s2"), boxes, scores, labels, mask_rows, pm, {})
    s1, s2 = load(tmp_path / "s1"), load(tmp_path / "s2")
    pos = s1["sample"].astype(np.int64)
    assert len(pos) == 10 and np.all(np.diff(pos) > 0) and all(np.array_equal(s1[k], s2[k]) for k in s1)
    assert np.array_equal(s1["scores"], scores.numpy()[pos]) and len(s1["mask_windows"]) == 4
    four = [dense[r] for r in mask_rows[pos[:4]].tolist()]
    assert np.array_equal(s1["mask_pixels"], np.concatenate([m.reshape(-1) for m in four]).astype(np.float32))
