"""bench.py host logic that runs without a GPU: both arms (`--impl b200`, `--impl reference`) describe ONE workload — the
`config` object of their JSON lines is the same dict, so the driver's ratio compares like with like."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def _args(**kw):
    base = dict(gpus=1, steps=20, warmup=5, impl="b200", config=2, batch=0, labels=0, size=480, gather="p2p_copy",
                backbone="clip_vitl16_384")
    base.update(kw)
    return argparse.Namespace(**base)


def test_both_arms_print_the_same_config():
    for world, cfg_id in ((1, 2), (8, 2), (1, 5)):
        a, r = _args(gpus=world, config=cfg_id), _args(gpus=world, config=cfg_id, impl="reference")
        ca, cr = bench.line_config(bench.make_config(a), a, world), bench.line_config(bench.make_config(r), r, world)
        assert ca == cr
        json.dumps(ca)
        assert ca["global_batch"] == ca["batch_per_gpu"] * world
        assert "flush" in ca["l2"] and "workload" in ca
    c = bench.line_config(bench.make_config(_args()), _args(), 1)
    assert c["batch_per_gpu"] == 8 and "K=150" in c["workload"] and "480x480" in c["workload"]


def test_dump_outputs_sample(tmp_path):
    """--dump-outputs: a large output is written as a fixed sample (the same flat indices in every run), small ones whole,
    every array float32 / float64 and all of them within 64 MiB."""
    import numpy as np
    import torch
    big = torch.arange(3 * bench.DUMP_SAMPLE, dtype=torch.float32).reshape(3, 1, -1)
    a, b = bench.sample_outputs(big), bench.sample_outputs(big)
    assert set(a) == {"logits", "logits_index", "logits_shape"}
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert a["logits"].shape == (bench.DUMP_SAMPLE,) and np.array_equal(a["logits"], a["logits_index"].astype(np.float32))
    assert list(a["logits_shape"]) == [3, 1, bench.DUMP_SAMPLE]
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    small = bench.sample_outputs(big[:, :, :100])
    assert np.array_equal(small["logits"], big[:, :, :100].reshape(-1).numpy()) and "logits_index" not in small
    bench.write_outputs(str(tmp_path / "out"), a)
    assert np.array_equal(np.load(tmp_path / "out" / "logits.npy"), a["logits"])
