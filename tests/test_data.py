"""The cached-latent data path (SURVEY.md 8f ranks 1-2) against the REFERENCE's own classes.

``tests/golden/data_golden.json`` holds content digests produced by executing the reference's ImageTextLatentDataset /
custom_collate_fn / BucketBatchSampler / build_epoch_shuffle_batch_schedule / pack_sdxl_sample_schedule on the synthetic cache
of tests/data_fixture.py (generator: tests/golden/make_data_golden.py).  The product must reproduce every item, batch and
schedule bit for bit."""
import json
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

from data_fixture import DataCfg, build_cache, item_digest  # noqa: E402

from aozora_sdxl_training_b200 import data  # noqa: E402

GOLD = json.load(open(os.path.join(HERE, "golden", "data_golden.json")))
sys.path.insert(0, os.path.join(HERE, "golden"))
from make_data_golden import SPREAD_CASES, VARIANTS, run, run_buckets, run_spread  # noqa: E402


def product_schedule(ds, total_steps, batch_size, seed):
    return data.epoch_shuffle_batch_schedule(ds.bucket_keys, total_steps, batch_size, seed)


@pytest.mark.parametrize("name", list(VARIANTS))
def test_dataset_collate_and_schedules_match_reference_golden(name, tmp_path):
    got = run(data.CachedLatentDataset, data.collate, product_schedule, data.pack_sample_schedule, str(tmp_path), VARIANTS[name])
    want = GOLD[name]
    assert got["len"] == want["len"] and got["order"] == want["order"] and got["bucket_keys"] == want["bucket_keys"]
    assert got["schedule"] == want["schedule"]                # batch schedules for batch sizes 1, 2, 4: same indices, same order
    assert got["packed"] == want["packed"]
    assert got["items"] == want["items"]                      # every tensor byte, size tuple and chosen caption file
    assert got["batches"] == want["batches"]
    assert any(d == "None" for row in got["items"] for d in row)      # the NaN latent was dropped, as in the reference


def test_time_ids_and_feeder(tmp_path):
    cfg = type("Cfg", (DataCfg,), dict(INSTANCE_DATASETS=build_cache(str(tmp_path))))
    ds = data.CachedLatentDataset(cfg)
    sched = data.pack_sample_schedule(data.epoch_shuffle_batch_schedule(ds.bucket_keys, 9, 4, cfg.SEED), 4)
    direct = [data.collate([ds[p] for p in b]) for b in sched]
    fed = list(data.BatchFeeder(ds, sched, depth=2, pin=False))
    assert len(fed) == len(direct) == 9
    for a, b in zip(fed, direct):
        assert item_digest({k: v for k, v in a.items() if k != "time_ids"}, str(tmp_path)) == item_digest(b, str(tmp_path))
        rows = a["time_ids"]
        for r, s, c, t in zip(rows, b.get("scaled_sizes", b["original_sizes"]), b["crop_coords"], b["target_sizes"]):
            assert r == [s[1], s[0], c[0], c[1], t[1], t[0]]          # train.py:2726-2729
    # resume in the middle of the schedule, and per-rank rows of every global batch
    assert [item_digest(x, str(tmp_path)) for x in data.BatchFeeder(ds, sched, start_step=6, pin=False)] == \
           [item_digest(x, str(tmp_path)) for x in fed[6:]]
    for step, b in enumerate(sched):
        parts = [data.rank_slice(b, r, 2) for r in range(2)]
        assert parts[0] + parts[1] == b and len(parts[0]) >= len(parts[1])
    r1 = list(data.BatchFeeder(ds, sched, rank=1, world=2, pin=False))
    assert all((not x) or len(x["latents"]) <= 2 for x in r1)
    with pytest.raises(ValueError):
        data.pack_sample_index(1 << 32, 0)


def test_spread_schedules_and_bucket_ladder_match_reference_golden():
    """Timestep-spread batch schedules (train.py:703-887) and the bucket ladder (train.py:894-999), against digests made by
    running the reference's functions."""
    from aozora_sdxl_training_b200 import host
    got = [run_spread(host.build_timestep_ticket_pool,
                      lambda keys, steps, bs, seed, pool, ranges: data.image_batch_schedule(keys, steps, bs, seed, pool, ranges, True), c)
           for c in SPREAD_CASES]
    assert got == GOLD["spread"]
    assert run_buckets(data.optimal_bucket, data.multi_bucket_resolutions, data.bucket_ladder) == GOLD["buckets"]
    assert data.resolve_max_bucket_resolution("abc") == 1024 and data.resolve_max_bucket_resolution(2359296) == 1536
