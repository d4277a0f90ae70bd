"""CPU tests: the oracle's host restatement AND the product's host logic against the frozen outputs of the
reference's own code (tests/golden/host_golden.json, made by tests/golden/make_golden.py)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from aozora_sdxl_training_b200 import host
from oracle import host_ref

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "host_golden.json")))


def sha_i64(values):
    return hashlib.sha256(np.asarray(values, dtype="<i8").tobytes()).hexdigest()


IMPLS = {
    "oracle": lambda c: host_ref.ticket_pool(c["allocation"], c["total"], 1000, c["seed"], c["stratified"]),
    "product": lambda c: host.build_timestep_ticket_pool(c["allocation"], c["total"], 1000, c["seed"], c["stratified"]),
}


@pytest.mark.parametrize("impl", list(IMPLS))
@pytest.mark.parametrize("name", list(GOLD["ticket_pools"]))
def test_ticket_pools_bit_exact(impl, name):
    g = GOLD["ticket_pools"][name]
    pool, ranges = IMPLS[impl](g["case"])
    assert len(pool) == g["n"]
    assert [int(x) for x in pool[:32]] == g["first"]
    assert sha_i64(pool) == g["sha256"]                      # every ticket, bit-exact
    assert [[int(a), int(b)] for a, b in ranges] == g["ranges"]


def test_scale_counts_and_logit_normal():
    for g in GOLD["scale_counts"].values():
        assert host_ref.largest_remainder_scale(g["counts"], g["total"]) == g["result"]
        assert host._scale_timestep_counts(g["counts"], g["total"]) == g["result"]
    gl = GOLD["gui_logit_normal_counts"]
    assert host_ref.logit_normal_counts(-0.5, 1.0, 1000) == gl["mu-0.5_sigma1_total1000"]
    assert host.logit_normal_allocation(-0.5, 1.0, 1000)["counts"] == gl["mu-0.5_sigma1_total1000"]
    assert host.logit_normal_allocation(0.0, 1.0, 1000)["counts"] == gl["mu0_sigma1_total1000"]


class _Cfg:
    MAX_TRAIN_STEPS = 5
    BATCH_SIZE = 3
    SEED = 42
    is_rectified_flow = False
    TIMESTEP_ALLOCATION = {"bin_size": 100, "counts": [45, 143, 176, 173, 154, 126, 94, 59, 26, 4]}
    TIMESTEP_STRATIFIED_SAMPLING = False


def test_sampler_pops_and_wrap():
    s = host.TimestepSampler(_Cfg, "cpu")
    assert [s.sample(3)[0].tolist() for _ in range(7)] == GOLD["sampler_pops"]
    r = host_ref.RefTimestepSampler(5, 3, 42, _Cfg.TIMESTEP_ALLOCATION, False)
    assert [r.sample(3)[0].tolist() for _ in range(7)] == GOLD["sampler_pops"]
    # resume semantics (train.py:2185-2197)
    s.set_current_step(2)
    assert s.state_dict() == {"pool_index": 6}
    s.load_state_dict({"pool_index": 16})
    assert s.pool_index == 1


def test_sampler_rank_slices_equal_single_process_pop():
    """Data-parallel ticket assignment == the single-process pop order of the global batch (SURVEY.md 8e)."""
    class C(_Cfg):
        BATCH_SIZE = 8
        MAX_TRAIN_STEPS = 6
    single = host.TimestepSampler(C, "cpu")
    ranks = [host.TimestepSampler(C, "cpu") for _ in range(4)]
    for _ in range(6):
        ref = single.sample(8)[0].tolist()
        got = sum((ranks[r].sample_rank(2, r, 4)[0].tolist() for r in range(4)), [])
        assert got == ref


def test_lr_curve():
    g = GOLD["lr_curve"]

    class Opt:
        param_groups = [{"lr": 0.0, "lr_scale": 1.0}]
    sch = host.CustomCurveLRScheduler(Opt, [list(p) for p in g["curve"]], g["total"])
    for st, want in g["lr"].items():
        sch.step(int(st))
        assert Opt.param_groups[0]["lr"] == want             # float64, exact
        assert host_ref.lr_at(g["curve"], int(st), g["total"]) == want
    with pytest.raises(ValueError):
        host.CustomCurveLRScheduler(Opt, [], 10)


def test_loss_tables():
    class LC:
        pass
    for g in GOLD["loss_tables"].values():
        LC.TIMESTEP_LOSS_WEIGHT_CURVE = g["points"]
        want = torch.tensor(g["values"])
        assert torch.equal(host.timestep_loss_curve_from_config(LC, 1000), want)
        assert torch.equal(host_ref.loss_weight_table(g["points"], 1000), want)
    LC.TIMESTEP_LOSS_WEIGHT_CURVE = None
    assert torch.equal(host.timestep_loss_curve_from_config(LC, 1000), torch.ones(1000))
    LC.TIMESTEP_LOSS_WEIGHT_CURVE = [[0.5, 1.0]]            # fewer than 2 valid points -> ones
    assert torch.equal(host.timestep_loss_curve_from_config(LC, 1000), torch.ones(1000))


def test_generators():
    g = host.seeded_torch_generator("cpu", 42, 1, 0x5D1)
    assert torch.rand(4, generator=g).tolist() == GOLD["rf_jitter_seed42_step1"]
    assert host_ref.rf_jitter(4, 42, 1).tolist() == GOLD["rf_jitter_seed42_step1"]
    gen = torch.Generator(device="cpu")
    n = host.generate_noise(torch.zeros(1, 4, 2, 2), gen, "cpu", step=3, seed=42)
    assert n.flatten().tolist() == GOLD["noise_seed42_step3"]
    assert host_ref.step_noise((1, 4, 2, 2), 42, 3).flatten().tolist() == GOLD["noise_seed42_step3"]


def test_weighted_mse_oracle():
    g = GOLD["weighted_mse"]
    gg = torch.Generator().manual_seed(g["seed"])
    pred = torch.randn(3, 4, 8, 8, generator=gg).to(torch.bfloat16)
    targ = torch.randn(3, 4, 8, 8, generator=gg)
    ts = torch.tensor([0, 495, 999])
    table = torch.tensor(GOLD["loss_tables"]["tri"]["values"])
    assert float(host_ref.weighted_mse(pred, targ, ts, table)) == g["value"]
    assert float(host_ref.weighted_mse(pred, targ, ts, None)) == g["value_unweighted"]


def test_exclusion_counts():
    """SURVEY.md a10: keyword semantics and the frozen-parameter census on the exact SDXL layout."""
    from aozora_sdxl_training_b200.unet import UNet2DConditionModel, sdxl_config
    with torch.device("meta"):
        m = UNet2DConditionModel(sdxl_config())
    assert host.apply_exclusion(m, ["down_blocks.0", "attn2"]) == 551_102_400
    assert sum(1 for p in m.parameters() if not p.requires_grad) == 372
    assert host.apply_exclusion(m, ["conv1", "conv2"]) == 296_782_720
    assert sum(1 for p in m.parameters() if not p.requires_grad) == 68
    assert host.apply_exclusion(m, []) == 0
    for name in ("down_blocks.0.resnets.0.conv1.weight", "mid_block.attentions.0.proj_in.bias"):
        assert host_ref.is_excluded(name, ["conv1", "conv2"]) == ("conv1" in name)


def test_unet_layout_matches_oracle_and_reference_keymap():
    from aozora_sdxl_training_b200.unet import UNet2DConditionModel, sdxl_config
    from oracle.unet_ref import RefUNet2DConditionModel, sdxl_config as ref_cfg
    with torch.device("meta"):
        prod = UNet2DConditionModel(sdxl_config())
        ref = RefUNet2DConditionModel(ref_cfg())
    pn = [(k, tuple(v.shape)) for k, v in prod.named_parameters()]
    rn = [(k, tuple(v.shape)) for k, v in ref.named_parameters()]
    assert pn == rn
    assert len(pn) == 1680 and sum(int(np.prod(s)) for _, s in pn) == 2_567_463_684
    names = [k for k, _ in pn]
    km = GOLD["key_map"]
    assert km["n"] == 1680
    assert hashlib.sha256("\n".join(names).encode()).hexdigest() == km["sha256_names"]


def test_raven_oracle_against_reference_trajectories():
    """oracle.host_ref.raven_update_ vs trajectories produced by the reference's own RavenAdamW / TitanAdamW."""
    blob = torch.load(os.path.join(HERE, "golden", "raven_golden.pt"))
    hp = blob["hparams"]
    for tag, tr in blob["traj"].items():
        torch.manual_seed(tr["p0_seed"])
        p = torch.randn(257).to(tr["p"].dtype)
        m = torch.zeros(257, dtype=tr["m"].dtype)
        v = torch.zeros(257, dtype=tr["v"].dtype)
        for s, g in enumerate(tr["grads"], start=1):
            if tag.startswith("titan"):
                g = g.float()           # Titan steps from fp32 copies of the gradients (titan.py:121-128)
            host_ref.raven_update_(p, g, m, v, lr=tr["lr"], betas=hp["betas"], eps=hp["eps"],
                                   weight_decay=hp["weight_decay"], debias_strength=hp["debias_strength"], step=s)
        assert torch.equal(p, tr["p"]), tag
        assert torch.equal(m, tr["m"]) and torch.equal(v, tr["v"]), tag


def test_stacked_projection_storage_keeps_the_state_dict_contract():
    """fuse_projection_storage() only changes WHERE q/k/v (and cross k/v) weights live: names, order, shapes and values of
    named_parameters() / state_dict() -- the reference's checkpoint contract (train.py:2478-2479, raven.py:157-168) -- stay."""
    import torch
    from aozora_sdxl_training_b200.unet import UNet2DConditionModel, _stacked, init_weights_, tiny_config
    m = init_weights_(UNet2DConditionModel(tiny_config())).to(torch.bfloat16)
    names = [n for n, _ in m.named_parameters()]
    before = {k: v.clone() for k, v in m.state_dict().items()}
    m.fuse_projection_storage()
    assert names == [n for n, _ in m.named_parameters()]
    for k, v in m.state_dict().items():
        assert torch.equal(v, before[k]) and v.is_contiguous(), k
    blk = m.mid_block.attentions[0].transformer_blocks[1]
    qkv = (blk.attn1.to_q.weight, blk.attn1.to_k.weight, blk.attn1.to_v.weight)
    w = _stacked(qkv)
    assert w is not None and w.shape == (3 * 256, 256) and torch.equal(w[256:512], blk.attn1.to_k.weight)
    assert _stacked((blk.attn2.to_k.weight, blk.attn2.to_v.weight)).shape == (512, 128)
    assert _stacked((blk.attn1.to_q.weight, blk.attn2.to_q.weight)) is None          # different storages
    blk.attn1.to_k.weight.requires_grad_(False)
    assert _stacked(qkv) is None                                                     # mixed requires_grad: separate GEMMs
    m2 = m.float()                                                                   # fresh storages: layout must be rebuilt
    assert not m2._fused_storage_ok
