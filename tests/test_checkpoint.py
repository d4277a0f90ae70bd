"""Checkpoint I/O (SURVEY.md 8f rank 3): LDM key mapping against the reference's own ``get_unet_key_mapping`` (frozen digest),
single-file load / export round trips, training-state file."""
import hashlib
import json
import os
import random

import numpy as np
import pytest
import torch

from aozora_sdxl_training_b200 import checkpoint as ck
from aozora_sdxl_training_b200.unet import UNet2DConditionModel, init_weights_, sdxl_config, tiny_config

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "host_golden.json")))


def full_sdxl_keys():
    with torch.device("meta"):
        return list(UNet2DConditionModel(sdxl_config()).state_dict().keys())


def mapping_digest(mapping):
    return hashlib.sha256("\n".join(f"{k} -> {v}" for k, v in mapping.items()).encode()).hexdigest()


def test_key_mapping_digest_matches_reference_golden():
    keys = full_sdxl_keys()
    assert len(keys) == 1680
    m = ck.unet_key_mapping(keys)
    assert len(set(m.values())) == 1680 and all(v.startswith("model.diffusion_model.") for v in m.values())
    assert mapping_digest(m) == GOLD["unet_key_mapping_sha256"]
    for hf, ldm in [("down_blocks.2.attentions.0.transformer_blocks.3.attn1.to_q.weight", "model.diffusion_model.input_blocks.7.1.transformer_blocks.3.attn1.to_q.weight"),
                    ("up_blocks.0.upsamplers.0.conv.weight", "model.diffusion_model.output_blocks.2.2.conv.weight"),
                    ("mid_block.resnets.1.conv2.bias", "model.diffusion_model.middle_block.2.out_layers.3.bias"),
                    ("down_blocks.1.downsamplers.0.conv.bias", "model.diffusion_model.input_blocks.6.0.op.bias"),
                    ("up_blocks.2.resnets.1.conv_shortcut.weight", "model.diffusion_model.output_blocks.7.0.skip_connection.weight")]:
        assert m[hf] == ldm                                              # SURVEY.md 8a appendix examples


def test_single_file_roundtrip_and_export(tmp_path):
    from safetensors.torch import load_file, save_file
    src = init_weights_(UNet2DConditionModel(tiny_config()), seed=3, std=0.05).to(torch.bfloat16)
    mp = ck.unet_key_mapping(list(src.state_dict().keys()))
    base = {mp[k]: v.detach().clone().contiguous() for k, v in src.state_dict().items()}
    base["first_stage_model.decoder.w"] = torch.randn(4, 4)                                  # non-UNet tensors ride along
    base["conditioner.embedders.0.ids"] = torch.arange(7)
    base_path = tmp_path / "base.safetensors"
    save_file(base, str(base_path))
    assert ck.peek_unet_channels(base_path) == (4, 4)
    # load through the inverse mapping into a fresh model (the reference's from_single_file call, train.py:1458-1464)
    got = ck.load_unet_single_file(base_path, torch_dtype=torch.bfloat16, config=tiny_config())
    assert list(got.state_dict().keys()) == list(src.state_dict().keys())
    for (k, a), (_, b) in zip(got.state_dict().items(), src.state_dict().items()):
        assert torch.equal(a, b), k
    # a missing tensor is an error, not a silent random init
    broken = dict(base)
    broken.pop(mp["conv_in.weight"])
    save_file(broken, str(tmp_path / "broken.safetensors"))
    with pytest.raises(KeyError):
        ck.load_unet_single_file(tmp_path / "broken.safetensors", config=tiny_config())
    # export: "train" (perturb), stack q/k/v storage (views of one buffer must not alias in the file), merge into the base
    with torch.no_grad():
        for p in got.parameters():
            p.add_(0.125)
    got.fuse_projection_storage()
    out_path = tmp_path / "out" / "model_step_3.safetensors"
    added = ck.save_model(out_path, got, base_path, torch.float16)
    assert added == []
    out = load_file(str(out_path))
    assert set(out) == set(base)
    assert out["first_stage_model.decoder.w"].dtype == torch.float16 and out["conditioner.embedders.0.ids"].dtype == torch.int64
    for k, v in got.state_dict().items():
        assert out[mp[k]].dtype == torch.float16 and torch.equal(out[mp[k]], v.to(torch.float16)), k
    again = ck.load_unet_single_file(out_path, torch_dtype=torch.float16, config=tiny_config())
    assert torch.equal(again.conv_in.weight, got.conv_in.weight.to(torch.float16))


def test_training_state_file(tmp_path):
    class FakeRaven:
        def __init__(self):
            self.loaded = None

        def save_cpu_state(self):
            return {"_momentum_dtype": torch.bfloat16, 0: {"step": 5, "exp_avg_cpu": torch.ones(3), "exp_avg_sq_cpu": torch.zeros(3)}}

        def load_cpu_state(self, st):
            self.loaded = st

    class Sampler:
        def __init__(self):
            self.pool_index = 37

        def state_dict(self):
            return {"pool_index": self.pool_index}

        def load_state_dict(self, st):
            self.pool_index = st["pool_index"]

    random.seed(11); np.random.seed(12); torch.manual_seed(13)
    path = tmp_path / "run_training_state_step_5.pt"
    ck.save_training_state(path, global_step=5, micro_step=10, optimizer=FakeRaven(), sampler_seed=42, sampler_epoch=3, timestep_sampler=Sampler())
    want = (random.random(), float(np.random.rand()), float(torch.rand(1)))
    random.seed(0); np.random.seed(0); torch.manual_seed(0)                    # disturb every stream, then resume
    opt, smp = FakeRaven(), Sampler()
    smp.pool_index = 0
    st = ck.load_training_state(path, optimizer=opt, timestep_sampler=smp, grad_accum=2)
    assert (st["global_step"], st["micro_step"], st["optimizer_step"], st["sampler_seed"], st["sampler_epoch"]) == (5, 10, 5, 42, 2)
    assert opt.loaded[0]["step"] == 5 and smp.pool_index == 37
    assert (random.random(), float(np.random.rand()), float(torch.rand(1))) == want
    # reference key set (train.py:2522-2530)
    assert set(torch.load(path, weights_only=False)) == {"global_step", "micro_step", "optimizer_state", "sampler_seed", "sampler_epoch",
                                                         "timestep_sampler_state", "random_state", "numpy_state", "torch_cpu_state", "torch_cuda_state"}
