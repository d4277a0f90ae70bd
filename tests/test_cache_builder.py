"""The latent / text cache builder (SURVEY.md 8f rank 4) against what the REFERENCE's own ``precompute_and_cache_latents`` wrote
for the same image folder with the same (deterministic, tiny) tokenizers, text encoders and VAE: every cache file must come out
with the same name and the same payload, tensor bytes included (digests frozen by tests/golden/make_cache_golden.py).  The
self-consistency tests: the cache is read back by ``data.CachedLatentDataset``, a second build is a no-op, a new image only adds
its own files."""
import json
import os
import sys
import types
import zlib

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

from aozora_sdxl_training_b200 import cache_builder as cb  # noqa: E402
from aozora_sdxl_training_b200 import data  # noqa: E402

PIL = pytest.importorskip("PIL.Image")


# ---- deterministic stand-ins for the models (batch-invariant: a row's output depends on that row only) -------------------
class TinyTokenizer:
    model_max_length = 77
    bos_token_id, eos_token_id, pad_token_id = 1, 2, 0

    def __init__(self, salt):
        self.salt = salt

    def _ids(self, text):
        return [3 + zlib.crc32((self.salt + w).encode()) % 500 for w in text.replace(",", " , ").split()]

    def __call__(self, text, add_special_tokens=True, truncation=False, padding=None, max_length=None, return_tensors=None):
        many = not isinstance(text, str)
        rows = [self._ids(t) for t in (text if many else [text])]
        if add_special_tokens:
            rows = [[self.bos_token_id] + r[:(max_length or 77) - 2 if truncation else None] + [self.eos_token_id] for r in rows]
        if padding == "max_length":
            rows = [(r + [self.pad_token_id] * max_length)[:max_length] for r in rows]
        if return_tensors == "pt":
            return types.SimpleNamespace(input_ids=torch.tensor(rows, dtype=torch.long))
        return types.SimpleNamespace(input_ids=rows if many else rows[0])


class _TextOut(tuple):
    hidden_states = None


class TinyTextEncoder(torch.nn.Module):
    def __init__(self, dim, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.table = torch.nn.Parameter(torch.randn(512, dim, generator=g), requires_grad=False)
        self.pos = torch.nn.Parameter(torch.randn(77, dim, generator=g) * 0.1, requires_grad=False)

    def forward(self, tokens, output_hidden_states=False):
        h0 = self.table[tokens] + self.pos[None, :tokens.shape[1]]
        h1 = torch.tanh(h0) + 0.5 * torch.cumsum(h0, dim=1) / (1 + torch.arange(tokens.shape[1])[None, :, None])
        h2 = h1 * 1.5 - 0.25
        out = _TextOut((h2.mean(dim=1), h2))
        out.hidden_states = (h0, h1, h2)
        return out


class TinyVAE(torch.nn.Module):
    def __init__(self, shift=None):
        super().__init__()
        self.config = types.SimpleNamespace(shift_factor=shift, scaling_factor=0.13025, latent_channels=4)
        self.mix = torch.nn.Parameter(torch.tensor([[0.6, -0.2, 0.1], [0.3, 0.3, 0.3], [-0.5, 0.4, 0.2], [0.1, 0.1, -0.7]]), requires_grad=False)

    def enable_tiling(self):
        pass

    def enable_slicing(self):
        pass

    def encode(self, x):
        pooled = torch.nn.functional.avg_pool2d(x, 8)
        lat = (pooled[:, None] * self.mix[None, :, :, None, None]).sum(dim=2)
        return types.SimpleNamespace(latent_dist=types.SimpleNamespace(mean=lat))


def models(shift=None):
    return (TinyTokenizer("a"), TinyTokenizer("b"), TinyTextEncoder(16, 1), TinyTextEncoder(24, 2), TinyVAE(shift))


# ---- a small image folder --------------------------------------------------------------------------------------------------
LONG = " ".join(f"word{i}" for i in range(170))          # three 75-token chunks


def make_folder(root, json_mode=False, extra=False):
    rng = np.random.default_rng(7)
    os.makedirs(os.path.join(root, "Nested Dir"), exist_ok=True)
    specs = [("cat_on_mat.png", (1300, 1100), "RGB", "a cat, on a mat"), ("Nested Dir/Tall.jpg", (900, 1500), "RGB", LONG),
             ("wide_one.webp", (1700, 800), "RGB", None), ("alpha.png", (1100, 1100), "RGBA", "with alpha"),
             ("small.bmp", (700, 650), "RGB", "small image, kept below the ladder"), ("pal.png", (1200, 1000), "P", "palette image")]
    if extra:
        specs.append(("zz_new.png", (1250, 1250), "RGB", "added later"))
    for name, (w, h), mode, caption in specs:
        path = os.path.join(root, name)
        if os.path.exists(path):
            continue
        arr = rng.integers(0, 256, size=(h // 8, w // 8, 4 if mode == "RGBA" else 3), dtype=np.uint8)
        img = PIL.fromarray(arr, "RGBA" if mode == "RGBA" else "RGB").resize((w, h), PIL.Resampling.BILINEAR)
        if mode == "P":
            img = img.convert("P")
        img.save(path)
        side = os.path.splitext(path)[0]
        if json_mode:
            doc = {"tags": f"tags of {name}", "nl": f"a sentence about {name}", "tags_nl": f"tags then text {name}", "nl_tags": "  "}
            if caption is None:
                doc = {"tags_nl": "only the primary"}
            json.dump(doc, open(side + ".json", "w"))
        elif caption is not None:
            open(side + ".txt", "w").write(caption + "\n")


def cfg_for(root, **kw):
    base = dict(INSTANCE_DATASETS=[{"path": root, "repeats": 1}], is_rectified_flow=False, SEED=3, CAPTION_SOURCE_TYPE="txt",
                CAPTION_CHUNKING_ENABLED=True, MULTI_BUCKET_ENABLED=True, MULTI_BUCKET_EXTRA_BUCKETS=1, SHOULD_UPSCALE=False,
                MAX_BUCKET_RESOLUTION=1024, CACHING_BATCH_SIZE=2, UNCONDITIONAL_DROPOUT=True, UNCONDITIONAL_DROPOUT_CHANCE=0.1,
                TEXT_CACHE_PRECISION="bfloat16", VAE_CACHE_PRECISION="float32", VAE_NORMALIZATION_MODE="scalar", REBUILD_CACHE=False,
                VAE_PATH="", SINGLE_FILE_CHECKPOINT_PATH=None, TEXT_CONDITIONING_SCALE_ENABLED=False)
    base.update(kw)
    return types.SimpleNamespace(**base)


CASES = {
    "txt_chunked_multibucket": dict(),
    "txt_plain_shift": dict(CAPTION_CHUNKING_ENABLED=False, MULTI_BUCKET_ENABLED=False, UNCONDITIONAL_DROPOUT=False,
                            TEXT_CACHE_PRECISION="fp32", VAE_CACHE_PRECISION="bf16", is_rectified_flow=True, CACHING_BATCH_SIZE=3),
    "json_variants": dict(CAPTION_SOURCE_TYPE="json", CAPTION_CHUNKING_ENABLED=False, MULTI_BUCKET_EXTRA_BUCKETS=2, SHOULD_UPSCALE=True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_cache_equals_the_frozen_reference_output(case, tmp_path):
    """Digests of what the reference's caching pass wrote (tests/golden/make_cache_golden.py)."""
    sys.path.insert(0, os.path.join(HERE, "golden"))
    from make_cache_golden import digest_cache
    gold = json.load(open(os.path.join(HERE, "golden", "cache_golden.json")))[case]
    root = str(tmp_path / "ds")
    opts = CASES[case]
    make_folder(root, json_mode=opts.get("CAPTION_SOURCE_TYPE") == "json")
    cfg = cfg_for(root, **opts)
    assert cb.cache_needs_build(cfg)
    cb.build_cache(cfg, *models(0.1 if case == "txt_plain_shift" else None), "cpu")
    cdir = os.path.join(root, cb.cache_folder_name(cfg))
    got = digest_cache(cdir, root, data.stable_item_key)
    assert sorted(got) == sorted(gold)
    assert got == gold
    assert not cb.cache_needs_build(cfg)

    # staleness the reference's check_if_caching_needed also reports: a missing latent file, another text-cache precision
    victim = next(n for n in sorted(got) if n.endswith("_lat.pt"))
    os.rename(os.path.join(cdir, victim), os.path.join(cdir, victim + ".bak"))
    assert cb.cache_needs_build(cfg)
    os.rename(os.path.join(cdir, victim + ".bak"), os.path.join(cdir, victim))
    assert not cb.cache_needs_build(cfg)
    assert cb.cache_needs_build(cfg_for(root, **{**opts, "TEXT_CACHE_PRECISION": "float16"}))


def test_token_chunks_and_text_batching():
    t1, t2, te1, te2, _ = models()
    rows = cb.chunked_tokens(t1, LONG, 3)
    assert rows.shape == (3, 77) and (rows[:, 0] == 1).all() and rows[0, 76] == 2 and rows[2, -1] == 0
    assert cb.chunk_count(LONG, t1) == 3 and cb.chunk_count("two words", t1) == 1
    caps = ["a cat", LONG, "", "x, y, z"]
    e, p = cb.embed_captions(caps, t1, t2, te1, te2, "cpu", chunked=True, total_chunks=3)
    assert e.shape == (4, 231, 40) and p.shape == (4, 24)
    for i, c in enumerate(caps):                              # one call for the batch == one call per caption
        e1, p1 = cb.embed_captions([c], t1, t2, te1, te2, "cpu", chunked=True, total_chunks=3)
        assert torch.equal(e1[0], e[i]) and torch.equal(p1[0], p[i])


def test_build_reuse_and_incremental_update(tmp_path):
    root = str(tmp_path / "ds")
    make_folder(root)
    cfg = cfg_for(root)
    cdir = os.path.join(root, cb.cache_folder_name(cfg))
    seen = []
    cb.build_cache(cfg, *models(), "cpu", progress=lambda kind, done, total: seen.append((kind, done, total)))
    assert seen and seen[-1][1] == seen[-1][2]
    assert not cb.cache_needs_build(cfg)
    ds = data.CachedLatentDataset(cfg)
    assert len(ds) == 6 * 2 - 1 or len(ds) > 6                # every image, plus the extra bucket variants that fit
    item = ds[data.pack_sample_index(0, 0)]
    assert item is not None and item["latents"].dim() == 3 and item["embeds"].shape[-1] == 40
    stamps = {n: os.stat(os.path.join(cdir, n)).st_mtime_ns for n in os.listdir(cdir)}
    cb.build_cache(cfg, *models(), "cpu")                     # current: nothing is rewritten
    assert stamps == {n: os.stat(os.path.join(cdir, n)).st_mtime_ns for n in os.listdir(cdir)}

    make_folder(root, extra=True)                             # one more image: only its files (and the index) are new
    assert cb.cache_needs_build(cfg)
    cb.build_cache(cfg, *models(), "cpu")
    after = {n: os.stat(os.path.join(cdir, n)).st_mtime_ns for n in os.listdir(cdir)}
    changed = sorted(n for n in after if stamps.get(n) != after[n])
    assert all(n.startswith("zz_new") or n in ("dataset_index.pt", "null_embeds.pt") for n in changed), changed
    assert any(n.startswith("zz_new") and n.endswith("_lat.pt") for n in changed)

    os.remove(os.path.join(root, "small.bmp"))                # a deleted image takes its cache files with it
    assert cb.cache_needs_build(cfg)
    cb.build_cache(cfg, *models(), "cpu")
    assert not [n for n in os.listdir(cdir) if n.startswith("small")] and not cb.cache_needs_build(cfg)
    with pytest.raises(RuntimeError):
        cb.build_cache(cfg_for(root, VAE_NORMALIZATION_MODE="flux_bn32"), *models(), "cpu")
    from aozora_sdxl_training_b200 import train_loop
    assert train_loop.ensure_cache(cfg, models(), "cpu") is False              # current: the loop's caching hook does nothing
    os.remove(os.path.join(cdir, "null_embeds.pt"))
    assert train_loop.ensure_cache(cfg, models(), "cpu") is True and os.path.exists(os.path.join(cdir, "null_embeds.pt"))
