"""CPU-side checks (no GPU): hparams registry equals the reference's, the C-ABI library loads and
exports every symbol include/jkb200.h declares, product modules carry the reference's parameter
names/shapes (strict state-dict contract), host helpers, and the no-CPU-fallback rule."""
import ast
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

from golden_util import Fixture, GOLDEN

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _clean(d):
    return {k: (list(v) if isinstance(v, tuple) else v) for k, v in d.items()}


def test_hparams_match_reference_dump():
    from jukebox_b200.hparams import HPARAMS_REGISTRY, DEFAULTS, setup_hparams
    from jukebox_b200.make_models import MODELS
    g = json.load(open(os.path.join(GOLDEN, "hparams.json")))
    assert set(g["registry"]) == set(HPARAMS_REGISTRY)
    for k, v in g["registry"].items():
        assert _clean(HPARAMS_REGISTRY[k]) == v, k
    for k, v in g["defaults"].items():
        assert _clean(DEFAULTS[k]) == v, k
    for k, v in g["resolved"].items():
        assert _clean(setup_hparams(k, {})) == v, k
    assert {k: list(v) for k, v in MODELS.items()} == g["models"]
    with pytest.raises(ValueError):
        setup_hparams("vqvae", dict(not_a_key=1))


def test_hparams_resolve_exactly_as_reference():
    """the reference's setup_hparams(k, {}) as Python literals: values compare with their types (tuple != list)"""
    from jukebox_b200.hparams import HPARAMS_REGISTRY, setup_hparams
    ref = json.load(open(os.path.join(GOLDEN, "hparams.json")))["resolved_repr"]
    assert set(ref) == set(HPARAMS_REGISTRY)
    for k, r in ref.items():
        assert ast.literal_eval(r) == dict(setup_hparams(k, {})), k


def test_library_exports_every_declared_symbol():
    from jukebox_b200 import _lib
    header = open(os.path.join(ROOT, "include", "jkb200.h")).read()
    declared = set(re.findall(r"\b(jk_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(handle, name), f"{name} not exported"
    assert _lib.lib().jk_version() >= 100
    assert _lib.lib().jk_last_error() is not None


def test_no_cpu_fallback():
    from jukebox_b200.transformer.transformer import Transformer
    tr = Transformer(64, 48, 2, 2, mask=True, attn_order=2, blocks=4).eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        tr(torch.zeros(1, 1, 64), sample=True, fp16=True)
    from jukebox_b200.vqvae.bottleneck import BottleneckBlock
    with pytest.raises(RuntimeError, match="CUDA"):
        BottleneckBlock(16, 64, 0.99).encode(torch.zeros(1, 4, 64))
    # nothing under jukebox_b200/ may reference the oracle
    for dirpath, _, files in os.walk(os.path.join(ROOT, "jukebox_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


@pytest.mark.parametrize("name", ["transformer_order9", "transformer_order6", "transformer_order12"])
def test_transformer_state_dict_names(name):
    from jukebox_b200.transformer.transformer import Transformer
    fx = Fixture(name)
    c = fx.cfg
    tr = Transformer(c["n_in"], c["n_ctx"], c["n_head"], c["n_depth"], mask=True, attn_order=c["attn_order"],
                     blocks=c["blocks"], encoder_dims=c["encoder_dims"], prime_len=c["prime_len"])
    mine = [(k, tuple(v.shape)) for k, v in tr.state_dict().items()]
    assert mine == fx.names


@pytest.mark.parametrize("tag", ["single_enc_dec", "upsampler", "sep_enc_dec"])
def test_simple_prior_state_dict_names(tag):
    from jukebox_b200.hparams import setup_hparams
    from jukebox_b200.make_models import make_vqvae, make_prior
    fx = Fixture(f"prior_{tag}")
    c = fx.cfg
    vq = make_vqvae(setup_hparams(c["vq_name"], dict(restore_vqvae="", **c["vq_over"])), "cpu")
    prior = make_prior(setup_hparams(c["pr_name"], dict(restore_prior="", **c["pr_over"])), vq, "cpu")
    mine = [(k, tuple(v.shape)) for k, v in prior.state_dict().items()]
    assert sorted(mine) == sorted(fx.names)
    assert prior.n_ctx == c["n_ctx"]


@pytest.mark.parametrize("tag", ["small", "3level"])
def test_vqvae_state_dict_names(tag):
    from jukebox_b200.hparams import setup_hparams
    from jukebox_b200.make_models import make_vqvae
    fx = Fixture(f"vqvae_{tag}")
    c = fx.cfg
    vq = make_vqvae(setup_hparams(c["hps_name"], dict(restore_vqvae="", **c["overrides"])), "cpu")
    mine = [(k, tuple(v.shape)) for k, v in vq.state_dict().items()]
    assert sorted(mine) == sorted(fx.names)
    assert [tuple(z) for z in vq.z_shapes] == [tuple(fx[f"z{l}"].shape[1:]) for l in range(c["levels"])]


def test_sample_utils():
    from jukebox_b200.utils.sample_utils import get_starts, split_batch
    assert get_starts(20, 8, 6) == [0, 6, 12]
    assert get_starts(8192 * 3, 8192, 6144)[-1] == 8192 * 2
    assert [x.shape[0] for x in split_batch(torch.zeros(7, 2), 7, 3)] == [3, 3, 1]
    assert split_batch(None, 7, 3) == [None, None, None]


def test_attn_order_tables():
    from jukebox_b200.transformer.transformer import attn_func_of
    from oracle.transformer_np import ATTN_ORDERS
    for order, fn in ATTN_ORDERS.items():
        assert [attn_func_of(order, d) for d in range(160)] == [fn(d) for d in range(160)], order


def test_labeller_y_layout():
    from jukebox_b200.data.labels import Labeller, get_relevant_lyric_tokens
    lab = Labeller(1, 12, 1000, v3=True)
    y = lab.get_y_from_ids(7, [3], list(range(12)), 5000, 100)
    assert y.tolist() == [5000, 100, 1000, 7, 3] + list(range(12))
    toks, idx = get_relevant_lyric_tokens(list(range(100)), 12, 5000, 2500, 1000)
    assert len(toks) == 12 and toks == [list(range(100))[i] for i in idx]
    toks, idx = get_relevant_lyric_tokens([5, 6], 4, 10, 0, 1)
    assert toks == [0, 0, 5, 6] and idx == [-1, -1, 0, 1]
