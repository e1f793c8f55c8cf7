"""Generate tests/golden/*.npz by running the UNMODIFIED reference on CPU.

Run in the build container only (needs /root/reference):

    python -m oracle.make_golden            # rewrites every fixture
    python -m oracle.make_golden hparams sample_level     # only the named golden_* fixtures

Each fixture stores: a JSON config, the (name, shape) list of the reference module's
state_dict, the seed the synthetic weights were drawn with (oracle/synth.py), the inputs
and the reference's outputs (fp32 path and, for the prior, the fp16 path on CPU).
Weights themselves are not stored - they are a pure function of (name, shape, seed).
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)

from oracle.ref_import import load_reference  # noqa: E402
from oracle.synth import synth_state_dict     # noqa: E402

load_reference()
import torch as t                              # noqa: E402


def load_synth(module, seed):
    sd = module.state_dict()
    named = [(k, tuple(v.shape)) for k, v in sd.items()]
    new = synth_state_dict(named, seed)
    # tied parameters (x_out.weight is x_emb.weight unless merged_decoder,
    # prior/autoregressive.py:95-98) appear twice in the state_dict: keep one value.
    first, aliases = {}, []
    for k, v in sd.items():
        ptr = v.data_ptr()
        if ptr in first:
            aliases.append([k, first[ptr]])
            new[k] = new[first[ptr]]
        else:
            first[ptr] = k
    module.load_state_dict({k: t.from_numpy(v).to(sd[k].dtype) for k, v in new.items()})
    return [(n, s, dict(aliases).get(n)) for n, s in named]


def save(name, cfg, named, **arrays):
    path = os.path.join(GOLDEN, name + ".npz")
    np.savez_compressed(path, cfg=json.dumps(cfg), names=json.dumps([[n, list(s), a] for n, s, a in named]),
                        **{k: (v.numpy() if isinstance(v, t.Tensor) else np.asarray(v))
                           for k, v in arrays.items()})
    print(f"wrote {path}  ({os.path.getsize(path) / 1e3:.1f} kB)")


# ----------------------------------------------------------------------------------------
def golden_transformer(tag, n_in, n_ctx, n_head, n_depth, attn_order, blocks, bs,
                       encoder_dims=0, prime_len=None, seed=1):
    from jukebox.transformer.transformer import Transformer
    tr = Transformer(n_in, n_ctx, n_head, n_depth, mask=True, attn_order=attn_order, blocks=blocks,
                     encoder_dims=encoder_dims, prime_len=prime_len)
    tr.eval()
    named = load_synth(tr, seed)
    g = t.Generator().manual_seed(seed)
    x = t.randn(bs, n_ctx, n_in, generator=g)
    enc = t.randn(bs, encoder_dims, n_in, generator=g) if encoder_dims else None
    outs = {}
    with t.no_grad():
        for fp16 in (False, True):
            tr.del_cache()
            ys = [tr(x[:, i:i + 1].contiguous(), encoder_kv=enc, sample=True, fp16=fp16) for i in range(n_ctx)]
            outs["y16" if fp16 else "y32"] = t.cat(ys, 1)
        tr.del_cache()
        if attn_order not in (12,):   # full forward-mode pass (the encoder path of enc-dec priors)
            outs["yfull32"] = tr(x, encoder_kv=enc, sample=False, fp16=False)
    cfg = dict(n_in=n_in, n_ctx=n_ctx, n_head=n_head, n_depth=n_depth, attn_order=attn_order,
               blocks=blocks, encoder_dims=encoder_dims, prime_len=prime_len, seed=seed,
               attn_funcs=[l.attn.attn_func for l in tr._attn_mods])
    arrays = dict(x=x, **outs)
    if enc is not None:
        arrays["encoder_kv"] = enc
    save(f"transformer_{tag}", cfg, named, **arrays)


def golden_ca2d(tag, input_dims, bins, width, depth, heads, attn_order, blocks, x_cond, y_cond,
                encoder_dims=0, prime_len=None, merged_decoder=False, bs=2, chunk_size=5, seed=2):
    from jukebox.prior.autoregressive import ConditionalAutoregressive2D
    m = ConditionalAutoregressive2D((input_dims,), bins, width=width, depth=depth, heads=heads,
                                    attn_order=attn_order, blocks=blocks, x_cond=x_cond, y_cond=y_cond,
                                    encoder_dims=encoder_dims, prime_len=prime_len,
                                    merged_decoder=merged_decoder)
    m.eval()
    named = load_synth(m, seed)
    g = t.Generator().manual_seed(seed)
    xc = t.randn(bs, input_dims, width, generator=g) if x_cond else None
    yc = t.randn(bs, 1, width, generator=g) if y_cond else None
    enc = t.randn(bs, encoder_dims, width, generator=g) if encoder_dims else None
    t.manual_seed(seed)
    with t.no_grad():
        tokens, preds32 = m.sample(bs, xc, yc, enc, fp16=False, temp=1.0, get_preds=True)
        # teacher-forced fp16 logits through the reference's chunked prefill path
        _, preds16 = m.primed_sample(bs, tokens[:, :-1].clone(), xc, yc, enc, fp16=True,
                                     get_preds=True, chunk_size=chunk_size)
        _, preds32p = m.primed_sample(bs, tokens[:, :-1].clone(), xc, yc, enc, fp16=False,
                                      get_preds=True, chunk_size=chunk_size)
    cfg = dict(input_dims=input_dims, bins=bins, width=width, depth=depth, heads=heads,
               attn_order=attn_order, blocks=blocks, x_cond=x_cond, y_cond=y_cond,
               encoder_dims=encoder_dims, prime_len=prime_len, merged_decoder=merged_decoder,
               seed=seed, chunk_size=chunk_size)
    arrays = dict(tokens=tokens, preds32=preds32, preds16=preds16, preds32_primed=preds32p)
    if xc is not None:
        arrays["x_cond"] = xc
    if yc is not None:
        arrays["y_cond"] = yc
    if enc is not None:
        arrays["encoder_kv"] = enc
    save(f"ca2d_{tag}", cfg, named, **arrays)


# ----------------------------------------------------------------------------------------
def _tiny_vqvae_hps(**over):
    from jukebox.hparams import setup_hparams
    return setup_hparams("small_vqvae", dict(sample_length=over.pop("sample_length", 2048), **over))


def golden_vqvae(tag, hps_name, overrides, bs, seed=3):
    from jukebox.hparams import setup_hparams
    from jukebox.make_models import make_vqvae
    hps = setup_hparams(hps_name, dict(restore_vqvae="", **overrides))
    vq = make_vqvae(hps, "cpu")
    named = load_synth(vq, seed)
    g = t.Generator().manual_seed(seed)
    x = 2 * t.rand(bs, hps.sample_length, 1, generator=g) - 1
    with t.no_grad():
        zs = vq.encode(x, bs_chunks=bs)
        x_ds = [vq.decode(zs[l:], start_level=l, bs_chunks=bs) for l in range(len(zs))]
        # pre-quantisation latents, to measure argmin margins in the tests
        x_in = vq.preprocess(x)
        lat = [vq.encoders[l](x_in)[-1] for l in range(vq.levels)]
    cfg = dict(hps_name=hps_name, overrides=overrides, seed=seed, levels=hps.levels,
               downs_t=list(hps.downs_t), strides_t=list(hps.strides_t), width=hps.width, depth=hps.depth,
               growth=hps.dilation_growth_rate, cycle=hps.dilation_cycle,
               multipliers=list(hps.hvqvae_multipliers) if hps.hvqvae_multipliers else None,
               reverse=hps.vqvae_reverse_decoder_dilation, l_bins=hps.l_bins, emb_width=hps.emb_width,
               sample_length=hps.sample_length)
    arrays = dict(x=x)
    for l in range(len(zs)):
        arrays[f"z{l}"] = zs[l]
        arrays[f"xd{l}"] = x_ds[l]
        arrays[f"lat{l}"] = lat[l]
    save(f"vqvae_{tag}", cfg, named, **arrays)


# ----------------------------------------------------------------------------------------
TINY_PRIORS = {
    # tag: (vqvae hps name, vqvae overrides, prior hps names, prior overrides)
    "single_enc_dec": ("small_vqvae", dict(sample_length=84 * 256),
                       "small_single_enc_dec_prior",
                       dict(n_ctx=84, prior_width=64, prior_depth=16, heads=2, blocks=8, n_tokens=12,
                            level=1, levels=2)),
    "upsampler": ("small_vqvae", dict(sample_length=64 * 32),
                  "small_upsampler",
                  dict(n_ctx=64, prior_width=64, prior_depth=6, heads=2, blocks=4, cond_width=32,
                       cond_depth=4, cond_dilation_cycle=2, level=0, levels=2, labels=False)),
    "sep_enc_dec": ("small_vqvae", dict(sample_length=64 * 256),
                    "small_sep_enc_dec_prior",
                    dict(n_ctx=64, prior_width=64, prior_depth=10, heads=2, blocks=4, n_tokens=16,
                         prime_width=64, prime_depth=3, prime_heads=2, prime_blocks=4, level=1, levels=2,
                         merged_decoder=True)),
}


def golden_simple_prior(tag, bs=2, seed=4, chunk_size=7):
    from jukebox.hparams import setup_hparams
    from jukebox.make_models import make_vqvae, make_prior
    vq_name, vq_over, pr_name, pr_over = TINY_PRIORS[tag]
    vq = make_vqvae(setup_hparams(vq_name, dict(restore_vqvae="", **vq_over)), "cpu")
    hps = setup_hparams(pr_name, dict(restore_prior="", **pr_over))
    prior = make_prior(hps, vq, "cpu")
    named = load_synth(prior, seed)
    g = t.Generator().manual_seed(seed)
    arrays = {}
    z_conds = None
    if prior.x_cond:
        z_conds = [t.randint(0, vq.l_bins, (bs, prior.n_ctx // prior.cond_downsample), generator=g)]
        arrays["z_cond"] = z_conds[0]
    y = None
    if hps.labels:
        ys = []
        for i in range(bs):
            lyric = t.randint(0, hps.n_vocab, (hps.n_tokens,), generator=g).tolist() if hps.n_tokens else []
            genres = [int(t.randint(0, hps.y_bins[0], (1,), generator=g))]
            artist = int(t.randint(0, hps.y_bins[1], (1,), generator=g))
            total = int(hps.min_duration * hps.sr * 3)
            ys.append(prior.labeller.get_y_from_ids(artist, genres, lyric, total, 1000 * i))
        y = t.from_numpy(np.stack(ys)).long()
        arrays["y"] = y
    with t.no_grad():
        x_cond, y_cond, prime = prior.get_cond(z_conds, y)
        if x_cond is not None:
            arrays["x_cond"] = x_cond
        if y_cond is not None:
            arrays["y_cond"] = y_cond
        t.manual_seed(seed)
        if prior.single_enc_dec:
            z_in, xc = prior.prior_preprocess([prime], [None, x_cond])
            toks, preds32 = prior.prior.primed_sample(bs, z_in, xc, y_cond, fp16=False, get_preds=True,
                                                      chunk_size=chunk_size)
            toks = toks.view(bs, -1)
            _, preds16 = prior.prior.primed_sample(bs, toks[:, :-1].clone(), xc, y_cond, fp16=True,
                                                   get_preds=True, chunk_size=chunk_size)
            arrays.update(tokens=toks, preds32=preds32, preds16=preds16, x_cond_full=xc)
            arrays["z"] = prior.prior_postprocess(toks.clone())
        else:
            enc_kv = prior.get_encoder_kv(prime, fp16=False, sample=True)
            toks, preds32 = prior.prior.sample(bs, x_cond, y_cond, enc_kv, fp16=False, get_preds=True)
            toks = toks.view(bs, -1)
            enc_kv16 = prior.get_encoder_kv(prime, fp16=True, sample=True)
            _, preds16 = prior.prior.primed_sample(bs, toks[:, :-1].clone(), x_cond, y_cond, enc_kv16,
                                                   fp16=True, get_preds=True, chunk_size=chunk_size)
            arrays.update(tokens=toks, preds32=preds32, preds16=preds16)
            if enc_kv is not None:
                arrays["encoder_kv32"] = enc_kv
                arrays["encoder_kv16"] = enc_kv16.float()
    cfg = dict(tag=tag, vq_name=vq_name, vq_over=vq_over, pr_name=pr_name, pr_over=pr_over, seed=seed,
               chunk_size=chunk_size, n_ctx=int(prior.n_ctx), single_enc_dec=bool(prior.single_enc_dec))
    save(f"prior_{tag}", cfg, named, **arrays)


def golden_hparams():
    from jukebox.hparams import HPARAMS_REGISTRY, DEFAULTS, setup_hparams
    from jukebox.make_models import MODELS

    def clean(d):
        return {k: (list(v) if isinstance(v, tuple) else v) for k, v in d.items()}
    out = dict(registry={k: clean(v) for k, v in HPARAMS_REGISTRY.items()},
               defaults={k: clean(v) for k, v in DEFAULTS.items()},
               models={k: list(v) for k, v in MODELS.items()},
               resolved={k: clean(setup_hparams(k, {})) for k in HPARAMS_REGISTRY},
               # Python literals keep what JSON loses: which values are tuples (ast.literal_eval reads them back)
               resolved_repr={k: repr(dict(setup_hparams(k, {}))) for k in HPARAMS_REGISTRY})
    path = os.path.join(GOLDEN, "hparams.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote", path)


def golden_sample_level():
    """the reference's window planning / stitching (jukebox/sample.py:17-96) driven by the recording dummy prior of
    tests/test_sample_plan_cpu.py, one record per case"""
    import jukebox.sample as ref
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_sample_plan_cpu import CASES, case_id, run_sample_level
    out = {}
    for case in CASES:
        total, n_ctx, hop, have, bs, mbs = case
        if total >= n_ctx and have > total:
            continue
        out[case_id(case)] = run_sample_level(ref, *case)
    path = os.path.join(GOLDEN, "sample_level.json")
    with open(path, "w") as f:
        json.dump(out, f, sort_keys=True)
    print("wrote", path)


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    golden_hparams()
    golden_sample_level()
    golden_transformer("order9", n_in=64, n_ctx=48, n_head=2, n_depth=8, attn_order=9, blocks=4, bs=3)
    golden_transformer("order6", n_in=64, n_ctx=48, n_head=2, n_depth=8, attn_order=6, blocks=4, bs=2,
                       encoder_dims=10)
    golden_transformer("order12", n_in=64, n_ctx=96, n_head=2, n_depth=16, attn_order=12, blocks=8, bs=2,
                       prime_len=12)
    golden_transformer("order2_ragged", n_in=192, n_ctx=60, n_head=4, n_depth=6, attn_order=2, blocks=5, bs=5)
    golden_ca2d("xy", 48, 50, 64, 6, 2, 2, 4, True, True)
    golden_ca2d("plain", 48, 50, 64, 3, 1, 0, None, False, False)
    golden_ca2d("encdec_merged", 48, 50, 64, 8, 2, 6, 4, True, True, encoder_dims=10, merged_decoder=True)
    golden_vqvae("small", "small_vqvae", dict(sample_length=8192), bs=1)
    golden_vqvae("3level", "vqvae", dict(sample_length=128 * 40), bs=2)
    for tag in TINY_PRIORS:
        golden_simple_prior(tag)


if __name__ == "__main__":
    if len(sys.argv) > 1:
        os.makedirs(GOLDEN, exist_ok=True)
        for name in sys.argv[1:]:
            globals()["golden_" + name]()
    else:
        main()
