#!/usr/bin/env python
"""bench.py - headline benchmark of the hot path (BASELINE.json: configs[1]).

    python bench.py --gpus 1 --steps 20 --warmup 5                    # our arm
    python bench.py --impl reference --gpus 1 --steps 20 --warmup 5   # the reference's CPU path (oracle port)
    torchrun ... bench.py --gpus N ...                                # one replica of the workload per rank
    python bench.py --workload small_upsampler | 5b_lyrics | vqvae_decode   # BASELINE configs[2], [3], [4]
    python bench.py ... --dump-outputs DIR                            # + what the last timed step computed, DIR/*.npy

Default workload "1b_lyrics": SimplePrior (prior_1b_lyrics hparams, n_ctx=8192 override -> 8576 positions incl.
384 lyric tokens), n_samples=16 per GPU, random-init synthetic weights, random labels and lyric tokens, fp16
sampling, temp 0.99.

One "step" = one EIGHTH of a sampling window: slice 0 = conditioning + 384-token lyric prefill + the first 1024
sampled positions, slices 1..7 = the next 1024 sampled positions each (one decode launch + one sampling launch
per position).  Steps cycle through the slices, so 8 consecutive steps are exactly one
`ConditionalAutoregressive2D.primed_sample` window (the same SamplingWindow code `sample` runs).  A step
processes n_samples x 1024 music tokens; metric = music tokens per second.

value       : device-resident inputs, CUDA-event time of the K timed steps, max over ranks
e2e         : ONE full window through the public call SimplePrior.sample(...) with labels copied from pinned
              host memory and the codes copied back to the host inside the timed region (plus NCCL
              scatter / gather for N > 1)
roofline    : the persistent decode kernel: algorithmic bytes per launch (fp16 Conv1D weights + fp32 x_out +
              LN / bias + KV rows read + KV rows written, SURVEY.md section 8d) / launch duration measured with
              CUDA events around single launches at 8 octile positions x 48 launches, vs MEASURED_PEAKS.json
cpu_baseline: oracle (numpy fp32 restatement of the reference) on the host cores, bounded sample; its fp16
              twin gives `parity_rel_err` against the GPU logits of the same positions
secondary   : VQ-VAE decode clips/s (BASELINE configs[4]) measured in the same run
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SLICES = 8

WORKLOADS = {
    # BASELINE configs[1]
    "1b_lyrics": dict(tag="1b_lyrics_top_prior_n_ctx8192_n_samples16", vq=("vqvae", dict(sample_length=1048576)),
                      prior=("prior_1b_lyrics", dict(n_ctx=8192)), n=16, chunk_size=32),
    # BASELINE configs[2] (README.md:115-117 recipe: the upsampler of the 2-level small_vqvae)
    "small_upsampler": dict(tag="small_upsampler_level0_n_ctx8192_n_samples16",
                            vq=("small_vqvae", dict(sample_length=8192 * 32)),
                            prior=("small_upsampler", dict(labels=False, level=0, levels=2)), n=16, chunk_size=32),
    # BASELINE configs[3]
    "5b_lyrics": dict(tag="5b_lyrics_top_prior_n_ctx8192_n_samples8", vq=("vqvae", dict(sample_length=1048576)),
                      prior=("prior_5b_lyrics", dict()), n=8, chunk_size=16),
}
SMALL = dict(tag="debug_small", vq=("vqvae", dict(sample_length=128 * 256)),
             prior=("prior_1b_lyrics", dict(n_ctx=256, prior_depth=16)), n=16, chunk_size=32)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="1b_lyrics", choices=list(WORKLOADS) + ["prior", "vqvae_decode"])
    ap.add_argument("--n-samples", type=int, default=0, help="samples per GPU (default: the workload's)")
    ap.add_argument("--cpu-tokens", type=int, default=0, help="positions per CPU-baseline step (0: calibrated)")
    ap.add_argument("--small", action="store_true", help="tiny debug configuration (not a valid bench number)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0), to compare two builds")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has none")
    if a.workload == "prior":
        a.workload = "1b_lyrics"
    return a


def workload_of(args):
    return SMALL if args.small else WORKLOADS[args.workload]


def bench_config(wl, n, n_ctx, positions, world):
    """the `config` object - identical for both arms (the driver compares them)"""
    return dict(workload=wl["tag"], n_ctx=n_ctx, positions_per_window=positions, n_samples_per_gpu=n,
                parallelism=f"replica x{world}",
                l2_policy="inputs larger than L2 (every token streams the full weight set from HBM)",
                step=f"1/{N_SLICES} window: {n_ctx // N_SLICES} sampled positions x n_samples "
                     "(slice 0 also holds conditioning + prefill of the given tokens)")


# ----------------------------------------------------------------------------------------------
def hps_pair(wl):
    from jukebox_b200.hparams import setup_hparams
    vq = setup_hparams(wl["vq"][0], dict(restore_vqvae="", **wl["vq"][1]))
    pr = setup_hparams(wl["prior"][0], dict(restore_prior="", **wl["prior"][1]))
    return vq, pr


def synth_fill(model, seed):
    """random-init synthetic weights with O(1) activations (same scale rules as oracle/synth.py),
    drawn on the GPU"""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            last = name.split(".")[-1]
            z = torch.randn(p.shape, generator=g, device=p.device, dtype=torch.float32)
            if p.dim() == 1:
                if last == "weight" and "ln" in name.split(".")[-2]:
                    z = 1.0 + 0.1 * z
                else:
                    z = 0.1 * z
            elif last == "w":
                z = z * ((1.5 if name.endswith("c_attn.w") else 1.0) / p.shape[0] ** 0.5)
            elif "pos_emb" in name:
                z = z * 0.5
            elif p.dim() == 3:
                z = z / (p.shape[1] * p.shape[2]) ** 0.5
            elif p.dim() == 2:
                z = z * (2.0 / p.shape[1] ** 0.5)
            p.copy_(z.to(p.dtype))


def build_prior(wl, seed=0):
    import torch
    from jukebox_b200.make_models import make_vqvae, make_prior
    vq_h, pr_h = hps_pair(wl)
    with torch.device("cuda"):
        vqvae = make_vqvae(vq_h, "cuda")
        prior = make_prior(pr_h, vqvae, "cuda")
    synth_fill(prior, seed)
    return prior, pr_h


def make_labels(prior, hps, n, seed):
    """random artist / genre ids and lyric tokens in the label layout of the workload (data/labels.py)"""
    import numpy as np
    import torch
    if not hps.labels:
        return None
    rng = np.random.RandomState(seed)
    n_genre, n_artist = hps.y_bins
    ys = []
    for _ in range(n):
        lyric = rng.randint(0, hps.n_vocab, size=prior.n_tokens).tolist()
        genres = [int(rng.randint(0, n_genre)) for _ in range(min(hps.max_bow_genre_size, 1 + rng.randint(0, 3)))]
        ys.append(prior.labeller.get_y_from_ids(int(rng.randint(0, n_artist)), genres, lyric, 180 * hps.sr, 0))
    y = torch.from_numpy(np.stack(ys)).long()
    y[:, 2] = int(prior.sample_length)
    return y


def make_z_conds(prior, n, seed):
    import torch
    if not prior.x_cond:
        return None
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, prior.l_bins, (n, prior.n_ctx // prior.cond_downsample), generator=g)]


def layer_geometry(prior):
    tr = prior.prior.transformer
    l0 = tr._attn_mods[0]
    return dict(W=tr.n_in, L=tr.n_ctx, S=l0.attn.n_state, M=l0.mlp.c_fc.n_out, bc=getattr(tr, "block_ctx", tr.n_ctx),
                P=l0.attn._prime_len if tr.prime_len else 0, E=tr.encoder_dims or 0,
                funcs=[b.attn_func for b in tr._attn_mods])


def weight_bytes(prior):
    tr = prior.prior.transformer
    W = tr.n_in
    wb = 0
    for blk in tr._attn_mods:
        for c in (blk.attn.c_attn, blk.attn.c_proj, blk.mlp.c_fc, blk.mlp.c_proj):
            wb += c.w.numel() * 2 + c.b.numel() * 4
        wb += 4 * W * 4
    return wb + prior.prior.bins * W * 4            # fp32 x_out, as the reference keeps it


def algorithmic_bytes(prior, n, positions):
    """sum over `positions` (0-indexed) of bytes_step(t, n) (SURVEY.md section 8d)"""
    g = layer_geometry(prior)
    wb = weight_bytes(prior)
    row = 2 * g["S"] * 2                            # one K row + one V row, fp16
    bc, P = g["bc"], g["P"]
    total = 0
    for p in positions:
        kv = 0
        for f in g["funcs"]:
            if f == 0:
                kv += (p + 1) + 1
            elif f == 1:
                kv += (p % bc + 1) + 1
            elif f == 2:
                kv += (p // bc + 1) + 1
            elif f == 3:
                kv += (bc if p >= bc else 0) + 1
            elif f == 7:
                kv += min(p + 1, P) + (1 if p < P else 0)
            elif f == 6:
                kv += g["E"]
        total += wb + n * kv * row
    return total, wb


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            return None
        sm, mx, reasons = [], 0, set()
        for line in out.strip().splitlines():
            f = [s.strip() for s in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def ncu_dram_bytes(path):
    """dram__bytes_read.sum + dram__bytes_write.sum of a committed ncu capture of the decode kernel (bytes per
    launch), or None"""
    try:
        tot = 0.0
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        for line in open(path):
            f = line.split()
            if len(f) >= 4 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and f[1] == "=":
                tot += float(f[2]) * scale.get(f[3], 1.0)
        return tot or None
    except Exception:
        return None


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 20          # elements kept of an output too large to dump whole


def dump_outputs(out_dir, arrays):
    """name -> float32 / float64 array, written as out_dir/<name>.npy (at most DUMP_LIMIT_BYTES in all)"""
    import numpy as np
    arrays = {k: np.ascontiguousarray(v) for k, v in arrays.items()}
    assert all(v.dtype in (np.float32, np.float64) for v in arrays.values())
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"{total} bytes of outputs exceed the dump limit of {DUMP_LIMIT_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def sample_of(x):
    """a fixed sample of DUMP_SAMPLE elements of a large CUDA tensor, flattened (indices seeded, sorted): the same
    positions from run to run for the same shape"""
    import numpy as np
    import torch
    flat = x.reshape(-1)
    if flat.numel() <= DUMP_SAMPLE:
        return flat.cpu().numpy()
    idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_SAMPLE, replace=False))
    return flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle (numpy restatement of the reference's CA2D.sample body) on the host cores
# ----------------------------------------------------------------------------------------------
def set_blas_threads(k):
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=k)
        return True
    except Exception:
        return False


def oracle_for(sd, cfg):
    from oracle.transformer_np import PriorOracle
    return PriorOracle(sd, cfg["input_dims"], cfg["bins"], cfg["width"], cfg["depth"], cfg["heads"],
                       attn_order=cfg["attn_order"], blocks=cfg["blocks"], x_cond=cfg["x_cond"], y_cond=cfg["y_cond"],
                       encoder_dims=cfg["encoder_dims"], merged_decoder=cfg["merged_decoder"],
                       prime_len=cfg["prime_len"])


def oracle_inputs(cfg, n, tokens, seed):
    import numpy as np
    rng = np.random.RandomState(seed)
    toks = rng.randint(0, min(79, cfg["bins"]), size=(n, tokens + 1))
    W = cfg["width"]
    yc = rng.standard_normal((n, 1, W)).astype(np.float32) if cfg["y_cond"] else None
    xc = (0.1 * rng.standard_normal((n, 1, W))).astype(np.float32) if cfg["x_cond"] else np.zeros((n, 1, W), np.float32)
    enc = rng.standard_normal((n, cfg["encoder_dims"], W)).astype(np.float32) if cfg["encoder_dims"] else None
    return toks, xc, yc, enc


def pick_threads(orc, cfg, n):
    """BLAS thread count by a short sweep (round 1: all 128 hardware threads on [16 x 2048] GEMVs were 4x slower
    than a quarter of them on one box).  Returns (threads, tokens/s of the probe)."""
    cores = os.cpu_count() or 1
    cands = sorted({max(1, min(cores, c)) for c in (8, 16, 32, 64, cores)})
    toks, xc, yc, enc = oracle_inputs(cfg, n, 2, 99)
    best = (cands[0], 0.0)
    for c in cands:
        if not set_blas_threads(c):
            return cores, 0.0
        orc.logits(toks, xc, yc, enc, False, n_steps=1)
        t0 = time.time()
        orc.logits(toks, xc, yc, enc, False, n_steps=2)
        v = n * 2 / (time.time() - t0)
        if v > best[1]:
            best = (c, v)
    set_blas_threads(best[0])
    return best


def cpu_sample(orc, cfg, n, tokens, seed=0):
    toks, xc, yc, enc = oracle_inputs(cfg, n, tokens, seed)
    t0 = time.time()
    out = orc.logits(toks, xc, yc, enc, False, n_steps=tokens)
    dt = time.time() - t0
    return n * tokens / dt, dt, (toks, xc, yc, enc, out)


def oracle_state_from(prior):
    sd = {k: v.detach().float().cpu().numpy() for k, v in prior.prior.state_dict().items()}
    return sd, oracle_cfg(prior)


def oracle_cfg(prior):
    ca = prior.prior
    tr = ca.transformer
    return dict(input_dims=tr.n_ctx, bins=ca.bins, width=tr.n_in, depth=tr.n_depth, heads=tr.n_head,
                blocks=tr.blocks, prime_len=tr.prime_len, attn_order=prior_attn_order(prior), x_cond=bool(ca.x_cond),
                y_cond=bool(ca.y_cond), encoder_dims=tr.encoder_dims or 0,
                merged_decoder=not ca.add_cond_after_transformer)


def prior_attn_order(prior):
    from jukebox_b200.transformer.transformer import attn_func_of
    funcs = [b.attn_func for b in prior.prior.transformer._attn_mods]
    for order in (0, 2, 12, 10, 6, 9, 8, 7, 1, 11):
        try:
            if [attn_func_of(order, d) for d in range(len(funcs))] == funcs:
                return order
        except Exception:
            pass
    raise RuntimeError("attention order of the prior not recognised")


def synth_oracle_state(wl):
    """reference arm without a GPU model: same shapes, numpy-generated weights"""
    import numpy as np
    import torch
    from jukebox_b200.make_models import make_vqvae, make_prior
    vq_h, pr_h = hps_pair(wl)
    with torch.device("meta"):
        vqvae = make_vqvae(vq_h, "meta")
        prior = make_prior(pr_h, vqvae, "meta")
    rng = np.random.default_rng(0)
    sd = {}
    for k, v in prior.prior.state_dict().items():
        shape = tuple(v.shape)
        a = rng.standard_normal(shape, dtype=np.float32)
        if len(shape) == 1:
            a = (1.0 + 0.1 * a) if (k.endswith("weight") and "ln" in k) else 0.1 * a
        elif k.endswith(".w"):
            a *= (1.5 if k.endswith("c_attn.w") else 1.0) / np.sqrt(shape[0])
        elif "pos_emb" in k:
            a *= 0.5
        else:
            a *= 2.0 / np.sqrt(shape[-1])
        sd[k] = a.astype(np.float32)
    return sd, oracle_cfg(prior), prior.n_ctx, prior.prior.input_dims


def run_reference(args, rank, world):
    """the reference's own CPU implementation of the path (its numpy port, all host cores through BLAS) on the
    same workload shape; each step a bounded sample sized so the whole run stays within ~2.5 minutes"""
    if rank != 0:
        return
    wl = workload_of(args)
    n = args.n_samples or wl["n"]
    with contextlib.redirect_stdout(sys.stderr):
        sd, cfg, n_ctx, positions = synth_oracle_state(wl)
        orc = oracle_for(sd, cfg)
    threads, probe = pick_threads(orc, cfg, n)
    tokens = args.cpu_tokens
    if tokens <= 0:     # calibrate: (warmup + steps) samples in ~150 s
        tokens = int(max(1, min(24, probe * 150.0 / max(1, args.warmup + args.steps) / n)))
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt, _ = cpu_sample(orc, cfg, n, tokens, seed=i)
        if i >= args.warmup:
            vals.append((v, dt))
    tot = sum(dt for _, dt in vals)
    value = n * tokens * len(vals) / tot
    sample = (f"{tokens} token positions (0..{tokens - 1}) x {n} samples per step, fp32 numpy port of the reference's "
              f"sample loop, {threads} BLAS threads (best of a sweep) of {os.cpu_count()} logical cores")
    line = dict(metric="top_prior_tokens_per_sec", value=value, unit="tokens/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * tot / len(vals), higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=bench_config(wl, n, n_ctx, positions, world),
                cpu_baseline=dict(value=value, unit="tokens/s", cores=threads, kind="port", sample=sample),
                e2e=dict(value=value, unit="tokens/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
def measure_vqvae(args, rank, world, local, steps, warmup, small=False, dump=None):
    """BASELINE configs[4]: 3-level VQ-VAE decode, sample_length 1048576, bs 16 per GPU; one step = every
    clip decoded at every level exactly as sample.py:108 does (decode(zs[l:], start_level=l, bs_chunks=N)).
    Returns the result dict (all ranks; times are max over ranks).  `dump`: directory that receives the audio the
    last timed step decoded from each start level l, a fixed sample of it (sample_of), as audio_level<l>.npy."""
    import torch
    import torch.distributed as dist
    from jukebox_b200.hparams import setup_hparams
    from jukebox_b200.make_models import make_vqvae
    from jukebox_b200 import _lib
    T = 1048576 if not small else 65536
    n = 16 if not small else 2
    with contextlib.redirect_stdout(sys.stderr), torch.device("cuda"):
        vq = make_vqvae(setup_hparams("vqvae", dict(sample_length=T, restore_vqvae="")), "cuda")
    synth_fill(vq, 5)
    for blk in vq.bottleneck.level_blocks:
        blk.k.normal_()
    g = torch.Generator(device="cuda").manual_seed(rank)
    zs_host = [torch.randint(0, vq.l_bins, (n, T // int(h)), generator=g, device="cuda").cpu().pin_memory()
               for h in vq.hop_lengths]

    def step(zs):
        return [vq.decode(zs[l:], start_level=l, bs_chunks=n) for l in range(vq.levels)]

    zs_dev = [z.cuda() for z in zs_host]
    for _ in range(max(warmup, 1)):
        step(zs_dev)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0 = _lib.CALLS
    last = None
    e0.record()
    for _ in range(steps):
        last = None                    # one step's audio is freed before the next is decoded, as when discarded
        last = step(zs_dev)
    e1.record()
    torch.cuda.synchronize()
    launches = _lib.CALLS - c0
    if dump and rank == 0:
        dump_outputs(dump, {f"audio_level{l}": sample_of(x) for l, x in enumerate(last)})
    del last
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    t0 = time.perf_counter()
    for _ in range(steps):
        outs = step([z.cuda(non_blocking=True) for z in zs_host])
        x_host = outs[0][:1].cpu()           # audio of the finest level, first clip (result read-back)
    torch.cuda.synchronize()
    wall = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(wall, op=dist.ReduceOp.MAX)
    del outs, zs_dev
    torch.cuda.empty_cache()
    clips = world * n * steps
    value = clips / (float(ms) * 1e-3)
    flops_clip = 373e9 * (T / 1048576)
    bytes_plan = 7.3e9 * (T / 1048576)
    peaks = load_peaks()
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    tf = float(peaks.get("bf16_tflops", 1690.0))
    t_clip = float(ms) * 1e-3 / (n * steps)
    traffic = ncu_dram_bytes(os.path.join(ROOT, "profiles", "ncu_vqvae_resblock_r02.txt"))
    return dict(metric="vqvae_decode_clips_per_sec", value=value, unit="clips/s (3 levels each)", n_gpus=world,
                steps=steps, warmup=warmup, ms_per_step=float(ms) / steps, higher_is_better=True, scaling="weak",
                dtype="f32", data="synthetic",
                config=dict(workload="vqvae_3level_decode_sample_length%d_bs%d" % (T, n),
                            l2_policy="activations (268 MB per conv at level 0) exceed L2"),
                e2e=dict(value=clips / float(wall), unit="clips/s",
                         h2d_bytes_per_step=int(sum(z.numel() for z in zs_host) * 8),
                         d2h_bytes_per_step=int(x_host.numel() * 4),
                         api="VQVAE.decode(zs[l:], start_level=l, bs_chunks=N) for l in 0..2"),
                gpu_launches=int(launches),
                roofline=dict(bound="hbm", achieved=bytes_plan / t_clip / 1e9, peak=hbm, unit="GB/s",
                              frac=bytes_plan / t_clip / 1e9 / hbm, traffic=traffic,
                              traffic_source="profiles/ncu_vqvae_resblock_r02.txt: dram bytes of ONE launch of the dominant "
                                             "kernel, resblock_t5_kernel<64> on [4, 262144, 64] (algorithmic: 537 MB in + out)",
                              note="per-block-fused activation plan 7.3 GB fp32 per clip (SURVEY 8d); compute side: "
                                   "%.1f TFLOP/s achieved of %.0f (bf16 dense peak)" % (flops_clip / t_clip / 1e12, tf)))


# ----------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import numpy as np
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from jukebox_b200 import build as jk_build
    if not os.path.exists(os.path.join(ROOT, "jukebox_b200", "libjkb200.so")):
        jk_build.build()
    with contextlib.redirect_stdout(sys.stderr):      # model-construction chatter must not precede the JSON line
        from jukebox_b200.utils.dist_sampling import scatter_rows, gather_rows, seed_per_rank
    seed_per_rank(0)
    if args.workload == "vqvae_decode":
        res = measure_vqvae(args, rank, world, local, args.steps, args.warmup, args.small, dump=args.dump_outputs)
        if rank == 0:
            res["vs_baseline"] = None
            print(json.dumps(res))
        if world > 1:
            dist.destroy_process_group()
        return

    from jukebox_b200 import _lib
    from jukebox_b200.prior.autoregressive import SamplingWindow
    wl = workload_of(args)
    quiet = contextlib.redirect_stdout(io.StringIO())
    with contextlib.redirect_stdout(sys.stderr):
        prior, hps = build_prior(wl, seed=rank)
    n = args.n_samples or wl["n"]
    ca = prior.prior
    L = ca.input_dims                       # positions per window incl. given (lyric) tokens
    n_ctx = prior.n_ctx
    sample_kw = dict(fp16=True, temp=0.99, chunk_size=wl["chunk_size"])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # conditioning for all ranks lives on rank 0's host; every rank needs its own slice
    y_all = make_labels(prior, hps, n * world, seed=1234)
    zc_all = make_z_conds(prior, n * world, seed=4321)
    y_all_host = y_all.pin_memory() if y_all is not None else None
    zc_all_host = [z.pin_memory() for z in zc_all] if zc_all is not None else None
    y_dev = y_all_host[rank * n:(rank + 1) * n].cuda() if y_all_host is not None else None
    zc_dev = [z[rank * n:(rank + 1) * n].cuda() for z in zc_all_host] if zc_all_host is not None else None

    def window_e2e():
        """public API with host buffers: labels / upper-level codes H2D (+ NCCL scatter), sample, codes D2H (+ gather)"""
        dev = torch.device("cuda", local)
        y = scatter_rows(y_all_host, n, dev) if y_all_host is not None else None
        zc = [scatter_rows(z, n, dev) for z in zc_all_host] if zc_all_host is not None else None
        z = prior.sample(n_samples=n, z=None, z_conds=zc, y=y, **sample_kw)
        return gather_rows(z).cpu()

    def begin_window():
        """conditioning + window begin (prefill of the given tokens); the reference's SimplePrior.sample head
        (prior/prior.py:262-279)"""
        with torch.no_grad():
            x_cond, y_cond, prime = prior.get_cond(zc_dev, y_dev)
            if prior.single_enc_dec:
                z_in, x_cond = prior.prior_preprocess([prime], [None, x_cond])
                enc_kv = None
            else:
                z_in = torch.zeros(n, 0, dtype=torch.long, device="cuda")
                enc_kv = prior.get_encoder_kv(prime, fp16=True, sample=True)
            return SamplingWindow(ca, n, z_in, x_cond, y_cond, enc_kv, True, 0.99, 0, 0.0, False, None)

    state = dict(win=None, k=0)
    per_slice = n_ctx // N_SLICES

    def slice_step():
        k = state["k"]
        if k == 0:
            state["win"] = begin_window()
        win = state["win"]
        lo = win.pos
        win.advance(win.P + per_slice * (k + 1) if k < N_SLICES - 1 else win.sample_tokens)
        state["last"] = (win, lo, win.pos)         # positions this step sampled (--dump-outputs)
        if k == N_SLICES - 1:
            if prior.single_enc_dec:
                prior.prior_postprocess(win.finish())
            else:
                win.finish()
            state["win"] = None
        state["k"] = (k + 1) % N_SLICES

    with quiet:
        for _ in range(args.warmup):
            slice_step()
    # ---- value: K slice-steps, device-resident inputs ------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls0 = _lib.CALLS
    first_slice = state["k"]
    torch.cuda.profiler.start()                # `ncu --profile-from-start off` captures the timed region only
    e0.record()
    with quiet:
        for _ in range(args.steps):
            slice_step()
    e1.record()
    barrier()
    torch.cuda.profiler.stop()
    launches_timed = _lib.CALLS - calls0       # C-ABI calls that launched our kernels in the timed region
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_value = float(ms)
    if args.dump_outputs and rank == 0:
        # the codes the last timed step sampled (token ids of the window, exact in float64) and the logits of its last
        # position; same arguments, same inputs: weights, labels and the sampler's Philox key all come from fixed seeds
        win, lo, hi = state["last"]
        dump_outputs(args.dump_outputs, dict(tokens=win.tokens[:, lo:hi].double().cpu().numpy(),
                                             logits=win.lbuf.float().cpu().numpy()))
    with quiet:                                # run the open window to its end (engine back to a clean state)
        while state["k"] != 0:
            slice_step()
    # ---- e2e: one full window through the public API with host buffers ---------------------------
    if world > 1:
        # NCCL sets a collective up on its first use (hundreds of ms for the first broadcast / gather of a process): a
        # sampler that runs window after window pays that once, so the two collectives of a window are warmed up here
        # on dummy rows; the timed window below still does its own scatter and gather
        with quiet:
            gather_rows(scatter_rows(torch.zeros(world * n, 4, dtype=torch.long).pin_memory(), n, torch.device("cuda", local)))
        torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    with quiet:
        z_host = window_e2e()
    barrier()
    wall_e2e = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(wall_e2e, op=dist.ReduceOp.MAX)
    ms_e2e = float(wall_e2e) * 1e3          # host-side wall time of the call, barrier to barrier (includes the D2H)
    clocks = sampler.stop() if sampler else None
    # ---- breakdown of the once-per-window work (untimed legs; reported) ----------------------------
    def timed(fn):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); r = fn(); b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b), r
    with quiet, torch.no_grad():
        t_cond, cond = timed(lambda: prior.get_cond(zc_dev, y_dev))
        t_enc = None
        if not prior.single_enc_dec and prior.n_tokens != 0 and prior.use_tokens:
            t_enc, _ = timed(lambda: prior.get_encoder_kv(cond[2], fp16=True, sample=True))
        t_begin, win = timed(begin_window)
    breakdown = dict(conditioning_ms=t_cond, lyric_encoder_ms=t_enc, window_begin_ms=t_begin,
                     note="window_begin = conditioning + encoder + c_enc_kv + prefill of the given tokens")
    # ---- roofline: single decode launches at 8 octile positions, CUDA events around each ----------------
    eng = ca._engine(n)
    toks = torch.randint(0, min(ca.bins, 79), (n, L), device="cuda")
    lbuf = torch.empty(n, ca.bins, device="cuda")
    reps = 48 if not args.small else 4
    octile = [min(L - reps - 1, max(win.P, int(L * (2 * i + 1) / 16))) for i in range(8)]
    kern_ms, positions = 0.0, []
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * reps)]
    for p0 in octile:
        eng.reset(p0)
        for _ in range(3):
            eng.step(n, tokens=toks, y_cond=win.y_cond, x_cond=win.x_cond, logits=lbuf, logit_bias=win.logit_bias)
        eng.reset(p0)
        torch.cuda.synchronize()
        for i in range(reps):
            ev[2 * i].record()
            eng.step(n, tokens=toks, y_cond=win.y_cond, x_cond=win.x_cond, logits=lbuf, logit_bias=win.logit_bias)
            ev[2 * i + 1].record()
        torch.cuda.synchronize()
        kern_ms += sum(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(reps))
        positions += list(range(p0, p0 + reps))
    glog = lbuf.clone()
    ca.transformer.del_cache()
    total_bytes, w_bytes = algorithmic_bytes(prior, n, positions)
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = total_bytes / (kern_ms * 1e-3) / 1e9
    cap = os.path.join(ROOT, "profiles", "ncu_decode_step_final_p4000_r02.txt")      # the shipped kernel, position 4000
    traffic = None if args.small or args.workload != "1b_lyrics" else ncu_dram_bytes(cap)
    roof = dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=traffic,
                traffic_source="profiles/ncu_decode_step_final_p4000_r02.txt (ncu --set full, one launch at position 4000; "
                               "positions 500 / 8000: ncu_decode_step_final_p500_r02.txt / _p8000_r02.txt)",
                kernel="jk_decode_step_kernel", launches=len(positions), avg_launch_us=1e3 * kern_ms / len(positions),
                positions=f"{reps} consecutive launches from each of {octile}",
                algorithmic_bytes_per_launch=total_bytes / len(positions), weight_bytes_per_launch=w_bytes,
                peak_source="MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s")
    # ---- secondary metric: VQ-VAE decode (BASELINE configs[4]) -----------------------------------------
    secondary = None
    if not args.no_secondary and args.workload == "1b_lyrics":
        try:
            secondary = measure_vqvae(args, rank, world, local, 2, 1, args.small)
        except Exception as e:      # the headline line must not die with the secondary leg
            secondary = dict(error=repr(e))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    tokens_per_step = n * per_slice
    value = world * tokens_per_step * args.steps / (ms_value * 1e-3)
    e2e_v = world * n * n_ctx / (ms_e2e * 1e-3)
    h2d = (y_all_host.numel() * 8 if y_all_host is not None else 0) + \
          (sum(z.numel() for z in zc_all_host) * 8 if zc_all_host is not None else 0)
    line = dict(metric="top_prior_tokens_per_sec", value=value, unit="tokens/s", n_gpus=world, steps=args.steps,
                warmup=args.warmup, ms_per_step=ms_value / args.steps, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="fp16", data="synthetic",
                config=bench_config(wl, n, n_ctx, L, world),
                slices=dict(first_timed=first_slice, per_window=N_SLICES, positions_per_slice=per_slice),
                e2e=dict(value=e2e_v, unit="tokens/s", h2d_bytes_per_step=int(h2d),
                         d2h_bytes_per_step=int(z_host.numel() * 8), ms_per_step=ms_e2e, windows=1,
                         step="one full window (8 slices) through the public call",
                         api=f"SimplePrior.sample(n_samples, z=None, z_conds, y, fp16=True, temp=0.99, "
                             f"chunk_size={wl['chunk_size']})"),
                gpu_launches=int(launches_timed), roofline=roof, clocks=clocks, once_per_window=breakdown)
    if secondary is not None:
        line["secondary"] = secondary
    if not args.no_cpu_baseline and world == 1:      # reported at N = 1 only (bounded sample, rank 0)
        try:
            sd, cfg = oracle_state_from(prior)
            orc = oracle_for(sd, cfg)
            threads, probe = pick_threads(orc, cfg, n)
            tokens = args.cpu_tokens or int(max(2, min(24, probe * 25.0 / n)))
            v, dt, (otoks, xc, yc, enc, _) = cpu_sample(orc, cfg, n, tokens)
            line["cpu_baseline"] = dict(value=v, unit="tokens/s", cores=threads, kind="port",
                                        sample=f"{tokens} token positions (0..{tokens - 1}) x {n} samples, fp32 numpy port "
                                               f"of the reference's sample loop, {threads} BLAS threads (best of a sweep) "
                                               f"of {os.cpu_count()} logical cores, {dt:.1f} s")
            # parity: the oracle's fp16 twin vs the decode kernel's logits on the same inputs, same positions
            np_pos = min(tokens, 8)
            ref16 = orc.logits(otoks, xc, yc, enc, True, n_steps=np_pos)
            gt = torch.from_numpy(otoks).cuda()
            gx = torch.from_numpy(np.broadcast_to(xc, (n, 1, cfg["width"])).copy()).cuda() if ca.x_cond else None
            gy = torch.from_numpy(yc).cuda().view(n, -1).contiguous() if yc is not None else None
            ca.transformer.del_cache()
            if enc is not None:
                eng.set_encoder_kv(torch.from_numpy(enc).cuda())
            got = []
            gb = None       # x_cond . x_out^T, as SamplingWindow computes it for the tensor-core logits product
            if gx is not None and ca.add_cond_after_transformer and eng.has_logits_gemm:
                from jukebox_b200.transformer import f32 as _f32
                gb = _f32.linear_nk(gx.reshape(n, cfg["width"]), ca.x_out.weight).view(n, 1, ca.bins)
            for _ in range(np_pos):
                eng.step(n, tokens=gt, y_cond=gy, x_cond=gx, logits=glog, logit_bias=gb)
                got.append(glog.clone())
            ca.transformer.del_cache()
            got = torch.stack(got, 1).cpu().numpy()
            line["parity_rel_err"] = float(np.abs(got - ref16).max() / np.abs(ref16).max())
            line["parity"] = dict(what="max|logits_gpu - logits_oracle_fp16| / max|logits_oracle_fp16|",
                                  positions=f"0..{np_pos - 1}", samples=n, full_size=not args.small)
        except Exception as e:
            line["cpu_baseline_error"] = repr(e)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
