"""Window planning / stitching of jukebox_b200.sample against the UNMODIFIED reference's own loop
(jukebox/sample.py:17-96), both driven with the same recording dummy prior on the CPU.  What the reference's loop
returned and how it called the prior, case by case, is pinned in tests/golden/sample_level.json
(oracle/make_golden.py: golden_sample_level)."""
import itertools
import json
import os

import pytest
import torch

from golden_util import GOLDEN
from jukebox_b200.sample import plan_windows, Window
from jukebox_b200.utils.sample_utils import get_starts


class RecordingPrior:
    """prior.sample appends tokens that encode (call index, position), and records how it was called"""

    def __init__(self, n_ctx):
        self.n_ctx = n_ctx
        self.calls = []

    def get_z_conds(self, zs, start, end):
        return None

    def get_y(self, labels, start):
        return None

    def sample(self, n_samples, z=None, z_conds=None, y=None, sample_tokens=None, **kw):
        total = self.n_ctx if sample_tokens is None else sample_tokens
        self.calls.append((n_samples, z.shape[1], total, tuple(sorted(kw))))
        new = total - z.shape[1]
        assert new > 0
        fresh = 1000 * len(self.calls) + torch.arange(z.shape[1], total).view(1, -1).repeat(n_samples, 1)
        return torch.cat([z, fresh], dim=1)


class Hps(dict):
    __getattr__ = dict.__getitem__


CASES = [(total, n_ctx, hop, have, bs, mbs)
         for total, n_ctx, hop in [(40, 16, 8), (40, 16, 4), (16, 16, 8), (37, 16, 12), (10, 16, 8), (5, 16, 8), (33, 16, 16)]
         for have in (0, 3, 11, 16, 20) for bs, mbs in ((3, 2), (4, 4))]


def case_id(case):
    return "-".join(str(v) for v in case)


def run_sample_level(mod, total, n_ctx, hop, have, bs, mbs):
    """`mod.sample_level` on one case: {"zs": codes, "calls": prior calls} as JSON values, or {"error": type name}"""
    prior = RecordingPrior(n_ctx)
    zs = [torch.arange(have).view(1, -1).repeat(bs, 1)]
    hps = Hps(n_samples=bs)
    kw = dict(temp=0.9, fp16=True, max_batch_size=mbs)
    try:
        zs = mod.sample_level(zs, None, kw, 0, prior, total, hop, hps)
    except Exception as e:              # both sides must fail alike (e.g. negative slices)
        return dict(error=type(e).__name__)
    return dict(zs=zs[0].tolist(), calls=[[n, p, t, list(keys)] for n, p, t, keys in prior.calls])


@pytest.mark.parametrize("total,n_ctx,hop,have,bs,mbs", CASES)
def test_sample_level_matches_reference(total, n_ctx, hop, have, bs, mbs):
    import jukebox_b200.sample as ours
    if total >= n_ctx and have > total:
        pytest.skip("more tokens than the level holds")
    with open(os.path.join(GOLDEN, "sample_level.json")) as f:
        want = json.load(f)[case_id((total, n_ctx, hop, have, bs, mbs))]
    got = run_sample_level(ours, total, n_ctx, hop, have, bs, mbs)
    if "error" in want:
        assert "error" in got, got
        return
    assert "error" not in got, got
    assert got["zs"] == want["zs"]
    assert got["calls"] == want["calls"]


def test_plan_windows_shapes():
    assert plan_windows(0, 40, 16, 8) == [Window(s, 16) for s in get_starts(40, 16, 8)]
    assert plan_windows(0, 10, 16, 8) == [Window(0, 10)]
    assert plan_windows(12, 10, 16, 8) == [Window(6, 16)]
    for total, n_ctx, hop in itertools.product((16, 17, 31, 64), (16,), (4, 8, 16)):
        wins = plan_windows(0, total, n_ctx, hop)
        assert wins[0].start == 0 and wins[-1].start + n_ctx == total
        assert all(b.start - a.start <= hop for a, b in zip(wins, wins[1:]))
