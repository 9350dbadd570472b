"""CPU pins of test_minibatch_envelope_edge_gpu.py: the row-blocked float64 restatement ``restate_mb`` equals the
minibatch oracles (numpy formula sheet, head autograd, NaN law) whatever its block size; the checker it feeds catches a
restatement that reads the last image's keys from the image before; and every GPU case sits at the edge of the
envelope, one image (one rank) short of the RuntimeError."""
import os
import re

import numpy as np
import pytest
import torch

import head_minibatch_oracle as hmo
import minibatch_oracle as mbo
import test_minibatch_envelope_edge_gpu as te
from test_benchmarked_sizes import _dense, _problem
from test_benchmarked_sizes_gpu import TOL, check_grads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(8, 6, 7), (12, 5, 5)]        # two layers; P = 40 > HW = 25 in the second (duplicate ids), not a multiple of 128
B, P = 3, 40                            # N = 120: block_rows = 7 straddles the image boundaries and does not divide N


def _oracle(src, tgt, ids, tau):
    out = [mbo.layer_loss_and_grad_np_mb(s.numpy(), t.numpy(), i.numpy(), tau, len(src)) for s, t, i in zip(src, tgt, ids)]
    return sum(l for l, _ in out) / len(src), [g for _, g in out]


def _max_logit(src, tgt, ids, tau):
    """max |q k^T / tau| of layer 0 over every (row, key) pair of the batch."""
    c = src[0].shape[1]
    k = torch.nn.functional.normalize(te._rows(src[0], ids[0]).reshape(-1, c), dim=1)
    q = torch.nn.functional.normalize(te._rows(tgt[0], ids[0]).reshape(-1, c), dim=1)
    return (q @ k.t() / tau).abs().max().item()


@pytest.mark.parametrize("tau", [0.07, 0.015])          # 0.015: 1 / tau > 50, the +-50 clamp binds
def test_restate_mb_equals_the_numpy_oracle(tau):
    src, tgt, ids = _problem(3, B, SHAPES, P)
    assert ids[1].unique().numel() < P
    assert (_max_logit(src, tgt, ids, tau) > 50.0) == (tau < 0.02)
    loss, ref, heads = te.restate_mb(src, tgt, ids, tau, block_rows=7)
    assert heads is None
    want, grads = _oracle(src, tgt, ids, tau)
    assert loss == pytest.approx(want, rel=1e-12)
    for got, r in zip(_dense(ref, SHAPES, B), grads):
        assert np.abs(got.numpy() - r).max() <= 1e-12 * np.abs(r).max()


def test_block_size_does_not_change_the_result():
    src, tgt, ids = _problem(8, B, SHAPES, P)
    l7, r7, _ = te.restate_mb(src, tgt, ids, 0.015, block_rows=7)
    ln, rn, _ = te.restate_mb(src, tgt, ids, 0.015, block_rows=B * P)
    assert l7 == pytest.approx(ln, rel=1e-13)
    for (pa, a), (pb, b) in zip(r7, rn):
        assert torch.equal(pa, pb) and (a - b).abs().max() <= 1e-13 * b.abs().max()


def test_head_restate_mb_equals_the_head_oracle_and_its_autograd():
    src, tgt, ids = _problem(4, B, SHAPES, P)
    g = torch.Generator().manual_seed(9)
    heads = [[0.3 * torch.randn(*s, generator=g, dtype=torch.float64) for s in ((32, c), (32,), (32, 32), (32,))]
             for c, _, _ in SHAPES]
    loss, ref, hg = te.restate_mb(src, tgt, ids, 0.07, heads, block_rows=7)
    t = [x.clone().requires_grad_() for x in tgt]
    hp = [[p.clone().requires_grad_() for p in h] for h in heads]
    want = hmo.head_minibatch_loss(src, t, ids, hp, 0.07)
    want.backward()
    assert loss == pytest.approx(want.item(), rel=1e-12)
    for got, x in zip(_dense(ref, SHAPES, B), t):
        assert (got - x.grad).abs().max() <= 1e-12 * x.grad.abs().max()
    for gs, ps in zip(hg, hp):
        for a, p in zip(gs, ps):
            assert (a - p.grad).abs().max() <= 1e-12 * p.grad.abs().max()


@pytest.mark.parametrize("side", ["tgt", "src"])
def test_nan_law_of_the_oracle(side):
    """A NaN in one sampled target patch: layer 1 contributes 0, its gradient is NaN in every channel of that patch
    and 0 elsewhere.  A NaN in one key instead: layer 1 contributes 0 and its gradient is 0.  Layer 0 is untouched."""
    src, tgt, ids = _problem(5, B, SHAPES, P)
    pos = ids[1][-1].item()
    (tgt if side == "tgt" else src)[1][B - 1, 2].view(-1)[pos] = float("nan")
    loss, ref, _ = te.restate_mb(src, tgt, ids, 0.07, block_rows=7)
    want, grads = _oracle(src, tgt, ids, 0.07)
    assert loss == pytest.approx(want, rel=1e-12) and want == pytest.approx(_oracle(src[:1], tgt[:1], ids[:1], 0.07)[0] / 2)
    dense = _dense(ref, SHAPES, B)
    for got, r in zip(dense, grads):
        assert np.array_equal(np.isnan(got.numpy()), np.isnan(r))
        fin = ~np.isnan(r)
        assert np.abs(got.numpy()[fin] - r[fin]).max() <= 1e-12 * np.abs(r[fin]).max(initial=1e-300)
    nan = torch.isnan(dense[1])
    if side == "tgt":
        assert nan[B - 1].view(SHAPES[1][0], -1)[:, pos].all() and int(nan.sum()) == SHAPES[1][0]
    else:
        assert not nan.any()
    assert (dense[1][~nan] == 0).all()


def test_a_slot_off_by_one_image_fails_the_checker():
    """A restatement that takes the last image's keys from the image before it -- what a wrong slot offset in
    k_loss_tc_mb_gn would compute -- fails check_grads at the tc_bf16x3 tolerance."""
    src, tgt, ids = _problem(6, 4, SHAPES, P)
    _, ref, _ = te.restate_mb(src, tgt, ids, 0.07)
    shifted = [s.clone() for s in src]
    for s in shifted:
        s[-1] = s[-2]
    _, wrong, _ = te.restate_mb(shifted, tgt, ids, 0.07)
    got = _dense(wrong, SHAPES, 4, torch.float32)
    assert check_grads(_dense(ref, SHAPES, 4, torch.float32), ref, ids, TOL["tc_bf16x3"][1], "reference") <= 1e-6
    with pytest.raises(AssertionError, match="block error"):
        check_grads(got, ref, ids, TOL["tc_bf16x3"][1], "slot off by one image")


@pytest.mark.parametrize("case", list(te.EDGE))
def test_case_is_at_the_edge_of_the_envelope(case):
    """Global keys in (65 280, 65 536]; mb_check accepts the case and refuses it with one more image (one more rank)."""
    from gan_variant_research_b200 import patchnce as pmod
    b, world, shapes, p, rows = te.EDGE[case]
    assert 65280 <= te.global_keys(case) <= pmod.MB_MAX_KEYS == 65536
    chans = [c for c, _, _ in shapes]
    pmod.mb_check(b, chans, [p] * len(shapes), "tc_bf16x3", rows=rows, world=world)
    more = dict(world=world + 1) if world > 1 else dict(batch=b + 1)
    with pytest.raises(RuntimeError, match="65536"):
        pmod.mb_check(more.get("batch", b), chans, [p] * len(shapes), "tc_bf16x3", rows=rows,
                      world=more.get("world", world))


def test_e4_taus_straddle_the_single_pass_condition():
    """loss_tc.cuh: single = multi && !((1 / tau) * 1.02f > kClamp), in fp32.  E4's two taus fall on either side;
    E5's tau binds the clamp itself."""
    with open(os.path.join(ROOT, "gan_variant_research_b200", "csrc", "common.cuh")) as f:
        k_clamp = np.float32(re.search(r"constexpr float kClamp = ([0-9.]+)f;", f.read()).group(1))
    two_pass = lambda tau: (np.float32(1.0) / np.float32(tau)) * np.float32(1.02) > k_clamp
    single, double = te.E4_TAUS
    assert not two_pass(single) and two_pass(double)
    assert 1.0 / te.E5_TAU > k_clamp
