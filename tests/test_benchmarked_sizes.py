"""CPU pins of the float64 restatement and the checker of test_benchmarked_sizes_gpu.py: the restatement equals the
oracle's numpy formula sheet and its head restatement; the checker accepts the reference and rejects one (image, layer)
block of 64 scaled by 1.005 and a single non-zero entry off the sampled positions.  Also the dispatch arithmetic the GPU
cases are chosen by (the fold boundaries, the persistent loss kernel's item schedule)."""
import numpy as np
import pytest
import torch

import test_benchmarked_sizes_gpu as tb
from oracle import patchnce_oracle as orc


def _problem(seed, b, shapes, p, tiny_patch=False):
    """CPU float64 maps, correlated src / tgt, and ids drawn with replacement (P > HW in the first layer: duplicates)."""
    g = torch.Generator().manual_seed(seed)
    src = [torch.randn(b, *s, generator=g, dtype=torch.float64) for s in shapes]
    tgt = [0.6 * x + 0.8 * torch.randn(x.shape, generator=g, dtype=torch.float64) for x in src]
    ids = [torch.randint(0, h * w, (p,), generator=g) for _, h, w in shapes]
    if tiny_patch:                                       # ||q|| < 1e-6: the g / eps branch of F.normalize's backward
        tgt[0][1].view(shapes[0][0], -1)[:, ids[0][3]] *= 1e-9
    return src, tgt, ids


def _dense(ref, shapes, b, dtype=torch.float64):
    """restate's (positions, (B, C, U)) columns scattered into dense (B, C, H, W) maps."""
    out = []
    for (pos, cols), (c, h, w) in zip(ref, shapes):
        d = torch.zeros(b, c, h * w, dtype=dtype)
        d[:, :, pos] = cols.to(dtype)
        out.append(d.view(b, c, h, w))
    return out


@pytest.mark.parametrize("tau", [0.07, 0.015])          # 0.015: 1 / tau > 50, the +-50 clamp binds
def test_restatement_equals_the_numpy_oracle(tau):
    shapes = [(8, 6, 6), (16, 5, 7), (24, 9, 4)]
    src, tgt, ids = _problem(3, 3, shapes, 40, tiny_patch=True)
    assert ids[0].unique().numel() < ids[0].numel()
    loss, ref, heads = tb.restate(src, tgt, ids, tau)
    assert heads is None
    want, _, grads = orc.patchnce_loss_and_grads_np([x.numpy() for x in src], [x.numpy() for x in tgt],
                                                    [i.numpy() for i in ids], tau)
    assert loss == pytest.approx(want, rel=1e-12)
    for got, r in zip(_dense(ref, shapes, 3), grads):
        assert np.abs(got.numpy() - r).max() <= 1e-12 * np.abs(r).max()


def test_head_restatement_equals_the_head_oracle_and_its_autograd():
    shapes = [(8, 6, 6), (16, 5, 7)]
    src, tgt, ids = _problem(4, 2, shapes, 30)
    g = torch.Generator().manual_seed(9)
    heads = [[0.3 * torch.randn(*s, generator=g, dtype=torch.float64) for s in ((32, c), (32,), (32, 32), (32,))]
             for c, _, _ in shapes]
    loss, ref, hg = tb.restate(src, tgt, ids, 0.07, heads)
    t = [x.clone().requires_grad_() for x in tgt]
    hp = [[p.clone().requires_grad_() for p in h] for h in heads]
    want = orc.patchnce_head_loss_torch(src, t, ids, hp, 0.07)
    want.backward()
    assert loss == pytest.approx(want.item(), rel=1e-12)
    for got, x in zip(_dense(ref, shapes, 2), t):
        assert (got - x.grad).abs().max() <= 1e-12 * x.grad.abs().max()
    for gs, ps in zip(hg, hp):
        for a, p in zip(gs, ps):
            assert (a - p.grad).abs().max() <= 1e-12 * p.grad.abs().max()


def test_relu_flip_allowance_marks_only_rows_on_the_boundary():
    shapes = [(8, 6, 6), (16, 5, 7)]
    src, tgt, ids = _problem(6, 2, shapes, 30)
    g = torch.Generator().manual_seed(2)
    heads = [[0.3 * torch.randn(*s, generator=g, dtype=torch.float64) for s in ((32, c), (32,), (32, 32), (32,))]
             for c, _, _ in shapes]
    w1, b1 = heads[1][0], heads[1][1]
    x = tgt[1][1].reshape(16, -1)[:, ids[1][4]]                 # image 1, id 4 of layer 1: unit 3 exactly at zero
    b1[3] = -(w1[3] @ x)
    flips = tb.relu_flip_allowance(src, tgt, ids, heads, 0.07)
    assert [f[3] for f in flips] == [0, int((ids[1] == ids[1][4]).sum())]
    cols, dw1, db1, _ = flips[1]
    assert cols.shape == (2, 16, 30) and dw1.shape == (32, 16) and db1.shape == (32,)
    hit = torch.zeros(2, 30, dtype=torch.bool)
    hit[1, ids[1] == ids[1][4]] = True
    assert (cols[1, :, ids[1] == ids[1][4]] > 0).all() and (cols.amax(1)[~hit] == 0).all()
    assert (db1[torch.arange(32) != 3] == 0).all() and db1[3] > 0 and (flips[0][0] == 0).all()


SHAPES4 = [(8, 6, 6), (16, 5, 7), (24, 9, 4), (8, 4, 4)]      # 16 images x 4 layers: 64 (image, layer) blocks


def _checker_case():
    src, tgt, ids = _problem(5, 16, SHAPES4, 24)
    tgt[2][7] *= 30.0                                     # image 7 of layer 2: gradients ~30x smaller than its neighbours'
    _, ref, _ = tb.restate(src, tgt, ids, 0.07)
    return ref, ids, _dense(ref, SHAPES4, 16, torch.float32)


def test_checker_accepts_the_reference():
    ref, ids, grads = _checker_case()
    assert tb.check_grads(grads, ref, ids, 5e-4, "reference") <= 1e-6      # float32 rounding only


def test_checker_rejects_one_block_of_64_scaled_by_1_005():
    ref, ids, grads = _checker_case()
    grads[2][7] *= 1.005
    # a single max-norm over the layer would let it through ...
    pos, want = ref[2]
    got = grads[2].view(16, 24, -1)[:, :, pos].double()
    assert (got - want).abs().max() / want.abs().max() < 5e-4
    # ... one block at a time does not
    with pytest.raises(AssertionError, match="layer 2 image 7"):
        tb.check_grads(grads, ref, ids, 5e-4, "scaled block")


def test_checker_rejects_a_single_non_zero_entry_off_the_samples():
    ref, ids, grads = _checker_case()
    l = 3
    off = [q for q in range(16) if q not in set(ids[l].tolist())]
    assert off
    grads[l].view(16, 8, -1)[11, 5, off[0]] = 1e-30
    with pytest.raises(AssertionError, match="1 non-zero entries off the sampled positions"):
        tb.check_grads(grads, ref, ids, 5e-4, "off-sample entry")


def test_checker_rejects_a_nan_the_reference_does_not_have():
    ref, ids, grads = _checker_case()
    grads[0].view(16, 8, -1)[4, 2, ids[0][0]] = float("nan")
    with pytest.raises(AssertionError, match="NaN pattern"):
        tb.check_grads(grads, ref, ids, 5e-4, "nan")


def _dump(tmp_path, ref, ids, shapes, b, grads, name):
    """bench.dump_outputs on CPU maps whose gradients are ``grads``, read back like the GPU test reads bench.py's."""
    import bench
    tgt = [torch.zeros(b, *s) for s in shapes]
    for t, g in zip(tgt, grads):
        t.grad = g
    bench.dump_outputs(str(tmp_path / name), torch.tensor(1.0), tgt, ids)
    return {f.stem: np.load(f) for f in (tmp_path / name).iterdir()}


def test_dump_checker_accepts_the_reference_and_rejects_a_write_off_the_samples(tmp_path):
    ref, ids, grads = _checker_case()
    d = _dump(tmp_path, ref, ids, SHAPES4, 16, grads, "ref")
    assert "images_sampled" not in d
    worst, flat, _ = tb.check_dump(d, SHAPES4, ids, ref, torch.float32, 5e-4, "reference")
    assert worst <= 1e-6 and flat <= 1e-6
    bad = [g.clone() for g in grads]
    bad[1][bad[1] == 0] = 1e-30                             # every entry off the samples (the flat sample sees them)
    d = _dump(tmp_path, ref, ids, SHAPES4, 16, bad, "off")
    with pytest.raises(AssertionError, match="grad_l1_flat: .* non-zero entries off the sampled positions"):
        tb.check_dump(d, SHAPES4, ids, ref, torch.float32, 5e-4, "off")
    bad = [g.clone() for g in grads]
    bad[2][7] *= 1.005
    d = _dump(tmp_path, ref, ids, SHAPES4, 16, bad, "scaled")
    with pytest.raises(AssertionError, match="grad_l2 image 7"):
        tb.check_dump(d, SHAPES4, ids, ref, torch.float32, 5e-4, "scaled")


def test_half_dtype_rounding_allowance_is_one_ulp_subnormals_included():
    x = torch.tensor([1.0, 3.0, 1e-6, 0.0], dtype=torch.float64)
    assert tb._ulp(x, torch.float16).tolist() == [2.0 ** -10, 2.0 ** -9, 2.0 ** -24, 2.0 ** -24]
    assert tb._ulp(x, torch.bfloat16)[:3].tolist() == [2.0 ** -7, 2.0 ** -6, 2.0 ** -27]
    assert (tb._ulp(x, torch.float32) == 0).all()


def test_fold_boundaries_at_bench_size():
    """b5 at P = 256 gathers with the id prep folded in up to B = 10 on NCHW maps and up to B = 5 on channels-last maps;
    the fp32 maps stay below the side-stream id draw there and pass it at B = 64."""
    from gan_variant_research_b200 import patchnce as pmod
    assert tb.gather_tc_ctas(tb.B5, 256, 10) <= tb.FOLD_MAX_CTAS < tb.gather_tc_ctas(tb.B5, 256, 11)
    assert tb.gather_nhwc_ctas(tb.B5, 256, 5) <= tb.FOLD_MAX_CTAS < tb.gather_nhwc_ctas(tb.B5, 256, 6)
    assert tb.map_bytes(tb.B5, 11, 4) < pmod._SIDE_STREAM_MIN_BYTES <= tb.map_bytes(tb.B5, 64, 2)


def test_loss_schedule_of_the_gpu_cases_on_148_sms():
    sm = 148
    assert tb.loss_schedule(sm, [(c, 256) for c, _, _ in tb.B5], 64) == (640, 148, 256, 48)    # bench.py's step
    for items, kind in tb.SCHEDULE:
        target = {"S-2": sm - 2, "S": sm, "S+2": sm + 2, "4.3S": 4.3 * sm}[items]
        b, layers, (n, grid, light, rot) = tb.schedule_case(sm, target, kind)
        assert len(layers) <= 8 and all(p <= 256 for *_, p in layers)
        assert n == b * sum((p + 127) // 128 for *_, p in layers) and grid == min(sm, n)
        assert n == target if isinstance(target, int) else abs(n - target) <= 0.05 * target
        assert (len({c for c, *_ in layers}) == 1) == (kind == "single")
        if kind == "below":
            assert 0 < light < grid // 3 and rot == light & ~1
        elif kind == "above":
            assert light >= grid // 3 and rot == grid // 3 & ~1
        else:
            assert rot == 0 and light == n
    assert tb.schedule_case(sm, sm - 2, "below") is None           # 146 = 2 * 73: two items per image at most
