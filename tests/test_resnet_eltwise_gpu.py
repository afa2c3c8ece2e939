"""Kernel-level parity of the ResNet encoder's BatchNorm, residual, dropout and head entry points (csrc/resnet.cu) through the
C ABI, each against a float64 reference computed on the host from the exact tensors the kernel read (fp16 activations, bf16
gradients, fp32 coefficients): what may differ is the rounding of the stored output and fp32 accumulation, so the bounds
are a few output ulps, or 1e-5 of the sum of the absolute terms where a sum cancels.  Plus the convolution fall-backs:
MMNN_RN_MMA=0 and MMNN_RN_WGRAD16=0 are read once per process, so each runs the per-kernel and whole-network tests in a
subprocess of its own.

Element counts (n8 = elements / 8, one thread's 16-byte vector): a partial first warp, a ragged last block, and more than
the 148 * 8 blocks of 256 threads that elt_grid caps the grid at, so that every thread walks the grid-stride loop ~10 times."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHANNELS = (8, 16, 64)
N8 = {"tiny": 24, "ragged": 9608, "large": 400003 * 8}
EPS = 1e-5


def _lib():
    from mmnn_sts_b200 import _lib as L
    return L.lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _ulp(x, mant):
    """Spacing of a float with `mant` stored mantissa bits at |x| (fp16: 10, fp32: 23), floored at the smallest subnormal."""
    lo = {10: 2.0 ** -24, 23: 2.0 ** -149}[mant]
    return torch.exp2(torch.floor(torch.log2(x.abs())) - mant).clamp_min(lo)


def _assert_within(got, ref, tol, what):
    err = (got.double().cpu() - ref).abs()
    bad = err > tol
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())} of {bad.numel()} beyond the bound, worst excess "
                                 f"{float((err - tol).max()):.3e}, max |ref| {float(ref.abs().max()):.3e}")


def _rows(size, C):
    return N8[size] * 8 // C


def _coef(g, C, mean=None, rstd=None):
    """[4][C] fp32 table scale, shift, mean, rstd (mmnn_rn_bn_coeffs layout)."""
    sc = (torch.rand(C, generator=g) + 0.5) * torch.where(torch.rand(C, generator=g) < 0.2, -1.0, 1.0)
    sh = torch.randn(C, generator=g) * 0.5
    mean = torch.randn(C, generator=g) if mean is None else mean
    rstd = torch.rand(C, generator=g) + 0.5 if rstd is None else rstd
    return torch.stack([sc, sh, mean, rstd]).float()


def _randh(g, rows, C, spread=2.0):
    """Random fp16 [rows][C] with a per-channel offset and scale."""
    mu = torch.randn(C, generator=g) * spread
    sd = torch.rand(C, generator=g) * 2 + 0.25
    return (torch.randn((rows, C), generator=g) * sd + mu).half()


# ------------------------------------------------------------------------------------------------ mmnn_rn_bn_coeffs
def _bn_coeffs_call(stats, count, gamma, beta, rmean, rvar, nbt, momentum, training, C, coef):
    return _lib().mmnn_rn_bn_coeffs(stats.data_ptr(), float(count), gamma.data_ptr(), beta.data_ptr(), rmean.data_ptr(),
                                    rvar.data_ptr(), nbt.data_ptr(), EPS, momentum, training, C, coef.data_ptr(), _st())


@pytest.mark.parametrize("training", [1, 0])
@pytest.mark.parametrize("C", CHANNELS)
def test_bn_coeffs_vs_float64(C, training):
    """coef against float64 at 2 fp32 ulps; the running update against torch's law (momentum, unbiased variance) at 1 fp32 ulp
    of the result, which is the kernel's single rounding of a float64 value.  At 10^6 values the unbiased factor moves the
    running variance by ~7e-7 relative (the old running variance is small next to the batch one), i.e. several ulps, so
    the biased variance is told apart at every count."""
    dev = torch.device("cuda", 0)
    gd = torch.Generator(device=dev).manual_seed(40 + C)
    g = torch.Generator().manual_seed(41 + C)
    e32, n_checked = float(np.float32(EPS)), 0
    for count in (24, 4096, 10 ** 6):
        mu = torch.randn(C, generator=g) * 3
        sd = torch.rand(C, generator=g) * 2 + 0.1
        x = (torch.randn((count, C), generator=gd, device=dev) * sd.to(dev) + mu.to(dev)).half()
        xd = x.double()
        stats = torch.cat([xd.sum(0), (xd * xd).sum(0)]).contiguous()
        del xd
        s = stats.cpu()
        for momentum in (0.1, 0.3):
            gamma = (torch.rand(C, generator=g) + 0.5).float()
            beta = torch.randn(C, generator=g).float()
            rmean0 = torch.randn(C, generator=g).float()
            rvar0 = (sd * sd * (0.02 + 0.06 * torch.rand(C, generator=g))).float()
            rmean, rvar = rmean0.to(dev), rvar0.to(dev)
            nbt = torch.tensor([7], dtype=torch.int64, device=dev)
            coef = torch.full((4, C), float("nan"), device=dev)
            assert _bn_coeffs_call(stats, count, gamma.to(dev), beta.to(dev), rmean, rvar, nbt, momentum, training, C, coef) == 0
            m, n = float(np.float32(momentum)), float(count)
            if training:
                mean = s[:C] / n
                var = (s[C:] / n - mean * mean).clamp_min(0.0)
                rm_ref = (1.0 - m) * rmean0.double() + m * mean
                rv_ref = (1.0 - m) * rvar0.double() + m * (var * n / (n - 1.0))
                if count <= 4096:
                    # the update law above is torch's own: F.batch_norm updates float64 buffers the same way
                    tm, tv = rmean0.double(), rvar0.double()
                    F.batch_norm(x.double().cpu(), tm, tv, None, None, True, m, e32)
                    torch.testing.assert_close(rm_ref, tm, rtol=1e-9, atol=1e-12)
                    torch.testing.assert_close(rv_ref, tv, rtol=1e-9, atol=1e-12)
            else:
                mean, var = rmean0.double(), rvar0.double()
                rm_ref, rv_ref = mean, var
            rstd = 1.0 / torch.sqrt(var + e32)
            scale = gamma.double() * rstd
            shift = beta.double() - mean * scale
            cf = coef.cpu()
            _assert_within(cf[0], scale, 2 * _ulp(scale, 23), f"scale C={C} n={count}")
            # shift = beta - mean * scale from the rounded mean and scale: 2 ulps of the result and of the product it cancels against
            _assert_within(cf[1], shift, 2 * (_ulp(shift, 23) + 2 * _ulp(mean * scale, 23)), f"shift C={C} n={count}")
            _assert_within(cf[2], mean, 2 * _ulp(mean, 23), f"mean C={C} n={count}")
            _assert_within(cf[3], rstd, 2 * _ulp(rstd, 23), f"rstd C={C} n={count}")
            if training:
                _assert_within(rmean, rm_ref, _ulp(rm_ref, 23), f"running_mean C={C} n={count} momentum={momentum}")
                _assert_within(rvar, rv_ref, _ulp(rv_ref, 23), f"running_var C={C} n={count} momentum={momentum}")
                assert int(nbt.item()) == 8
            else:
                assert torch.equal(rmean.cpu(), rmean0) and torch.equal(rvar.cpu(), rvar0)
                assert int(nbt.item()) == 7
            n_checked += 1
    assert n_checked == 6


def test_bn_coeffs_rejects_unsupported_channel_counts():
    """C outside 1..64 returns -2 and writes nothing: no coefficients, no running statistics, no num_batches_tracked.
    The buffers are sized for 65 channels, so the call cannot read or write outside them whatever it does."""
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(5)
    Cmax = 65
    stats = torch.cat([torch.randn(Cmax, generator=g, dtype=torch.float64) * 100,
                       torch.rand(Cmax, generator=g, dtype=torch.float64) * 1000 + 1000]).to(dev)
    gamma, beta = torch.rand(Cmax, generator=g).to(dev), torch.randn(Cmax, generator=g).to(dev)
    for C in (65, 0):
        rmean, rvar = torch.randn(Cmax, generator=g).to(dev), torch.rand(Cmax, generator=g).to(dev) + 0.5
        nbt = torch.tensor([3], dtype=torch.int64, device=dev)
        coef = torch.full((4, Cmax), 1234.5, device=dev)
        before = [t.clone() for t in (rmean, rvar, nbt, coef)]
        assert _bn_coeffs_call(stats, 100.0, gamma, beta, rmean, rvar, nbt, 0.1, 1, C, coef) == -2, C
        torch.cuda.synchronize()
        for name, t, t0 in zip(("running_mean", "running_var", "num_batches_tracked", "coef"), (rmean, rvar, nbt, coef), before):
            assert torch.equal(t, t0), f"C={C}: {name} was written by a rejected call"


# ------------------------------------------------------------------------------------------------ mmnn_rn_bn_act
def _act_ref(raw, coef, res_mode, res, coef2, relu):
    """float64 o = [relu](raw * scale + shift [+ res | + res * scale2 + shift2]) and the sum of |terms| (for the fp32
    rounding slack where the terms cancel)."""
    r = raw.double()
    a = r * coef[0].double()
    o, terms = a + coef[1].double(), a.abs() + coef[1].double().abs()
    if res_mode == 1:
        o, terms = o + res.double(), terms + res.double().abs()
    if res_mode == 2:
        a2 = res.double() * coef2[0].double()
        o, terms = o + a2 + coef2[1].double(), terms + a2.abs() + coef2[1].double().abs()
    return (o.clamp_min(0.0) if relu else o), terms


def _act_call(raw, coef, res_mode, res, coef2, y, C, relu, drop_p, seed, mask):
    p = lambda t: t.data_ptr() if t is not None else None
    return _lib().mmnn_rn_bn_act(p(raw), p(coef), res_mode, p(res), p(coef2), p(y), raw.numel(), C, relu, drop_p, seed, p(mask),
                                 _st())


def _check_f16(y, ref, terms, what):
    # one fp16 rounding of an fp32 fmaf result: 1 fp16 ulp, plus fp32 slack where the terms cancel
    _assert_within(y, ref, _ulp(ref, 10) + 2.0 ** -22 * terms, what)


@pytest.mark.parametrize("size", list(N8))
@pytest.mark.parametrize("C", CHANNELS)
def test_bn_act_vs_float64(C, size):
    """res_mode 0 / 1 / 2 with and without ReLU; an injected uint8 dropout mask with drop_p = p (kept values scaled by
    1 / (1 - p), dropped ones exactly 0) and with drop_p = 0 (scale 1)."""
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(7 * C + len(size))
    rows = _rows(size, C)
    raw, res, raw2 = _randh(g, rows, C), _randh(g, rows, C), _randh(g, rows, C)
    coef, coef2 = _coef(g, C), _coef(g, C)
    raw_d, res_d, raw2_d, coef_d, coef2_d = (t.to(dev) for t in (raw, res, raw2, coef, coef2))
    y = torch.empty_like(raw_d)
    for res_mode in (0, 1, 2):
        other, other_d = (res, res_d) if res_mode == 1 else (raw2, raw2_d)
        for relu in (0, 1):
            y.fill_(float("nan"))
            assert _act_call(raw_d, coef_d, res_mode, other_d if res_mode else None, coef2_d if res_mode == 2 else None, y, C,
                             relu, 0.0, 0, None) == 0
            ref, terms = _act_ref(raw, coef, res_mode, other, coef2, relu)
            _check_f16(y, ref, terms, f"bn_act C={C} {size} res_mode={res_mode} relu={relu}")
    # injected masks on the down-sample form (the last block of every stage carries the dropout)
    keep = torch.rand((rows, C), generator=g) >= 0.25
    mask_d = keep.to(torch.uint8).to(dev)
    ref, terms = _act_ref(raw, coef, 2, raw2, coef2, 1)
    for p in (0.2, 0.0):
        s = 1.0 / (1.0 - float(np.float32(p)))
        y.fill_(float("nan"))
        assert _act_call(raw_d, coef_d, 2, raw2_d, coef2_d, y, C, 1, p, 99, mask_d) == 0
        yc = y.cpu()
        assert bool((yc[~keep] == 0).all()), f"dropped elements not zero (p={p})"
        _check_f16(yc[keep], ref[keep] * s, terms[keep] * s, f"bn_act C={C} {size} injected mask p={p}")


def _hash_keep(seed, n, p):
    """Host replay of csrc/resnet.cu hash_uniform (splitmix64 finaliser of seed + e * golden ratio, top 24 bits as a float in
    [0, 1)) for e = 0 .. n-1: the keep mask u >= p in float32, bit for bit."""
    e = np.arange(n, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + e * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
    u = (z >> np.uint64(40)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return torch.from_numpy(u >= np.float32(p))


@pytest.mark.parametrize("size", list(N8))
@pytest.mark.parametrize("C", CHANNELS)
def test_bn_act_hashed_dropout_keep_mask_exact(C, size):
    """The hashed dropout's keep pattern equals the host replay of hash_uniform bit for bit (element index = flat index into
    the channels-last tensor), for two seeds (one with high bits set), and the kept values are the undropped ones / (1 - p)."""
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(11 * C + len(size))
    rows = _rows(size, C)
    raw, res = _randh(g, rows, C), _randh(g, rows, C)
    coef = _coef(g, C)
    raw_d, res_d, coef_d = raw.to(dev), res.to(dev), coef.to(dev)
    y0 = torch.empty_like(raw_d)
    assert _act_call(raw_d, coef_d, 1, res_d, None, y0, C, 0, 0.0, 0, None) == 0
    ref, terms = _act_ref(raw, coef, 1, res, None, 0)
    ref, terms = ref.flatten(), terms.flatten()
    nz = y0.cpu().flatten() != 0                     # where the undropped value is nonzero the pattern is visible
    assert float(nz.double().mean()) > 0.99
    p = 0.2
    s = 1.0 / (1.0 - float(np.float32(p)))
    y = torch.empty_like(raw_d)
    for seed in (12345, 0x7A3F12345678ABCD):
        assert _act_call(raw_d, coef_d, 1, res_d, None, y, C, 0, p, seed, None) == 0
        yc = y.cpu().flatten()
        keep = _hash_keep(seed, rows * C, p)
        assert torch.equal((yc != 0)[nz], keep[nz]), f"seed {seed}: {int(((yc != 0) != keep)[nz].sum())} keep decisions differ"
        assert bool((yc[~keep] == 0).all())
        _check_f16(yc[keep], ref[keep] * s, terms[keep] * s, f"hashed dropout C={C} {size} seed={seed}")


# ------------------------------------------------------------------------------------------------ BatchNorm backward
# (TWO = down-sample branch present, eval_mode, post_scale, dz output): every value of every flag, and TWO x eval_mode in full
BWD_CASES = [(False, 0, 1.0, False), (True, 0, 1.25, True), (False, 1, 1.25, True), (True, 1, 1.0, False)]


@pytest.mark.parametrize("size", list(N8))
@pytest.mark.parametrize("C", CHANNELS)
def test_bn_backward_vs_float64(C, size):
    """mmnn_rn_act_bwd_reduce + mmnn_rn_bn_bwd_apply against (a) the kernels' formula in float64 (sums, dgamma / dbeta as the
    fp32 rounding of the sums, draw / draw2, dz) and (b) torch autograd in float64 through
    post_scale * [y > 0] * (F.batch_norm(raw) [+ F.batch_norm(raw2)]) with batch statistics (eval_mode 0) or the running
    ones (eval_mode 1): (b) shows the two passes compute BatchNorm's backward, not only their own algebra.  The ReLU mask is
    taken from the stored fp16 y in both, so rounding flips of y cannot enter."""
    dev = torch.device("cuda", 0)
    lib = _lib()
    g = torch.Generator().manual_seed(13 * C + len(size))
    rows = _rows(size, C)
    raw, raw2 = _randh(g, rows, C), _randh(g, rows, C)
    dy = (torch.randn((rows, C), generator=g) * 0.5).bfloat16()
    raw_d, raw2_d, dy_d = raw.to(dev), raw2.to(dev), dy.to(dev)
    r64, r264, dy64 = raw.double(), raw2.double(), dy.double()
    e32 = float(np.float32(EPS))
    bn = {}                                          # per branch: gamma, beta, running mean / var (fp32)
    for b, r in (("1", r64), ("2", r264)):
        bn[b] = dict(gamma=(torch.rand(C, generator=g) + 0.5).float(), beta=torch.randn(C, generator=g).float(),
                     rmean=(r.mean(0) + 0.3 * torch.randn(C, generator=g, dtype=torch.float64)).float(),
                     rvar=(r.var(0) * (0.5 + torch.rand(C, generator=g, dtype=torch.float64))).float())
    for two, eval_mode, post, want_dz in BWD_CASES:
        what = f"C={C} {size} two={two} eval={eval_mode} post={post} dz={want_dz}"
        coefs, xh, shift, z = {}, {}, {}, 0.0
        for b, r in (("1", r64), ("2", r264)) if two else (("1", r64),):
            q = bn[b]
            if eval_mode:
                mean, var = q["rmean"].double(), q["rvar"].double()
            else:
                mean, var = r.mean(0), r.var(0, unbiased=False)
            rstd = 1.0 / torch.sqrt(var + e32)
            sc = q["gamma"].double() * rstd
            coefs[b] = torch.stack([sc, q["beta"].double() - mean * sc, mean, rstd]).float()
            cf = coefs[b].double()
            xh[b] = (r - cf[2]) * cf[3]               # x-hat from the stored fp32 table, as the kernels form it
            shift[b] = (mean - cf[2]).abs() * cf[3]   # how far the fp32 mean moves x-hat off the exact one
            z = z + cf[0] * r + cf[1]
        y = (post * z).clamp_min(0.0).half()           # the forward pass's stored output: only its sign is read
        mask = (y > 0).double()
        dz = dy64 * float(np.float32(post)) * mask
        c1, c2 = coefs["1"].to(dev), coefs["2"].to(dev) if two else None
        y_d = y.to(dev)
        sums = torch.zeros(3 * C, dtype=torch.float64, device=dev)
        assert lib.mmnn_rn_act_bwd_reduce(dy_d.data_ptr(), y_d.data_ptr(), post, raw_d.data_ptr(), c1.data_ptr(),
                                          raw2_d.data_ptr() if two else None, c2.data_ptr() if two else None, sums.data_ptr(),
                                          rows * C, C, _st()) == 0
        draw = torch.full_like(dy_d, float("nan"))
        draw2 = torch.full_like(dy_d, float("nan")) if two else None
        dzo = torch.full_like(dy_d, float("nan")) if want_dz else None
        outs = [torch.full((C,), float("nan"), device=dev) for _ in range(4 if two else 2)]
        p = lambda t: t.data_ptr() if t is not None else None
        assert lib.mmnn_rn_bn_bwd_apply(dy_d.data_ptr(), y_d.data_ptr(), post, raw_d.data_ptr(), c1.data_ptr(), p(raw2_d if two else None),
                                        p(c2), sums.data_ptr(), 1.0 / rows, eval_mode, draw.data_ptr(), p(draw2), p(dzo),
                                        outs[0].data_ptr(), outs[1].data_ptr(), p(outs[2] if two else None),
                                        p(outs[3] if two else None), rows * C, C, _st()) == 0
        sk = sums.cpu()
        dgamma, dbeta = outs[0].cpu(), outs[1].cpu()
        # (a) the kernels' formula
        s_ref = [dz.sum(0), (dz * xh["1"]).sum(0)] + ([(dz * xh["2"]).sum(0)] if two else [])
        s_abs = [dz.abs().sum(0), (dz * xh["1"]).abs().sum(0)] + ([(dz * xh["2"]).abs().sum(0)] if two else [])
        for i, (sr, sa) in enumerate(zip(s_ref, s_abs)):
            _assert_within(sk[i * C:(i + 1) * C], sr, 1e-5 * sa, f"sums[{i}] {what}")
        assert torch.equal(dbeta, sk[:C].float()) and torch.equal(dgamma, sk[C:2 * C].float()), what
        if two:
            dgamma2, dbeta2 = outs[2].cpu(), outs[3].cpu()
            assert torch.equal(dbeta2, sk[:C].float()) and torch.equal(dgamma2, sk[2 * C:].float()), what
        if want_dz:
            assert torch.equal(dzo.cpu(), (dy.float() * post * (y > 0).float()).bfloat16()), what
        m1 = torch.zeros(C, dtype=torch.float64) if eval_mode else s_ref[0] / rows
        bounds = {}
        for b, got in (("1", draw), ("2", draw2)) if two else (("1", draw),):
            sc = coefs[b][0].double()
            m2 = torch.zeros(C, dtype=torch.float64) if eval_mode else s_ref[1 if b == "1" else 2] / rows
            ref = sc * (dz - m1 - xh[b] * m2)
            bounds[b] = 2.0 ** -8 * ref.abs() + 1e-5 * sc.abs() * (dz.abs() + m1.abs() + (xh[b] * m2).abs())
            _assert_within(got, ref, bounds[b], f"draw{b} (kernel formula) {what}")
            # against the exact statistics, x-hat is off by shift[b]: draw by sc * shift * (m2 + x-hat * m1) to first order
            bounds[b] = bounds[b] + 2 * sc.abs() * shift[b] * (m2.abs() + (xh[b] * m1).abs())
        # (b) autograd through F.batch_norm
        leaves, zb = {}, 0.0
        for b, r in (("1", r64), ("2", r264)) if two else (("1", r64),):
            q = bn[b]
            xa = r.clone().requires_grad_(True)
            ga, ba = q["gamma"].double().requires_grad_(True), q["beta"].double().requires_grad_(True)
            rm, rv = (q["rmean"].double(), q["rvar"].double()) if eval_mode else (None, None)
            zb = zb + F.batch_norm(xa, rm, rv, ga, ba, not eval_mode, 0.0, e32)
            leaves[b] = (xa, ga, ba)
        (post * zb * mask * dy64).sum().backward()
        for b, got_raw in (("1", draw), ("2", draw2)) if two else (("1", draw),):
            xa, ga, ba = leaves[b]
            _assert_within(got_raw, xa.grad, 2.0 ** -8 * xa.grad.abs() + bounds[b], f"draw{b} (autograd) {what}")
            dg, db_ = (dgamma, dbeta) if b == "1" else (outs[2].cpu(), outs[3].cpu())
            ga_abs = (dz * xh[b]).abs().sum(0)
            _assert_within(dg, ga.grad, 1e-5 * ga_abs + shift[b] * s_abs[0] + _ulp(ga.grad, 23), f"dgamma{b} (autograd) {what}")
            _assert_within(db_, ba.grad, 1e-5 * s_abs[0] + _ulp(ba.grad, 23), f"dbeta{b} (autograd) {what}")


# ------------------------------------------------------------------------------------------------ head
@pytest.mark.parametrize("C", CHANNELS)
def test_head_vs_float64(C):
    """mmnn_rn_head_fwd (mean over V -> Linear -> sigmoid) and mmnn_rn_head_bwd at B in {1, 7}, V in {1, 8, 5000}, K in
    {1, 5, 64}.  The backward reads the forward's stored fp32 `out` / `pooled`, which the reference takes as they are; dW / db
    start nonzero and must be added to."""
    dev = torch.device("cuda", 0)
    lib = _lib()
    g = torch.Generator().manual_seed(17 * C)
    for B in (1, 7):
        for V in (1, 8, 5000):
            for K in (1, 5, 64):
                what = f"C={C} B={B} V={V} K={K}"
                y = torch.randn((B, V, C), generator=g).clamp_min(0.0).half()       # a ReLU output
                W = torch.randn((K, C), generator=g) * 0.5
                bias = torch.randn(K, generator=g) * 0.2
                y_d, W_d, b_d = y.to(dev), W.to(dev), bias.to(dev)
                pooled = torch.full((B, C), float("nan"), device=dev)
                out = torch.full((B, K), float("nan"), device=dev)
                assert lib.mmnn_rn_head_fwd(y_d.data_ptr(), B, V, C, W_d.data_ptr(), b_d.data_ptr(), K, pooled.data_ptr(),
                                            out.data_ptr(), _st()) == 0
                y64, W64 = y.double(), W.double()
                p_ref = y64.mean(1)
                _assert_within(pooled, p_ref, 1e-5 * y64.abs().sum(1) / V, f"pooled {what}")
                z = p_ref @ W64.T + bias.double()
                z_abs = p_ref.abs() @ W64.abs().T + bias.double().abs()
                _assert_within(out, torch.sigmoid(z), 1e-5 * z_abs + 2.0 ** -21, f"out {what}")
                # backward
                dout = torch.randn((B, K), generator=g)
                dW0, db0 = torch.randn((K, C), generator=g), torch.randn(K, generator=g)
                dW, db = dW0.to(dev), db0.to(dev)
                dy = torch.full((B, V, C), float("nan"), dtype=torch.bfloat16, device=dev)
                assert lib.mmnn_rn_head_bwd(dout.to(dev).data_ptr(), out.data_ptr(), pooled.data_ptr(), W_d.data_ptr(), B, V, C, K,
                                            dy.data_ptr(), dW.data_ptr(), db.data_ptr(), _st()) == 0
                o, pk = out.double().cpu(), pooled.double().cpu()
                dl = dout.double() * o * (1.0 - o)
                dW_ref, dW_abs = dW0.double() + dl.T @ pk, dW0.double().abs() + dl.abs().T @ pk.abs()
                _assert_within(dW, dW_ref, 1e-5 * dW_abs + _ulp(dW_ref, 23), f"dW += {what}")
                db_ref, db_abs = db0.double() + dl.sum(0), db0.double().abs() + dl.abs().sum(0)
                _assert_within(db, db_ref, 1e-5 * db_abs + _ulp(db_ref, 23), f"db += {what}")
                dp = (dl @ W64 / V)[:, None, :].expand(B, V, C)
                dp_abs = (dl.abs() @ W64.abs() / V)[:, None, :].expand(B, V, C)
                _assert_within(dy, dp, 2.0 ** -8 * dp.abs() + 1e-5 * dp_abs, f"dy {what}")


def test_head_rejects_unsupported_shapes():
    """C must divide 128 and be <= 64, K <= 64: each violation returns -2 from both passes and writes nothing.  Buffers are
    sized for the largest request, so the calls cannot leave them whatever they do."""
    dev = torch.device("cuda", 0)
    lib = _lib()
    B, V, Cm, Km = 2, 3, 128, 65
    y = torch.ones((B, V, Cm), dtype=torch.float16, device=dev)
    W, bias = torch.ones((Km, Cm), device=dev), torch.ones(Km, device=dev)
    for C, K in ((24, 5), (128, 5), (16, 65)):
        pooled = torch.full((B, Cm), 7.0, device=dev)
        out = torch.full((B, Km), 7.0, device=dev)
        dy = torch.full((B, V, Cm), 7.0, dtype=torch.bfloat16, device=dev)
        dW, db = torch.full((Km, Cm), 7.0, device=dev), torch.full((Km,), 7.0, device=dev)
        assert lib.mmnn_rn_head_fwd(y.data_ptr(), B, V, C, W.data_ptr(), bias.data_ptr(), K, pooled.data_ptr(), out.data_ptr(),
                                    _st()) == -2, (C, K)
        assert lib.mmnn_rn_head_bwd(out.data_ptr(), out.data_ptr(), pooled.data_ptr(), W.data_ptr(), B, V, C, K, dy.data_ptr(),
                                    dW.data_ptr(), db.data_ptr(), _st()) == -2, (C, K)
        torch.cuda.synchronize()
        for t in (pooled, out, dy, dW, db):
            assert bool((t == 7.0).all()), (C, K)


# ------------------------------------------------------------------------------------------------ convolution fall-backs
# test_resnet_gpu.py: every conv geometry, the fused layer1.0 pair (its -9 contract under MMNN_RN_MMA=0), eval forward and
# backward, and the two whole-network training steps; plus this file's kernel tests
_RESNET_SELECTION = ("test_conv_kernels_match_torch", "test_fused_downsample_pair", "test_eval_", "test_train_step_matches",
                     "test_train_step_larger_volume")
_KERNEL_SELECTION = ("test_bn_coeffs", "test_bn_act", "test_bn_backward", "test_head_")


def _expected_count():
    from tests.test_resnet_gpu import GEOMS
    resnet = len(GEOMS) + 1 + 2 + 1 + 1
    kernels = 2 * len(CHANNELS) + 1 + 3 * len(CHANNELS) * len(N8) + len(CHANNELS) + 1
    return resnet + kernels


def _run_with(var):
    env = dict(os.environ)
    env[var] = "0"
    # the same interpreter with the same isolation flags (e.g. -s: no user site-packages) as this process
    flags = [f for f, on in (("-I", sys.flags.isolated), ("-E", sys.flags.ignore_environment), ("-s", sys.flags.no_user_site)) if on]
    cmd = [sys.executable] + flags + ["-m", "pytest", "-q", "-p", "no:cacheprovider", "tests/test_resnet_gpu.py",
                                      os.path.relpath(__file__, ROOT), "-k", " or ".join(_RESNET_SELECTION + _KERNEL_SELECTION)]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    tail = r.stdout[-3000:] + r.stderr[-2000:]
    assert r.returncode == 0, f"{var}=0: pytest exited {r.returncode}\n{tail}"
    summary = r.stdout.strip().splitlines()[-1]
    passed = re.search(r"(\d+) passed", summary)
    assert passed is not None and int(passed.group(1)) == _expected_count(), f"{var}=0: {summary}"
    assert not re.search(r"skipped|failed|error|xfail|xpass", summary), f"{var}=0: {summary}"
    print(f"[{var}=0] {summary}")


def test_fallback_fma_convolutions():
    """MMNN_RN_MMA=0: every convolution on the FMA-pipe kernels (rn_conv_kernel / rn_wgrad_kernel); the model then takes
    its fall-back branches in layer1.0 (separate forward convolutions, two-launch data gradient with the second in place)."""
    _run_with("MMNN_RN_MMA")


def test_fallback_bf16_weight_gradient():
    """MMNN_RN_WGRAD16=0: the weight gradients on rn_wgrad_mma_kernel (bf16 operands) instead of the fp16 double buffer."""
    _run_with("MMNN_RN_WGRAD16")
