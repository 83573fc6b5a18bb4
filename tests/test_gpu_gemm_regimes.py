"""The tcgen05 GEMMs of csrc/gemm_tc.cu against float64 in every tiling regime they run in.

X * W (k_xw_tc, k_xw_bf16) puts 256-row tiles on min(tiles, SMs) CTAs: one tile per CTA, or several per CTA (a CTA
then reuses one TMEM accumulator, flipping its phase per tile), or, on the feature path only, split-K with the partials
added in order by k_xw_splitk_reduce.  dW (k_dw_tc, k_dw_bf16) is one wave of (256-column tile x node split) CTAs, or
several waves of one split when K > 256 * SMs.  dX (k_dx_tc) is persistent over 128 x 256 tiles with two TMEM
accumulators used in turn; accumulator 0 comes back on its second phase only when a CTA runs a third tile.  Every case
restates the planner for the device's SM count (xw_plan, dw_plan, dx_plan) and asserts the regime its id names, so a
planner change reports the coverage it loses instead of silently covering less.

Inputs are chosen so that an error cannot hide: bag-of-words counts (TF32-exact) and dense signed tanh features (not),
non-zeros of full weight in the last row, the last column and the whole last 32-column block, a dW gradient with
one-signed columns (where a biased rounding of the lo split accumulates), NaN canaries around every output, and a second
call that must be bit-identical.  References are float64 matmuls on the device (not through this library).
Bars: X * W 2e-6 of max|ref| on bag-of-words and 1e-5 on dense rows of up to 768 terms; dX 1e-5; dW max(1e-5, 2 x
the error of the fp32 control on the same inputs) up to 768 node rows per split; plain tf32 2e-3.  Longer sums in one
TMEM accumulator scale the 1e-5 by terms / 768 (the reason is beside each bar)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from bigcn_b200.data import Batch, make_batch, make_batch_shard
from test_gpu_input_grad import fixed_oracle, masks_for, with_x

pytestmark = pytest.mark.gpu

MODES = ("fp32", "tf32", "tf32x2", "tf32x3", "bf16")    # fp32 (the exact FFMA scan) is the control
NAN = float("nan")


def cdiv(a, b):
    return -(-a // b)


# ---------------------------------------------------------------------------------------------- the planners, restated
def xw_plan(n, k, sms, partial=False):
    """xw_tc_weights / xw_bf16 + xw_split_k: 256-row tiles on min(tiles, SMs) CTAs, K blocks of 32.  Split-K only with
    a partial buffer (bigcn_features_forward), when tiles * 4 <= SMs and there are at least 6 K blocks."""
    tiles, kb = cdiv(n, 256), cdiv(k, 32)
    splits, kb_per = 1, kb
    if partial and tiles * 4 <= sms and kb >= 6:
        want = min(sms // tiles, kb // 3)
        if want > 1:
            kb_per = cdiv(kb, want)
            splits = cdiv(kb, kb_per)
    return dict(tiles=tiles, per_cta=cdiv(tiles, min(tiles, sms)), splits=splits,
                last_split_kb=kb - (splits - 1) * kb_per)


def dw_plan(n, k, sms):
    """dw_tc / dw_bf16 + dw_node_splits: ceil(K / 256) column tiles x node splits of a multiple of 32 rows"""
    tiles = cdiv(k, 256)
    if n == 0:
        return dict(tiles=tiles, splits=0, waves=0, rows=0)
    want = max(1, min(sms // tiles, cdiv(n, 128)))
    rps = cdiv(cdiv(n, want), 32) * 32
    splits = cdiv(n, rps)
    return dict(tiles=tiles, splits=splits, waves=cdiv(tiles * splits, sms), rows=rps)


def dx_plan(n, k, sms):
    """dx_tc: persistent CTAs over ceil(N / 128) x ceil(K / 256) tiles"""
    tiles = cdiv(n, 128) * cdiv(k, 256)
    return dict(tiles=tiles, per_cta=cdiv(tiles, min(tiles, sms)))


def assert_regime(plan, want):
    got = {key: plan[key] for key in want}
    assert got == want, f"the case no longer covers its regime: planned {plan}, meant {want}"


def regime_id(prefix, regime):
    return prefix + "-" + "-".join(f"{v}{key}" for key, v in regime.items())


@pytest.fixture(scope="module")
def sms(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


# ---------------------------------------------------------------------------------------------- inputs and bars
def gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def features(kind, n, k, dev, seed):
    """[n, k] fp32: bag-of-words counts in 1..3 (TF32-exact) or tanh(N(0,1)) (not).  Every row, the last one
    included, holds counts in the whole last 32-column block (the K tail) and so in the last column."""
    g = gen(dev, seed)
    if kind == "dense":
        return torch.tanh(torch.randn(n, k, generator=g, device=dev))
    x = torch.zeros(n, k, device=dev)
    x.scatter_(1, torch.randint(0, k, (n, 12), generator=g, device=dev),
               torch.randint(1, 4, (n, 12), generator=g, device=dev).float())
    tail = (k - 1) // 32 * 32
    x[:, tail:] = torch.randint(1, 4, (n, k - tail), generator=g, device=dev).float()
    return x


def weights(k, dev, seed):
    g = gen(dev, seed)
    return [torch.randn(64, k, generator=g, device=dev) * 0.05 for _ in range(2)]


def rel_err(got, want):
    got, want = got.double(), want.double()
    return float((got - want).abs().max() / want.abs().max())


def assert_bf16_close(got, want, atol):
    """each element within 2^-8 |ref| + atol max|ref|: one bf16 rounding of an fp32-class value (on the device)"""
    got, want = got.double(), want.double()
    excess = float(((got - want).abs() - (2.0 ** -8 * want.abs() + atol * want.abs().max())).max())
    assert excess <= 0, excess


def bf16_k(k):
    """bf16 rows need K % 8 == 0: the 4- and 36-column tails become 8 and 40"""
    return cdiv(k, 8) * 8


def report(*what):
    print("[gemm-regimes]", *what)


def clib():
    import bigcn_b200
    return bigcn_b200.lib()


def stream():
    return torch.cuda.current_stream().cuda_stream


def mode_id(mode):
    from bigcn_b200 import _lib as L
    return L.GEMM_MODE[mode]


# ---------------------------------------------------------------------------------------------- X * W alone
XW_CASES = [pytest.param(n, k, dict(tiles=cdiv(n, 256), per_cta=1), id=f"N{n}-K{k}-tail-1tile-per-CTA")
            for n in (1, 255, 257) for k in (4, 36, 776, 5000)] + [
    pytest.param(37889, 768, dict(tiles=149, per_cta=2), id="N37889-K768-149tiles-2per-CTA-last-tile-1row"),
    pytest.param(75777, 768, dict(tiles=297, per_cta=3), id="N75777-K768-297tiles-3per-CTA"),
    pytest.param(40000, 5000, dict(tiles=157, per_cta=2), id="N40000-K5000-157tiles-2per-CTA")]


@pytest.mark.parametrize("n,k,regime", XW_CASES)
def test_xw_regimes(dev, sms, n, k, regime):
    """ops.xw (never split) in every mode, n_w = 1 and 2, both kinds of x; bigcn_xw with ldy = n_out + 4 into a NaN
    buffer with spare rows after N: bit-identical to the op in [N, n_out], the padding untouched."""
    from bigcn_b200 import ops
    from bigcn_b200._lib import check
    bad = []                                           # every error of the case is reported before the verdict
    for kk in sorted({k, bf16_k(k)}):
        modes = [m for m in MODES if (bf16_k(k) if m == "bf16" else k) == kk]
        assert_regime(xw_plan(n, kk, sms), dict(regime, splits=1))
        ws = weights(kk, dev, seed=kk)
        wcat = torch.cat(ws).double()
        for kind in ("bow", "dense"):
            x32 = features(kind, n, kk, dev, seed=n + kk)
            for mode in modes:
                x = x32.to(torch.bfloat16) if mode == "bf16" else x32
                want = x.double() @ wcat.t()
                for n_w in (1, 2):
                    got = ops.xw(x, ws[:n_w], mode)
                    assert torch.equal(got, ops.xw(x, ws[:n_w], mode)), (mode, kind, n_w)
                    e = rel_err(got, want[:, :64 * n_w])
                    report("xw", n, kk, mode, kind, n_w, f"{e:.3e}")
                    if mode == "tf32":
                        ok = e < 2e-3                                  # one TF32 pass: 10-bit mantissas
                    elif mode == "tf32x2" and kind == "dense":         # W split only: x itself is rounded to TF32
                        ok = e < 2e-3 and (kk < 36 or e > 1e-5)
                    elif kind == "bow":
                        ok = e < 2e-6
                    else:
                        # dense rows: 1e-5 up to 768 terms.  Longer rows scale it by K / 768: every K step adds its
                        # products into the fp32 TMEM accumulator, and on dense signed rows that error grows like K
                        # (tf32x3 at K = 5000: 3.4-4.4e-5, 6.4x its K = 776 value) where the fp32 scan's grows like
                        # sqrt(K) (2.5-3.0e-6).  Bag-of-words rows, with ~20 non-zero terms, stay at 2e-6.
                        ok = e < 1e-5 * max(1.0, kk / 768)
                    if not ok:
                        bad.append((mode, kind, n_w, e))
                ldy = 128 + 4
                y = torch.full((n + 3, ldy), NAN, device=dev)
                scr = torch.empty(clib().bigcn_xw_scratch_floats(kk, 2), device=dev)
                check(clib().bigcn_xw(x.data_ptr(), n, kk, ws[0].data_ptr(), ws[1].data_ptr(), kk, y.data_ptr(), ldy,
                                      mode_id(mode), scr.data_ptr(), stream()), "xw")
                assert torch.equal(y[:n, :128], got), (mode, kind)
                assert bool(y[:n, 128:].isnan().all()) and bool(y[n:].isnan().all()), (mode, kind)
    assert not bad, bad


# ---------------------------------------------------------------------------------------------- dW alone
DW_K = {4: (1, 148), 200: (1, 148), 776: (4, 37), 5000: (20, 7), 40000: (157, 1)}   # K: (column tiles, full splits)


def _dw_cases():
    out = []
    for k, (tiles, full) in DW_K.items():
        big = 23679 if tiles <= 148 else 4097      # 23,679 = 148 splits of 160 rows (37 of 640, 7 of 3392) less one
        for n in (0, 1, 31, 33, 129, big):
            splits = 0 if n == 0 else 1 if n <= 128 or tiles > 148 else 2 if n == 129 else full
            regime = dict(tiles=tiles, splits=splits, waves=cdiv(tiles * splits, 148))
            out.append(pytest.param(n, k, regime, id=regime_id(f"K{k}-N{n}", regime)))
    return out


@pytest.mark.parametrize("n,k,regime", _dw_cases())
def test_dw_regimes(dev, sms, n, k, regime):
    """n_w = 1 through torch.ops.bigcn_b200.xw_wgrad (twice, bit-identical); n_w = 2 through bigcn_xw_wgrad with
    ldw = K + 4 into NaN: the padding columns untouched.  tf32x2 is mixed's dW1.  N = 0 returns zeros."""
    import bigcn_b200.torch_ops  # noqa: F401  (registers the ops)
    from bigcn_b200._lib import check
    g = gen(dev, 7 + n)
    t = torch.randn(n, 128, generator=g, device=dev)
    t[:, ::2] = t[:, ::2].abs()                        # one-signed columns: a biased lo rounding accumulates
    bad = []                                           # every error of the case is reported before the verdict
    for kk in sorted({k, bf16_k(k)}):
        modes = [m for m in MODES if (bf16_k(k) if m == "bf16" else k) == kk]
        plan = dw_plan(n, kk, sms)
        assert_regime(plan, regime)
        for kind in ("bow", "dense"):
            x32 = features(kind, n, kk, dev, seed=n + kk + 1)
            for mode in modes:
                x = x32.to(torch.bfloat16) if mode == "bf16" else x32
                want = t.double().t() @ x.double()
                scr = torch.empty(clib().bigcn_xw_wgrad_scratch_floats(n, kk, 2), device=dev)

                def wgrad2(md, xin):
                    dw = torch.full((2, 64, kk + 4), NAN, device=dev)
                    check(clib().bigcn_xw_wgrad(xin.data_ptr(), n, kk, t.data_ptr(), 2, dw[0].data_ptr(),
                                                dw[1].data_ptr(), kk + 4, mode_id(md), scr.data_ptr(), stream()),
                          "xw_wgrad")
                    assert bool(dw[:, :, kk:].isnan().all()), (md, kind)
                    return dw[:, :, :kk].reshape(128, kk)
                got1 = torch.ops.bigcn_b200.xw_wgrad(x, t[:, :64], mode)
                assert torch.equal(got1, torch.ops.bigcn_b200.xw_wgrad(x, t[:, :64], mode)), (mode, kind)
                got2 = wgrad2(mode, x)
                if n == 0:
                    assert not bool(got1.any()) and not bool(got2.any()), mode
                    continue
                ctrl = rel_err(wgrad2("fp32", x.float()), want)     # the fp32 scan on the same (widened) x
                # 1e-5 up to 768 node rows per split, then scaled by rows / 768: as for X * W, the TMEM accumulator's
                # error grows with the terms it sums, and one-signed columns of T times bag-of-words counts add them all
                # with one sign (tf32x3 at 3,392 and 4,128 rows per split: 2.6-3.8e-5 against an fp32 control of 3-6e-7)
                bar = max(1e-5 * max(1.0, plan["rows"] / 768), 2 * ctrl)
                for n_w, got in ((1, got1), (2, got2)):
                    e = rel_err(got, want[:64 * n_w])
                    report("dw", n, kk, mode, kind, n_w, f"{e:.3e}", f"control {ctrl:.3e}")
                    if mode == "tf32" or (mode == "tf32x2" and kind == "dense"):
                        ok = e < 2e-3                                # x (and in tf32 T) rounded to TF32 once
                    else:
                        ok = e < bar
                    if not ok:
                        bad.append((mode, kind, n_w, e, ctrl))
    assert not bad, bad


# ---------------------------------------------------------------------------------------------- dX alone
def _dx_cases():
    out = []
    for n in (1, 129, 40000):
        for k in (8, 257, 768, 5000):
            regime = dx_plan(n, k, 148)
            out.append(pytest.param(n, k, regime, id=regime_id(f"N{n}-K{k}", regime)))
    return out


@pytest.mark.parametrize("n,k,regime", _dx_cases())
def test_dx_regimes(dev, sms, n, k, regime):
    """ops.x_dgrad with fp32 and bf16 output, n_w = 1 and 2, twice each (bit-identical); bigcn_x_dgrad into larger NaN
    buffers: once 4 bytes off the 16-byte boundary (the scalar store path although K % 4 == 0 for most K), once
    aligned with bf16 output.  Both bit-identical to the op inside [N, K], the rest untouched."""
    from bigcn_b200 import ops
    from bigcn_b200._lib import check
    assert_regime(dx_plan(n, k, sms), regime)
    if n == 40000 and k == 768:
        assert regime["tiles"] > 2 * 148                # a CTA reaches accumulator 0 on its second phase
    g = gen(dev, n + k)
    ws = [torch.randn(64, k, generator=g, device=dev) * 0.05 for _ in range(2)]
    for n_w in (1, 2):
        t = torch.randn(n, 64 * n_w, generator=g, device=dev)
        want = t.double() @ torch.cat(ws[:n_w]).double()
        got = ops.x_dgrad(t, ws[:n_w])
        assert torch.equal(got, ops.x_dgrad(t, ws[:n_w])), n_w
        e = rel_err(got, want)
        report("dx", n, k, "fp32-out", n_w, f"{e:.3e}")
        assert e <= 1e-5, (n_w, e)
        gb = ops.x_dgrad(t, ws[:n_w], torch.bfloat16)
        assert torch.equal(gb, ops.x_dgrad(t, ws[:n_w], torch.bfloat16)), n_w
        assert_bf16_close(gb, want, 1e-5)
    scr = torch.empty(clib().bigcn_x_dgrad_scratch_floats(n, k, 2), device=dev)
    buf = torch.full((n * k + 8,), NAN, device=dev)
    check(clib().bigcn_x_dgrad(t.data_ptr(), 2, ws[0].data_ptr(), ws[1].data_ptr(), k, n, k, buf[1:].data_ptr(), None,
                               scr.data_ptr(), stream()), "x_dgrad")
    assert torch.equal(buf[1:1 + n * k].view(n, k), got)
    assert bool(buf[0].isnan()) and bool(buf[1 + n * k:].isnan().all())
    bufb = torch.full((n * k + 16,), NAN, dtype=torch.bfloat16, device=dev)
    check(clib().bigcn_x_dgrad(t.data_ptr(), 2, ws[0].data_ptr(), ws[1].data_ptr(), k, n, k, None, bufb.data_ptr(),
                               scr.data_ptr(), stream()), "x_dgrad")
    assert torch.equal(bufb[:n * k].view(n, k), gb)
    assert bool(bufb[n * k:].isnan().all())


# ---------------------------------------------------------------------------------------------- input contract
def test_tensor_core_input_contract(dev):
    """A misaligned x in tf32x3 and K % 4 != 0 in tf32 raise BigcnError and write nothing; gemm_mode='auto' resolves
    the same misaligned dense x to the exact fp32 scan, which matches the oracle."""
    import bigcn_b200
    from bigcn_b200 import ops
    n, k = 300, 768
    x = features("dense", n, k, dev, seed=1)
    flat = torch.zeros(n * k + 4, device=dev)
    xm = flat[1:1 + n * k].view(n, k)                  # contiguous, one float off the 16-byte boundary
    xm.copy_(x)
    x770 = features("dense", n, 770, dev, seed=2)
    for xin, mode, match in ((xm, "tf32x3", "16-byte"), (x770, "tf32", "multiple of 4")):
        kk = xin.shape[1]
        ws = weights(kk, dev, seed=kk)
        with pytest.raises(bigcn_b200.BigcnError, match=match):
            ops.xw(xin, ws, mode)
        y = torch.full((n, 128), NAN, device=dev)
        scr = torch.empty(clib().bigcn_xw_scratch_floats(kk, 2), device=dev)
        rc = clib().bigcn_xw(xin.data_ptr(), n, kk, ws[0].data_ptr(), ws[1].data_ptr(), kk, y.data_ptr(), 128,
                             mode_id(mode), scr.data_ptr(), stream())
        assert rc != 0 and bool(y.isnan().all()), mode
    b = make_batch("pheme", 24, seed=3, train=False)
    ref = fixed_oracle(768, seed=4).double().eval()
    m = bigcn_b200.BiGCN(768, 64, 64, dev).to(dev).eval()
    m.load_state_dict(ref.state_dict())
    bd = Batch(**{key: getattr(b, key).to(dev) for key in Batch._tensor_keys})
    nb, kb = b.x.shape
    flat = torch.zeros(nb * kb + 4, device=dev)
    bd.x = flat[1:1 + nb * kb].view(nb, kb)
    bd.x.copy_(b.x.to(dev))
    assert m.TDrumorGCN.resolved_gemm_mode(bd.x) == "fp32"
    got = m(bd)
    m.check_inputs()
    assert rel_err(got.cpu(), ref(b)) < 2.2e-5


# ---------------------------------------------------------------------------------------------- the feature path
def sizes_for(n):
    """PHEME-shaped trees of 101 nodes and one remainder tree: exactly n nodes"""
    return np.array([101] * (n // 101) + ([n % 101] if n % 101 else []), dtype=np.int64)


def to_dev(b, dev, x_dtype=torch.float32):
    d = Batch(**{key: getattr(b, key).to(dev) for key in Batch._tensor_keys})
    d.x = d.x.to(x_dtype).contiguous()
    return d


def assert_argmax(got, want, err):
    """identical argmax on every tree whose oracle margin between the top two classes exceeds twice the measured
    log-prob error: a closer pair is a tie at this precision"""
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    top2 = want.topk(2, dim=1).values
    clear = (top2[:, 0] - top2[:, 1]) > 2 * err * float(want.abs().max())
    assert torch.equal(got.argmax(1)[clear], want.argmax(1)[clear])
    assert float(clear.double().mean()) > 0.5


FEATURE_CASES = [
    pytest.param(9472, 768, dict(tiles=37, splits=4), False, id="N9472-K768-37tiles-4splits-eval"),
    pytest.param(9473, 768, dict(tiles=38, per_cta=1, splits=1), True, id="N9473-K768-38tiles-nosplit-last-tile-1row"),
    pytest.param(75777, 768, dict(tiles=297, per_cta=3, splits=1), True, id="N75777-K768-297tiles-3per-CTA"),
    pytest.param(255, 776, dict(tiles=1, splits=7, last_split_kb=1), False, id="N255-K776-1tile-7splits-1block-tail-eval")]


@pytest.mark.parametrize("n,k,regime,train", FEATURE_CASES)
def test_feature_path_regimes(dev, sms, n, k, regime, train):
    """BiGCN on dense PHEME-shaped features of exactly N rows against the fp64 oracle, in 'auto' (-> tf32x3), 'bf16'
    (the oracle on the bf16 x widened) and 'tf32'.  Eval (autograd and no-grad paths): log-probs 2.2e-5 (tf32: 1e-2
    and the argmax).  Train, with the kernel's Philox mask injected and x.requires_grad (dX at a high tile count
    inside the model): log-probs as in eval, and an x.grad of x's dtype.

    The gradients are not compared with the oracle at these sizes.  With ~26 k pre-activations per tree, some lie
    within rounding distance of zero: the kernel's ReLU and the oracle's can then differ, and with them every gradient
    of that tree (tf32x3 at N = 9,473: two trees, about 1e-3 in the TD parameter gradients, while the fp32 mode of the
    same model stays at 2e-6).  dX itself is held to 1e-5 at 939 and 6,260 tiles by test_dx_regimes, and the
    gradients to 1e-4 at smaller N by the model tests."""
    import bigcn_b200
    assert_regime(xw_plan(n, k, sms, partial=True), regime)
    b = make_batch("pheme", 0, seed=n, train=True, in_feats=k, sizes=sizes_for(n))
    assert b.x.shape == (n, k)
    ref = fixed_oracle(k, seed=5).double()
    keep = None
    for x_dt, modes in ((torch.float32, ("auto", "tf32")), (torch.bfloat16, ("bf16",))):
        bc = with_x(b, b.x.to(x_dt).float())
        ref.eval()
        with torch.no_grad():
            want = ref(bc)
        if train:
            ref.train()
        for mode in modes:
            m = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=mode).to(dev).eval()
            m.load_state_dict(ref.state_dict())
            bd = to_dev(bc, dev, x_dt)
            if mode == "auto":
                assert m.TDrumorGCN.resolved_gemm_mode(bd.x) == "tf32x3"
            ltol = 1e-2 if mode == "tf32" else 2.2e-5
            for grad in (True, False):
                with torch.set_grad_enabled(grad):
                    got = m(bd)
                m.check_inputs()
                e = rel_err(got.detach().cpu(), want)
                report("features eval", n, k, mode, f"grad={grad}", f"{e:.3e}")
                assert e < ltol, (mode, grad, e)
                if mode == "tf32":
                    assert_argmax(got, want, e)
            if not train:
                continue
            m.train()
            for mod in (m.TDrumorGCN, m.BUrumorGCN):
                mod.seed, mod._calls = 777, 0
            x = bd.x.detach().clone().requires_grad_(True)
            out = m(with_x(bd, x))
            F.nll_loss(out, bd.y).backward()
            m.check_inputs()
            if keep is None:
                keep = masks_for(m.TDrumorGCN.last_seed, n, k)
            if mode != "tf32":               # the oracle's train forward, once per x (the same mask for every mode)
                with torch.no_grad():
                    wt = ref(bc, keep_td=keep[0], keep_bu=keep[1])
            e = rel_err(out.detach().cpu(), wt)
            report("features train", n, k, mode, "logp", f"{e:.3e}")
            assert e < ltol, (mode, e)
            assert x.grad.dtype == x_dt and x.grad.shape == (n, k) and bool(x.grad.isfinite().all()), mode


def test_fused_trainer_step_at_bench_batch_tf32x3(dev, sms):
    """bench.py's first batch (128 Twitter16-shaped trees, seed 1000, K = 5000) in gemm_mode='tf32x3': one
    FusedTrainer.step against the fp64 oracle handed the kernel's Philox mask, at the bars of
    test_fused_trainer_step_at_bench_configuration (loss and log-probs 1e-5, the ten gradients 1e-4)."""
    import bigcn_b200
    from bigcn_b200.trainer import _ORDER
    from oracle import gcn_oracle
    K = 5000
    b = make_batch_shard("twitter16", 128, 1000)[0]
    n = int(b.x.shape[0])
    assert n > 20000
    assert_regime(xw_plan(n, K, sms, partial=True), dict(per_cta=1, splits=1))
    assert_regime(dw_plan(n, K, sms), dict(tiles=20, splits=7, waves=1))
    ref = fixed_oracle(K, seed=0).double().train()
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="tf32x3", validate="off").to(dev).train()
    m.load_state_dict(ref.state_dict())
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, graphs=False)
    seed = 12345
    loss = tr.step(to_dev(b, dev), seed=seed)
    tr.check_inputs()
    keep = [torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, d, np.arange(n), 64 + K, 0.5)) for d in (0, 1)]
    want = ref(b, keep_td=keep[0], keep_bu=keep[1])
    want_loss = F.nll_loss(want, b.y)
    want_loss.backward()
    e = rel_err(tr.last_logp.cpu(), want)
    report("bench batch tf32x3 logp", f"{e:.3e}")
    assert e < 1e-5
    assert abs(float(loss.item()) - float(want_loss)) <= 1e-5 * max(1.0, abs(float(want_loss)))
    for name, q in ref.named_parameters():
        e = rel_err(tr.gviews[name].cpu(), q.grad)
        report("bench batch tf32x3", name, f"{e:.3e}")
        assert e < 1e-4, (name, e)


# ---------------------------------------------------------------------------------------------- gemm_mode='mixed'
@pytest.mark.parametrize("shape,k,trees", [("twitter15", 5000, 10), ("pheme", 768, 40)])
def test_mixed_mode_training(dev, shape, k, trees):
    """'mixed': the exact fp32 scan forward, dW1 by the TF32X2 split (T split hi + lo, x as it is).  Against the fp64
    oracle with the Philox mask injected.  Bag-of-words counts are TF32-exact: log-probs 1e-5 and all ten gradients
    1e-4.  Dense signed features are not: the forward and eight gradients keep their bars, while the two conv1 weight
    gradients are pinned above 1e-5 and below 2e-3 (one TF32 rounding of each x, at most 2^-10 relative)."""
    import bigcn_b200
    b = make_batch(shape, trees, seed=6, train=True, in_feats=k)
    n = b.x.shape[0]
    ref = fixed_oracle(k, seed=7).double().train()
    m = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode="mixed").to(dev).train()
    m.load_state_dict(ref.state_dict())
    for mod in (m.TDrumorGCN, m.BUrumorGCN):
        mod.seed, mod._calls = 777, 0
    got = m(to_dev(b, dev))
    m.check_inputs()
    keep = masks_for(m.TDrumorGCN.last_seed, n, k)
    want = ref(b, keep_td=keep[0], keep_bu=keep[1])
    e = rel_err(got.detach().cpu(), want)
    report("mixed", shape, "logp", f"{e:.3e}")
    assert e < (1e-5 if shape != "pheme" else 2.2e-5)
    F.nll_loss(want, b.y).backward()
    F.nll_loss(got, b.y.to(dev)).backward()
    for (name, p), q in zip(m.named_parameters(), ref.parameters()):
        e = rel_err(p.grad.cpu(), q.grad)
        report("mixed", shape, name, f"{e:.3e}")
        if shape == "pheme" and name.endswith("conv1.lin.weight"):
            assert 1e-5 < e < 2e-3, (name, e)
        else:
            assert e < 1e-4, (name, e)
