"""GPU tests of the tcgen05/TMA GEMM modes of X * W^T (north_star: TF32 mode within 1e-2
relative with identical argmax; the split mode restores fp32-class accuracy on BoW counts)."""
import numpy as np
import pytest
import torch

from oracle import bigcn_oracle
from bigcn_b200.data import make_batch

pytestmark = pytest.mark.gpu


def rel_err(got, want):
    want = want.detach().cpu().double()
    got = got.detach().cpu().double()
    return float((got - want).abs().max()) / max(float(want.abs().max()), 1e-30)


@pytest.mark.parametrize("n_trees,k", [(3, 5000), (9, 5000), (2, 64), (5, 768)])
def test_xw_tensor_core_matches_fp64(dev, n_trees, k):
    from bigcn_b200 import ops
    torch.manual_seed(0)
    shape = "pheme" if k == 768 else "twitter15"
    b = make_batch(shape, n_trees, seed=11, train=False, in_feats=k)
    x_tf32_exact = shape != "pheme"            # BoW counts are TF32-representable, tanh(N(0,1)) features are not
    w_td, w_bu = torch.randn(64, k) * 0.05, torch.randn(64, k) * 0.05
    want = b.x.double() @ torch.cat([w_td, w_bu]).double().t()
    x = b.x.to(dev)
    got = ops.xw(x, [w_td.to(dev), w_bu.to(dev)], "tf32")
    assert got.shape == want.shape
    assert rel_err(got, want) < 2e-3           # one TF32 pass: 10-bit mantissa on W
    got3 = ops.xw(x, [w_td.to(dev), w_bu.to(dev)], "tf32x3")
    tol3 = 2e-6 if k != 768 else 1e-5          # dense 768-term rows: fp32 accumulation order in the MMA
    assert rel_err(got3, want) < tol3          # X and W both split hi/lo: fp32-class on ANY input
    got2 = ops.xw(x, [w_td.to(dev), w_bu.to(dev)], "tf32x2")
    if x_tf32_exact:
        assert rel_err(got2, want) < tol3      # W split only: exact when X is TF32-representable
    else:
        assert 1e-5 < rel_err(got2, want) < 2e-3   # ... and visibly not when it is not (why TF32X3 splits X too)
    one = ops.xw(x, [w_bu.to(dev)], "tf32x3")  # single direction, N = 64 MMA
    assert rel_err(one, want[:, 64:]) < tol3
    # fp32 scan and tensor-core split agree
    ref = ops.xw(x, [w_td.to(dev), w_bu.to(dev)], "fp32")
    assert rel_err(got3, ref) < tol3


def test_model_in_tf32_mode(dev):
    import bigcn_b200
    torch.manual_seed(1)
    b = make_batch("twitter15", 16, seed=2, train=False)
    ref = bigcn_oracle.BiGCN(5000, 64, 64).eval()
    want = ref(b)
    for mode, tol in (("tf32", 1e-2), ("tf32x3", 1e-5)):
        m = bigcn_b200.BiGCN(5000, 64, 64, dev, gemm_mode=mode).to(dev).eval()
        m.load_state_dict(ref.state_dict())
        got = m(b.to(dev) if not b.x.is_cuda else b)
        m.check_inputs()
        e = rel_err(got, want)
        assert e < tol + (1.2e-5 if mode == "tf32x3" else 0), f"{mode}: {e:.3e}"
        assert torch.equal(got.argmax(1).cpu(), want.argmax(1)), mode


def test_training_gradients_tensor_core(dev):
    """dW1 through the MN-major tcgen05 GEMM: fp32-class in the split mode, 1e-2 in plain TF32."""
    import bigcn_b200
    from oracle import gcn_oracle
    b = make_batch("twitter15", 10, seed=4, train=True)
    n = b.x.shape[0]
    for mode, gtol, ltol in (("tf32x3", 1e-4, 2.2e-5), ("tf32", 1e-2, 1e-2)):
        torch.manual_seed(3)
        ref = bigcn_oracle.BiGCN(5000, 64, 64).train()
        m = bigcn_b200.BiGCN(5000, 64, 64, dev, gemm_mode=mode).to(dev).train()
        m.load_state_dict(ref.state_dict())
        got = m(make_dev(b, dev))
        seed = m.TDrumorGCN.last_seed
        ktd = torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, 0, np.arange(n), 5064, 0.5))
        kbu = torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, 1, np.arange(n), 5064, 0.5))
        want = ref(b, keep_td=ktd, keep_bu=kbu)
        assert rel_err(got, want) < ltol, mode
        torch.nn.functional.nll_loss(want, b.y).backward()
        torch.nn.functional.nll_loss(got, b.y.to(dev)).backward()
        for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
            e = rel_err(p.grad, q.grad)
            assert e < gtol, f"{mode} {name}: {e:.3e}"


@pytest.mark.parametrize("shape,k", [("twitter16", 520), ("pheme", 768)])
def test_gcnconv_tensor_core_backward(dev, shape, k):
    """tf32x3 on BoW counts and on dense signed features (not TF32-representable: needs the X split)."""
    import bigcn_b200
    from oracle import gcn_oracle
    torch.manual_seed(5)
    b = make_batch(shape, 7 if shape != "pheme" else 60, seed=6, train=True, in_feats=k)
    ref = gcn_oracle.GCNConv(k, 64)
    conv = bigcn_b200.GCNConv(k, 64, gemm_mode="tf32x3").to(dev)
    conv.load_state_dict(ref.state_dict())
    want = ref(b.x, b.edge_index)
    got = conv(b.x.to(dev), b.edge_index.to(dev))
    assert rel_err(got, want) < 1e-5
    g = torch.randn_like(want)
    want.backward(g); got.backward(g.to(dev))
    assert rel_err(conv.lin.weight.grad, ref.lin.weight.grad) < 1e-4
    assert rel_err(conv.bias.grad, ref.bias.grad) < 1e-4


def make_dev(b, dev):
    from bigcn_b200.data import Batch
    return Batch(**{k: getattr(b, k).to(dev) for k in Batch._tensor_keys})


def test_ffma_mix_kernels_match_oracle(dev):
    """The FFMA kernels of conv2.lin and its backward (k_prop1_mix, k_bwd_mix) against the oracle: train-mode log-probs
    1e-5 with the kernel's Philox mask injected, all ten gradients 1e-4, then eval mode."""
    import bigcn_b200
    from oracle import gcn_oracle
    for shape, k, trees in (("twitter15", 5000, 9), ("pheme", 768, 40)):
        b = make_batch(shape, trees, seed=21, train=True, in_feats=k)
        n = b.x.shape[0]
        torch.manual_seed(8)
        ref = bigcn_oracle.BiGCN(k, 64, 64).train()
        with torch.no_grad():
            for p in ref.parameters():
                if p.dim() == 1:
                    p.uniform_(-0.1, 0.1)
        m = bigcn_b200.BiGCN(k, 64, 64, dev).to(dev).train()
        m.load_state_dict(ref.state_dict())
        got = m(make_dev(b, dev))
        m.check_inputs()
        seed = m.TDrumorGCN.last_seed
        ktd = torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, 0, np.arange(n), 64 + k, 0.5))
        kbu = torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, 1, np.arange(n), 64 + k, 0.5))
        want = ref(b, keep_td=ktd, keep_bu=kbu)
        assert rel_err(got, want) < (1e-5 if k == 5000 else 2.2e-5), shape
        torch.nn.functional.nll_loss(want, b.y).backward()
        torch.nn.functional.nll_loss(got, b.y.to(dev)).backward()
        for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
            e = rel_err(p.grad, q.grad)
            assert e < 1e-4, f"{shape} {name}: {e:.3e}"
        # eval mode: the root projection P is added instead
        m.eval(); ref.eval()
        assert rel_err(m(make_dev(b, dev)), ref(b)) < (1e-5 if k == 5000 else 2.2e-5)
