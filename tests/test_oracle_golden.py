"""Pin oracle/moco_oracle.py against outputs of the UNMODIFIED reference
(tests/golden/*.npz, produced by tests/golden/gen_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import moco_oracle as O
from tests.helpers import load_contrast_golden


@pytest.fixture(scope="module")
def ids(golden_dir):
    return np.load(os.path.join(golden_dir, "shuffle_ids.npz"))


@pytest.fixture(scope="module")
def contrast(golden_dir):
    return load_contrast_golden(golden_dir)


@pytest.fixture(scope="module")
def shuffle(golden_dir):
    return np.load(os.path.join(golden_dir, "shuffle.npz"))


def test_shuffle_ids_bit_exact(ids):
    keys = [k for k in ids.files if k.startswith("fwd_")]
    assert len(keys) >= 8
    for k in keys:
        _, bsz, epoch = k.split("_")
        fwd, bwd = O.get_shuffle_ids(int(bsz), int(epoch))
        assert fwd.dtype == np.int64 and bwd.dtype == np.int64
        np.testing.assert_array_equal(fwd, ids[k])
        np.testing.assert_array_equal(bwd, ids["bwd_" + k[4:]])
        np.testing.assert_array_equal(fwd[bwd], np.arange(int(bsz)))


def test_mt19937_known_answer():
    # first outputs of mt19937 seeded with 5489 (the C++11 default seed): 3499211612, 581869302 ...
    raw = O.MT19937(5489).random_raw(3)
    assert [int(x) for x in raw] == [3499211612, 581869302, 3890346734]
    # and across a twist boundary: 10000th output of default-seeded mt19937 is 4123659995 (C++11 [rand.predef])
    assert int(O.MT19937(5489).random_raw(10000)[-1]) == 4123659995


@pytest.mark.parametrize("name", ["c1head", "wrap", "c256", "ragged"])
def test_contrast_head_matches_reference(contrast, name):
    N, C, K, A, steps = (int(v) for v in contrast[f"{name}_meta"])
    T = float(contrast[f"{name}_T"][0])
    mem = O.MemoryMoCoOracle(contrast[f"{name}_memory0"], T, index=0)
    for s in range(steps):
        q, k, k_all = (contrast[f"{name}_s{s}_{x}"] for x in ("q", "k", "k_all"))
        idx_before, idx_after = (int(v) for v in contrast[f"{name}_s{s}_index"])
        assert mem.index == idx_before
        pre = mem.memory.copy()
        out = mem.logits(q, k)
        ref = contrast[f"{name}_s{s}_logits"]
        assert out.shape == ref.shape == (N, K + 1)
        np.testing.assert_allclose(out, ref, rtol=2e-5, atol=2e-5)
        assert abs(O.nce_softmax_loss(ref) - float(contrast[f"{name}_s{s}_loss"][0])) < 1e-5
        assert abs(O.prob_metric(ref) - float(contrast[f"{name}_s{s}_prob"][0])) < 1e-6
        dq = O.nce_backward_dq(q, k, pre, T)
        np.testing.assert_allclose(dq, contrast[f"{name}_s{s}_dq"], rtol=1e-4, atol=1e-6)
        ids = mem.enqueue(k_all)
        np.testing.assert_array_equal(ids, (idx_before + np.arange(A)) % K)
        assert mem.index == idx_after
    np.testing.assert_array_equal(mem.memory, contrast[f"{name}_memory_final"])


def test_state_dict_contract(contrast):
    assert list(contrast["state_dict_keys"]) == ["memory", "params"]
    np.testing.assert_array_equal(contrast["state_dict_params"], np.array([-1]))


@pytest.mark.parametrize("tag,world,n,epoch", [("w1_n8_e3", 1, 8, 3), ("w2_n4_e7", 2, 4, 7), ("w4_n6_e2", 4, 6, 2)])
def test_shufflebn_matches_reference(shuffle, tag, world, n, epoch):
    xs = [shuffle[f"{tag}_r{r}_x"] for r in range(world)]
    outs, bwd = O.forward_shuffle(xs, epoch)
    for r in range(world):
        np.testing.assert_array_equal(outs[r], shuffle[f"{tag}_r{r}_x_shuf"])
        np.testing.assert_array_equal(bwd, shuffle[f"{tag}_r{r}_binds"])
    feats = [shuffle[f"{tag}_r{r}_feat"] for r in range(world)]
    f_all, f_loc = O.backward_shuffle(feats, bwd, return_local=True)
    for r in range(world):
        np.testing.assert_array_equal(f_all, shuffle[f"{tag}_r{r}_feat_all"])
        np.testing.assert_array_equal(f_loc[r], shuffle[f"{tag}_r{r}_feat_local"])
        # S6: the local result corresponds row-for-row with this rank's original x
        np.testing.assert_array_equal(f_loc[r], xs[r].reshape(n, -1)[:, :16])


def test_bf16_round_matches_torch():
    import torch
    x = np.random.RandomState(0).randn(1000).astype(np.float32) * 3
    ref = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    np.testing.assert_array_equal(O.bf16_round(x), ref)


@pytest.mark.parametrize("tag", ["m999", "m99", "m0"])
def test_moment_update_bit_exact(golden_dir, tag):
    """oracle.moment_update vs the reference's util.moment_update (util.py:124-127), fp32 bit patterns."""
    z = np.load(os.path.join(golden_dir, "ema.npz"))
    n, m = int(z[f"{tag}_n"][0]), float(z[f"{tag}_m"][0])
    ema = [z[f"{tag}_ema0_{i}"] for i in range(n)]
    for s in range(int(z[f"{tag}_steps"][0])):
        ema = O.moment_update([z[f"{tag}_s{s}_p_{i}"] for i in range(n)], ema, m)
        for i, a in enumerate(ema):
            np.testing.assert_array_equal(a.view(np.uint32), z[f"{tag}_s{s}_ema_{i}"].view(np.uint32))


@pytest.mark.parametrize("name", ["c1head", "wrap", "c256", "ragged"])
def test_one_sweep_algorithm_matches_reference(contrast, name):
    """The one-pass kernel's algorithm (fixed first-tile stabiliser, no rescaling, slice merge), restated in numpy,
    against the reference's own lse-derived outputs and gradient on the golden inputs."""
    g = contrast
    N, C, K, A, steps = (int(v) for v in g[f"{name}_meta"])
    T = float(g[f"{name}_T"][0])
    orc = O.MemoryMoCoOracle(g[f"{name}_memory0"], T)
    for s in range(steps):
        q, k, k_all = g[f"{name}_s{s}_q"], g[f"{name}_s{s}_k"], g[f"{name}_s{s}_k_all"]
        pre = orc.memory.copy()
        for tile, slices in ((128, 4), (64, 3), (16, 7)):
            lse, prob, dq = O.one_sweep_head(q, k, pre, T, tile=tile, slices=slices)
            logits = g[f"{name}_s{s}_logits"]
            ref_lse = O.logsumexp_rows(logits)
            assert np.abs(lse - ref_lse).max() < 2e-5 * max(1.0, np.abs(ref_lse).max())
            assert abs(float(prob.mean()) - float(g[f"{name}_s{s}_prob"][0])) < 1e-4 * float(g[f"{name}_s{s}_prob"][0]) + 1e-9
            ref_dq = g[f"{name}_s{s}_dq"]
            assert np.abs(dq - ref_dq).max() / np.abs(ref_dq).max() < 1e-4
        orc.forward(q, k, k_all)


def test_one_sweep_overflow_contract():
    """A logit more than ~88 nats above its slice's first-tile maximum overflows the fp32 sum: the result is
    non-finite (loud), never a finite wrong number; within the limit the sweep is exact."""
    rng = np.random.default_rng(3)
    N, C, K, T = 8, 32, 1024, 0.07
    unit = lambda n: O.l2_normalize(rng.standard_normal((n, C)).astype(np.float32))
    q, k, mem = unit(N) * 12.0, unit(N), unit(K)
    mem[900] = q[2] / 12.0                                    # logit 12 / 0.07 = 171 nats, far from tile 0 of its slice
    lse, prob, dq = O.one_sweep_head(q, k, mem, T, tile=128, slices=2)
    assert not np.isfinite(lse[2])
    ok = [i for i in range(N) if i != 2]
    out = O.MemoryMoCoOracle(mem, T).logits(q, k)
    assert np.abs(lse[ok] - O.logsumexp_rows(out)[ok]).max() < 1e-3
    lse1, _, dq1 = O.one_sweep_head(q / 12.0, k, mem, T, tile=128, slices=2)     # normalised features: exact
    out1 = O.MemoryMoCoOracle(mem, T).logits(q / 12.0, k)
    assert np.abs(lse1 - O.logsumexp_rows(out1)).max() < 2e-5 * np.abs(out1).max()
    ref_dq = O.nce_backward_dq(q / 12.0, k, mem, T)
    assert np.abs(dq1 - ref_dq).max() / np.abs(ref_dq).max() < 1e-4


def test_normalize_head_matches_reference(golden_dir):
    """Normalize (resnet.py:24-33) -> head -> gradient w.r.t. the RAW encoder output, against the reference's own
    autograd (tests/golden/normalize.npz)."""
    g = np.load(os.path.join(golden_dir, "normalize.npz"))
    for name in ("n128", "n64"):
        N, C, K, A = (int(v) for v in g[f"{name}_meta"])
        T = float(g[f"{name}_T"][0])
        loss, prob, dxq, q, k = O.head_with_normalize(g[f"{name}_xq"], g[f"{name}_xk"], g[f"{name}_memory0"], T)
        np.testing.assert_allclose(q, g[f"{name}_q"], rtol=0, atol=1e-6)
        np.testing.assert_allclose(k, g[f"{name}_k"], rtol=0, atol=1e-6)
        assert abs(loss - float(g[f"{name}_loss"][0])) < 1e-5
        assert abs(prob - float(g[f"{name}_prob"][0])) < 1e-6
        ref = g[f"{name}_dxq"]
        assert np.abs(dxq - ref).max() / np.abs(ref).max() < 1e-4
        # enqueue of the normalised keys (Contrast.py:29-34)
        orc = O.MemoryMoCoOracle(g[f"{name}_memory0"], T)
        orc.enqueue(O.l2_normalize(g[f"{name}_xk_all"]))
        np.testing.assert_allclose(orc.memory, g[f"{name}_memory_final"], rtol=0, atol=1e-6)
        # the kernels' operand contract (bf16 q^ for the negatives) stays within the bf16 quantisation of the logits
        l2, p2, d2, _, _ = O.head_with_normalize(g[f"{name}_xq"], g[f"{name}_xk"], g[f"{name}_memory0"], T, True)
        assert abs(l2 - loss) < 5e-3 and np.abs(d2 - dxq).max() / np.abs(dxq).max() < 2e-2


# ---------------------------------------------------------------------------------------------------------------------
# encoder-side ops (BatchNorm group, stem max-pool, space-to-depth conv1): oracle/encoder_ops_oracle.py against tensors
# captured inside the reference's own ResNet / Bottleneck modules (tests/golden/gen_golden.py:gen_encoder_ops)
# ---------------------------------------------------------------------------------------------------------------------
def _enc(golden_dir):
    return np.load(os.path.join(golden_dir, "encoder_ops.npz"))


def _close(a, b, rtol=2e-5, atol=2e-5):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol * max(1.0, float(np.abs(b).max())))


def test_encoder_oracle_stem_bn_relu_maxpool_matches_reference_modules(golden_dir):
    """resnet.py:155-158: conv1 output -> bn1 -> relu -> maxpool, forward and autograd."""
    from oracle import encoder_ops_oracle as E
    g = _enc(golden_dir)
    x = g["stem_conv1"]
    y, mean, invstd = E.bn_act_forward(x, g["stem_gamma"], g["stem_beta"], None, True)
    pooled, taps = E.maxpool3x3s2_forward(y)
    _close(pooled, g["stem_pooled"])
    dy = E.maxpool3x3s2_backward(g["stem_dpooled"], taps, y.shape)
    dx, dgamma, dbeta, dres = E.bn_act_backward(x, g["stem_gamma"], g["stem_beta"], dy, None, True)
    assert dres is None
    _close(dx, g["stem_dconv1"], 2e-4, 2e-5)
    _close(dgamma, g["stem_dgamma"], 2e-4, 2e-5)
    _close(dbeta, g["stem_dbeta"], 2e-4, 2e-5)
    mean_, var_ = E.batchnorm_stats(x)
    rm, rv = E.running_stats_update(g["stem_running_mean0"], g["stem_running_var0"], mean_, var_,
                                    x.shape[0] * x.shape[2] * x.shape[3])
    _close(rm, g["stem_running_mean"])
    _close(rv, g["stem_running_var"])


def test_encoder_oracle_bn_add_relu_matches_reference_bottleneck(golden_dir):
    """resnet.py:95-102: conv3 output -> bn3 -> += residual -> relu, incl. the gradient that reaches the residual."""
    from oracle import encoder_ops_oracle as E
    g = _enc(golden_dir)
    x, res = g["blk_conv3"], g["blk_res"]
    y, _, _ = E.bn_act_forward(x, g["blk_gamma"], g["blk_beta"], res, True)
    _close(y, g["blk_out"])
    dx, dgamma, dbeta, dres = E.bn_act_backward(x, g["blk_gamma"], g["blk_beta"], g["blk_dout"], res, True)
    _close(dx, g["blk_dconv3"], 2e-4, 2e-5)
    _close(dres, g["blk_dres"])
    _close(dgamma, g["blk_dgamma"], 2e-4, 2e-5)
    _close(dbeta, g["blk_dbeta"], 2e-4, 2e-5)


def test_space_to_depth_stem_is_the_reference_conv1(golden_dir):
    """resnet.py:112,155: the 7x7 / 2 / pad 3 convolution the reference ran == the 4x4 / 1 / pad 0 convolution over the
    space-to-depth layout with the re-indexed weights -- oracle restatement, and moco_b200.encoders.StemConv on CPU."""
    from oracle import encoder_ops_oracle as E
    g = _enc(golden_dir)
    xs, ws = E.s2d_layout(g["stem_x"]), E.stem_weight_s2d(g["stem_w"])
    assert xs.shape == (4, 16, 19, 19) and ws.shape == (64, 16, 4, 4)
    _close(E.conv2d_valid(xs, ws), g["stem_conv1"], 2e-5, 2e-5)
    from moco_b200.encoders import StemConv
    stem = StemConv()
    with torch.no_grad():
        stem.weight.copy_(torch.from_numpy(g["stem_w"]))
        np.testing.assert_array_equal(stem.s2d_weight().numpy(), ws)
        _close(stem(torch.from_numpy(xs)).numpy(), g["stem_conv1"], 2e-5, 2e-5)
        _close(stem(torch.from_numpy(g["stem_x"])).numpy(), g["stem_conv1"], 2e-5, 2e-5)


def test_norm_modules_off_the_gpu_reproduce_the_reference_modules(golden_dir):
    """BatchNormAct2d / MaxPool3x3s2 on CPU tensors (their torch path) against the same captured tensors."""
    from moco_b200.bn import BatchNormAct2d, MaxPool3x3s2
    g = _enc(golden_dir)
    bn = BatchNormAct2d(64, relu=True)
    with torch.no_grad():
        bn.weight.copy_(torch.from_numpy(g["blk_gamma"]))
        bn.bias.copy_(torch.from_numpy(g["blk_beta"]))
    x = torch.from_numpy(g["blk_conv3"]).requires_grad_(True)
    res = torch.from_numpy(g["blk_res"]).requires_grad_(True)
    y = bn(x, res)
    y.backward(torch.from_numpy(g["blk_dout"]))
    _close(y.detach().numpy(), g["blk_out"])
    _close(x.grad.numpy(), g["blk_dconv3"], 2e-5, 2e-5)
    _close(res.grad.numpy(), g["blk_dres"])
    _close(bn.running_var.numpy(), g["blk_running_var"])
    stem_bn = BatchNormAct2d(64, relu=True)
    with torch.no_grad():
        stem_bn.weight.copy_(torch.from_numpy(g["stem_gamma"]))
        stem_bn.bias.copy_(torch.from_numpy(g["stem_beta"]))
    _close(MaxPool3x3s2()(stem_bn(torch.from_numpy(g["stem_conv1"]))).detach().numpy(), g["stem_pooled"])
