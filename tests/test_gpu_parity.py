"""GPU parity tests (run with ``-m gpu`` on a B200): the CUDA path, called through the C ABI
(ctypes -> libmoco_b200.so) by the Python mirror of the reference API, against
(a) the golden vectors produced by the unmodified reference and (b) the numpy oracle on seeded
inputs.  Tolerances: logits 1e-3 relative to max|logit| (BASELINE.json north_star) on identical
bf16-representable inputs -- in practice ~1e-6; queue contents / indices / shuffles bit-exact."""
import os

import numpy as np
import pytest
import torch

from oracle import moco_oracle as O
from tests.helpers import load_contrast_golden, oracle_head_chunked, rand_unit

pytestmark = pytest.mark.gpu

LOGIT_RTOL = 1e-3          # north_star tolerance
TIGHT = 2e-5               # what identical bf16 inputs + fp32 accumulation actually give


def _flags():
    from moco_b200 import _lib
    TP = _lib.NCE_TWO_PASS
    return {"auto": _lib.NCE_AUTO, "simt": _lib.NCE_FORCE_SIMT, "tc1": _lib.NCE_SINGLE_CTA,
            # one sweep for loss + dq (what AUTO picks at MoCo temperatures) vs statistics pass + dq pass
            "onepass": _lib.NCE_SINGLE_CTA | _lib.NCE_ONE_PASS, "twopass": _lib.NCE_SINGLE_CTA | TP,
            # CTA-pair statistics kernel (the one round-1 alternative that measured faster; the losers were removed)
            "tc2": _lib.NCE_CTA_PAIR | TP}


@pytest.fixture(scope="module")
def contrast_golden(golden_dir):
    return load_contrast_golden(golden_dir)


def test_library_is_the_cuda_one():
    from moco_b200 import _lib
    lib = _lib.load()
    import ctypes
    sm, major = ctypes.c_int(), ctypes.c_int()
    assert lib.moco_device_info(ctypes.byref(sm), ctypes.byref(major), None) == 0
    assert major.value == 10 and sm.value >= 100, "expected a Blackwell (sm_100) device"


@pytest.mark.parametrize("flag", ["auto", "simt", "tc1", "tc2"])
@pytest.mark.parametrize("name", ["c1head", "wrap", "c256", "ragged"])
def test_golden_dense_api(contrast_golden, name, flag):
    """Unchanged reference call-site (train.py:262-264,273): contrast(q,k,k_all) -> criterion(out)
    -> backward, step after step, vs. the reference's own outputs."""
    from moco_b200.NCE import MemoryMoCo, NCESoftmaxLoss, fused_prob
    g = contrast_golden
    N, C, K, A, steps = (int(v) for v in g[f"{name}_meta"])
    T = float(g[f"{name}_T"][0])
    mod = MemoryMoCo(C, K, T)
    assert sorted(mod.state_dict().keys()) == ["memory", "params"]
    mod.memory.copy_(torch.from_numpy(g[f"{name}_memory0"]))
    mod = mod.cuda()
    mod.kernel_flags = _flags()[flag]
    crit = NCESoftmaxLoss().cuda()
    for s in range(steps):
        q = torch.from_numpy(g[f"{name}_s{s}_q"]).cuda().requires_grad_(True)
        k = torch.from_numpy(g[f"{name}_s{s}_k"]).cuda()
        k_all = torch.from_numpy(g[f"{name}_s{s}_k_all"]).cuda()
        assert mod.index == int(g[f"{name}_s{s}_index"][0])
        out = mod(q, k, k_all)
        ref = g[f"{name}_s{s}_logits"]
        assert out.shape == (N, K + 1) and out.dtype == torch.float32 and out.is_contiguous()
        err = np.abs(out.detach().cpu().numpy() - ref).max() / np.abs(ref).max()
        assert err < TIGHT < LOGIT_RTOL, err
        loss = crit(out)
        assert abs(float(loss) - float(g[f"{name}_s{s}_loss"][0])) < 1e-4
        assert abs(float(fused_prob(out)) - float(g[f"{name}_s{s}_prob"][0])) < 1e-5
        # the generic definitions on the dense logits agree with the fused scalars
        assert abs(float(torch.softmax(out, 1)[:, 0].mean()) - float(g[f"{name}_s{s}_prob"][0])) < 1e-5
        loss.backward()
        dq_ref = g[f"{name}_s{s}_dq"]
        dq_err = np.abs(q.grad.cpu().numpy() - dq_ref).max() / np.abs(dq_ref).max()
        assert dq_err < 5e-3, dq_err          # P is rounded to bf16 before the P.Queue MMA
        assert mod.index == int(g[f"{name}_s{s}_index"][1])
    # FIFO contents bit-exact (Contrast.py:32-34), including the mid-batch wrap of "wrap"
    np.testing.assert_array_equal(mod.memory.cpu().numpy(), g[f"{name}_memory_final"])
    np.testing.assert_array_equal(mod.memory_bf16.float().cpu().numpy(), g[f"{name}_memory_final"])


@pytest.mark.parametrize("name", ["c1head", "c256"])
def test_golden_dense_backward_through_logits(contrast_golden, name):
    """Autograd through the dense `out` itself (arbitrary upstream gradient), not via the fused loss."""
    from moco_b200.NCE import MemoryMoCo
    g = contrast_golden
    N, C, K, A, steps = (int(v) for v in g[f"{name}_meta"])
    T = float(g[f"{name}_T"][0])
    mod = MemoryMoCo(C, K, T)
    mod.memory.copy_(torch.from_numpy(g[f"{name}_memory0"]))
    mod = mod.cuda()
    q = torch.from_numpy(g[f"{name}_s0_q"]).cuda().requires_grad_(True)
    k = torch.from_numpy(g[f"{name}_s0_k"]).cuda()
    out = mod(q, k, torch.from_numpy(g[f"{name}_s0_k_all"]).cuda())
    out = out * 1.0                                   # drops the fused attachment
    loss = torch.nn.functional.cross_entropy(out, torch.zeros(N, dtype=torch.long, device="cuda"))
    loss.backward()
    dq_ref = g[f"{name}_s0_dq"]
    assert np.abs(q.grad.cpu().numpy() - dq_ref).max() / np.abs(dq_ref).max() < 1e-4


CASES = {
    # BASELINE.json configs (head shapes): name -> (N, C, K, T)
    "c1": (32, 128, 1024, 0.07),
    "c2": (256, 128, 16384, 0.07),
    "c3": (256, 128, 65536, 0.07),
    "c4_shard": (2048, 128, 16384, 0.07),     # all 2048 queries x one 16384-row shard
    "c5": (512, 256, 262144, 0.07),
    "ragged": (130, 192, 1000, 0.2),
    "k126689": (128, 128, 126689, 0.1),       # scripts/...sh:12 queue length (not a multiple of anything)
    "tiny": (1, 64, 1, 0.07),
}


@pytest.mark.parametrize("flag,case", [(f, c) for c in CASES for f in ("tc1", "twopass", "tc2")] +
                         [("onepass", "c3"), ("onepass", "k126689"), ("auto", "c2"), ("auto", "ragged")])
def test_fused_vs_oracle(case, flag):
    from moco_b200.NCE import MemoryMoCo
    N, C, K, T = CASES[case]
    rng = np.random.default_rng(hash(case) % 2**31 if False else sum(map(ord, case)))
    q, k = rand_unit(rng, N, C), rand_unit(rng, N, C)
    memory = O.bf16_round((rng.random((K, C), dtype=np.float32) * 2 - 1) * O.queue_init_bound(C)) \
        if case in ("c1", "tiny") else rand_unit(rng, K, C)
    lse, loss, prob, dq = oracle_head_chunked(q, k, memory, T)
    mod = MemoryMoCo(C, K, T)
    mod.memory.copy_(torch.from_numpy(memory))
    mod = mod.cuda()
    mod.kernel_flags = _flags()[flag]
    qt = torch.from_numpy(q).cuda().requires_grad_(True)
    kt = torch.from_numpy(k).cuda()
    k_all = kt[: min(N, K)]
    l, p = mod.forward_loss(qt, kt, k_all)
    assert abs(float(l) - loss) < 2e-4 * max(1.0, abs(loss)), (float(l), loss)
    assert abs(float(p) - prob) < 1e-3 * prob + 1e-9
    lse_gpu = mod._scratch[(N, C, K, qt.device)].lse.cpu().numpy()
    assert np.abs(lse_gpu - lse).max() < 2e-4
    l.backward()
    err = np.abs(qt.grad.cpu().numpy() - dq).max() / np.abs(dq).max()
    assert err < 5e-3, err
    # enqueue happened after the logits were taken (S2) and in order (S3/S4)
    assert mod.index == min(N, K) % K
    exp = memory.copy()
    exp[O.enqueue_ids(0, min(N, K), K)] = k[: min(N, K)]
    np.testing.assert_array_equal(mod.memory.cpu().numpy(), exp)


def _head_gpu(q, k, memory, T, flags):
    from moco_b200.NCE import MemoryMoCo
    N, C = q.shape
    mod = MemoryMoCo(C, memory.shape[0], T)
    mod.memory.copy_(torch.from_numpy(memory))
    mod = mod.cuda()
    mod.kernel_flags = flags
    qt = torch.from_numpy(q).cuda().requires_grad_(True)
    kt = torch.from_numpy(k).cuda()
    l, p = mod.forward_loss(qt, kt, kt)
    l.backward()
    return float(l), float(p), qt.grad.cpu().numpy()


@pytest.mark.parametrize("flag", ["auto", "onepass", "twopass"])
def test_low_temperature_both_sweeps(flag):
    """T = 0.03 (1/T > MOCO_ONE_PASS_MAX_INV_T): AUTO takes the two-pass kernels; the one-pass kernel, forced, is
    still exact for unit-norm features (logit span 2/T = 67 nats < 88)."""
    from moco_b200 import _lib
    rng = np.random.default_rng(11)
    N, C, K, T = 96, 128, 5000, 0.03
    q, k, memory = rand_unit(rng, N, C), rand_unit(rng, N, C), rand_unit(rng, K, C)
    memory[777] = q[5]                                   # a logit at +1/T far from the first tile
    memory[4999] = -q[6]                                 # and one at -1/T
    lse, loss, prob, dq = oracle_head_chunked(q, k, memory, T)
    before = _lib.launches
    l, p, g = _head_gpu(q, k, memory, T, _flags()[flag])
    n_launch = _lib.launches - before - 1                # minus f32->bf16 of the queue
    # one sweep: the tcgen05 kernel + ONE tail kernel that also enqueues; two-pass: prep, stats, combine, dq,
    # dq_reduce + the enqueue kernel
    assert n_launch == (2 if flag == "onepass" else 6), n_launch
    assert abs(l - loss) < 2e-4 * max(1.0, abs(loss)), (l, loss)
    assert abs(p - prob) < 1e-3 * prob + 1e-9
    assert np.abs(g - dq).max() / np.abs(dq).max() < 5e-3


@pytest.mark.parametrize("flag", ["onepass", "twopass"])
def test_unnormalised_inputs_stay_exact(flag):
    """Un-normalised q (norm 12) with its exact direction queued in the LAST tile of a queue long enough that every
    CTA sweeps >= 2 tiles: that logit exceeds its CTA's first-tile maximum by > 127 binades, which the one-sweep
    kernel cannot represent (its partial sum overflows).  The tail kernel detects such rows and recomputes them
    exactly on CUDA cores, so the drop-in never diverges from the reference (which returns a finite loss for any q);
    the two-pass kernels are exact by construction."""
    rng = np.random.default_rng(12)
    N, C, K, T = 64, 128, 2 * 160 * 128, 0.07
    q, k, memory = rand_unit(rng, N, C), rand_unit(rng, N, C), rand_unit(rng, K, C)
    q = O.bf16_round(q * 12.0)
    memory[K - 7] = O.bf16_round(q[3] / 12.0)
    lse, loss, prob, dq = oracle_head_chunked(q, k, memory, T)
    l, p, g = _head_gpu(q, k, memory, T, _flags()[flag])
    assert np.isfinite(l) and abs(l - loss) < 2e-4 * max(1.0, abs(loss)), (l, loss)
    assert abs(p - prob) < 1e-3 * prob + 1e-9
    assert np.isfinite(g).all() and np.abs(g - dq).max() / np.abs(dq).max() < 5e-3


@pytest.mark.parametrize("name", ["n128", "n64"])
def test_fused_normalize_matches_reference_and_oracle(golden_dir, name):
    """SURVEY 8 f2: raw encoder outputs in, L2 normalisation (resnet.py:24-33) inside the head's kernels -- forward for
    q, k and the enqueued keys, backward for q.  Against the reference's own Normalize + MemoryMoCo + autograd
    (tests/golden/normalize.npz; bf16 operand quantisation bounds the difference) and tightly against the oracle
    with the kernels' operand contract."""
    from moco_b200 import _lib
    from moco_b200.NCE import MemoryMoCo
    g = np.load(os.path.join(golden_dir, "normalize.npz"))
    N, C, K, A = (int(v) for v in g[f"{name}_meta"])
    T = float(g[f"{name}_T"][0])
    mod = MemoryMoCo(C, K, T)
    mod.memory.copy_(torch.from_numpy(g[f"{name}_memory0"]))
    mod = mod.cuda()
    xq = torch.from_numpy(g[f"{name}_xq"]).cuda().requires_grad_(True)
    before = _lib.launches
    loss, prob = mod.forward_loss(xq, torch.from_numpy(g[f"{name}_xk"]).cuda(), torch.from_numpy(g[f"{name}_xk_all"]).cuda(),
                                  normalize=True)
    assert _lib.launches - before == 3                     # f32->bf16 of the fresh queue + sweep + tail: no torch normalise
    loss.backward()
    got = xq.grad.cpu().numpy()
    # vs the reference itself
    ref = g[f"{name}_dxq"]
    assert abs(float(loss) - float(g[f"{name}_loss"][0])) < 5e-3
    assert abs(float(prob) - float(g[f"{name}_prob"][0])) < 5e-3 * float(g[f"{name}_prob"][0]) + 1e-6
    assert np.abs(got - ref).max() / np.abs(ref).max() < 2e-2
    # vs the oracle under the kernels' operand contract: tight
    l2, p2, d2, _, _ = O.head_with_normalize(g[f"{name}_xq"], g[f"{name}_xk"], g[f"{name}_memory0"], T, True)
    assert abs(float(loss) - l2) < 2e-4 and abs(float(prob) - p2) < 1e-3 * p2
    assert np.abs(got - d2).max() / np.abs(d2).max() < 5e-3
    # the enqueued rows are the NORMALISED keys: fp32 master within an ulp of the reference's, ring position advanced
    np.testing.assert_allclose(mod.memory.cpu().numpy(), g[f"{name}_memory_final"], rtol=0, atol=2e-7)
    assert mod.index == A % K


def test_device_side_ring_index_survives_graph_replay():
    """SURVEY 8 f2 / Contrast.py:12,32-34: with the ring position in a Python int a captured step would replay the same
    slots forever; MemoryMoCo(device_index=True) keeps it on the device, advanced by the tail kernel."""
    from moco_b200.NCE import MemoryMoCo
    from moco_b200.NCE.Contrast import _nce_forward
    rng = np.random.default_rng(21)
    N, C, K, T = 64, 128, 320, 0.07                       # K not a multiple of the batch: wraps on the 5th replay
    memory = rand_unit(rng, K, C)
    mods = []
    for dev_index in (False, True):
        m = MemoryMoCo(C, K, T, device_index=dev_index)
        m.memory.copy_(torch.from_numpy(memory))
        mods.append(m.cuda())
    eager, graphed = mods
    sq, sk = torch.zeros(N, C, device="cuda"), torch.zeros(N, C, device="cuda")
    graphed._queue_bf16(); graphed._index_dev()
    _nce_forward(graphed, sq, sk, False, True, graphed.kernel_flags, k_all=sk)     # eager warm-up (enqueues zeros)
    graphed.memory.copy_(torch.from_numpy(memory).cuda()); graphed._invalidate(); graphed._queue_bf16()
    graphed.index = 0
    graphed._index_dev()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _, loss_prob, dq, _, _ = _nce_forward(graphed, sq, sk, False, True, graphed.kernel_flags, k_all=sk)
    graphed.index = 0
    graphed._index_shadow = 0
    for step in range(7):
        q, k = rand_unit(rng, N, C), rand_unit(rng, N, C)
        qt = torch.from_numpy(q).cuda().requires_grad_(True)
        l, p = eager.forward_loss(qt, torch.from_numpy(k).cuda(), torch.from_numpy(k).cuda())
        l.backward()
        sq.copy_(torch.from_numpy(q)); sk.copy_(torch.from_numpy(k))
        g.replay()
        assert float(loss_prob[0]) == float(l) and float(loss_prob[1]) == float(p), step
        assert torch.equal(dq.to(qt.grad.dtype), qt.grad), step
    torch.cuda.synchronize()
    assert torch.equal(graphed.memory, eager.memory)
    assert graphed.sync_index() == eager.index == (7 * N) % K


def test_fp32_inputs_are_rounded_to_bf16_exactly_once():
    """Arbitrary fp32 (not bf16-representable) q/k/queue.  The kernel's contract (include/moco_b200.h):
    negatives = <bf16(q), bf16(queue)> with fp32 accumulation, positive = <q, k> in fp32.  Against the
    oracle fed the same rounded operands the logits are tight (north_star: 1e-3 relative on identical
    inputs); against the un-rounded fp32 oracle the only difference is the bf16 operand quantisation
    (2^-9 per element), bounded here and quantified in DESIGN.md."""
    from moco_b200.NCE import MemoryMoCo
    rng = np.random.default_rng(5)
    N, C, K, T = 64, 128, 4096, 0.07
    q = O.l2_normalize(rng.standard_normal((N, C)).astype(np.float32))
    k = O.l2_normalize(rng.standard_normal((N, C)).astype(np.float32))
    memory = O.l2_normalize(rng.standard_normal((K, C)).astype(np.float32))
    ref = O.MemoryMoCoOracle(memory, T).logits(q, k)
    ref_rounded = O.MemoryMoCoOracle(O.bf16_round(memory), T).logits(O.bf16_round(q), k)
    mod = MemoryMoCo(C, K, T)
    mod.memory.copy_(torch.from_numpy(memory))
    mod = mod.cuda()
    out = mod(torch.from_numpy(q).cuda(), torch.from_numpy(k).cuda(), torch.from_numpy(k).cuda())
    got = out.cpu().numpy()
    err_same_inputs = np.abs(got[:, 1:] - ref_rounded[:, 1:]).max() / np.abs(ref_rounded).max()
    assert err_same_inputs < TIGHT < LOGIT_RTOL, err_same_inputs
    err_vs_fp32 = np.abs(got - ref).max() / np.abs(ref).max()
    assert err_vs_fp32 < 5e-3, err_vs_fp32            # bf16 operand quantisation (measured ~2.3e-3 of max|logit|)
    # the positive logit is computed in fp32 from the fp32 inputs: tight against the fp32 oracle
    assert np.abs(got[:, 0] - ref[:, 0]).max() < 1e-4
    # the fp32 master queue keeps the exact fp32 keys, the working copy their bf16 rounding
    np.testing.assert_array_equal(mod.memory[:N].cpu().numpy(), k)
    np.testing.assert_array_equal(mod.memory_bf16[:N].float().cpu().numpy(), O.bf16_round(k))


def test_bf16_inputs_accepted():
    from moco_b200.NCE import MemoryMoCo
    rng = np.random.default_rng(6)
    N, C, K, T = 128, 128, 2048, 0.07
    q, k, memory = rand_unit(rng, N, C), rand_unit(rng, N, C), rand_unit(rng, K, C)
    _, loss, prob, _ = oracle_head_chunked(q, k, memory, T, want_dq=False)
    mod = MemoryMoCo(C, K, T)
    mod.memory.copy_(torch.from_numpy(memory))
    mod = mod.cuda()
    l, p = mod.forward_loss(torch.from_numpy(q).cuda().bfloat16(), torch.from_numpy(k).cuda().bfloat16(),
                            torch.from_numpy(k).cuda().bfloat16())
    assert abs(float(l) - loss) < 2e-4 and abs(float(p) - prob) < 1e-3 * prob


def test_deterministic_and_no_state_leak():
    from moco_b200.NCE import MemoryMoCo
    rng = np.random.default_rng(7)
    N, C, K, T = 256, 128, 16384, 0.07
    q, k, memory = rand_unit(rng, N, C), rand_unit(rng, N, C), rand_unit(rng, K, C)
    outs = []
    for _ in range(3):
        mod = MemoryMoCo(C, K, T)
        mod.memory.copy_(torch.from_numpy(memory))
        mod = mod.cuda()
        qt = torch.from_numpy(q).cuda().requires_grad_(True)
        l, p = mod.forward_loss(qt, torch.from_numpy(k).cuda(), torch.from_numpy(k).cuda())
        l.backward()
        outs.append((float(l), float(p), qt.grad.cpu().numpy().copy()))
    for o in outs[1:]:
        assert o[0] == outs[0][0] and o[1] == outs[0][1]
        np.testing.assert_array_equal(o[2], outs[0][2])


@pytest.mark.parametrize("K,C,n_all,index", [(40, 64, 16, 32), (126689, 128, 1024, 126000), (65536, 128, 2048, 0),
                                             (1000, 100, 10, 995), (8, 64, 8, 3)])
def test_enqueue_ring_bit_exact(K, C, n_all, index):
    from moco_b200.NCE import MemoryMoCo
    rng = np.random.default_rng(K + n_all)
    memory = rng.standard_normal((K, C)).astype(np.float32)
    orc = O.MemoryMoCoOracle(memory, 0.07, index=index)
    mod = MemoryMoCo(C, K, 0.07)
    mod.memory.copy_(torch.from_numpy(memory))
    mod = mod.cuda()
    mod.index = index
    for step in range(3):
        k_all = rng.standard_normal((n_all, C)).astype(np.float32)
        ids = orc.enqueue(k_all)
        np.testing.assert_array_equal(ids, (np.arange(n_all) + (index + step * n_all) % K) % K)
        mod.enqueue(torch.from_numpy(k_all).cuda())
        assert mod.index == orc.index
    np.testing.assert_array_equal(mod.memory.cpu().numpy(), orc.memory)
    np.testing.assert_array_equal(mod._queue_bf16().float().cpu().numpy(), O.bf16_round(orc.memory))


def test_enqueue_rejects_oversized_batch():
    from moco_b200.NCE import MemoryMoCo
    mod = MemoryMoCo(64, 8, 0.07).cuda()
    with pytest.raises(RuntimeError, match="n_all"):
        mod.enqueue(torch.zeros(9, 64, device="cuda"))


def test_state_dict_roundtrip_reference_format():
    from moco_b200.NCE import MemoryMoCo
    a = MemoryMoCo(128, 256, 0.07).cuda()
    a.enqueue(torch.nn.functional.normalize(torch.randn(32, 128, device="cuda"), dim=1))
    sd = {k: v.cpu() for k, v in a.state_dict().items()}
    assert sorted(sd) == ["memory", "params"] and sd["memory"].dtype == torch.float32
    assert sd["params"].tolist() == [-1]
    b = MemoryMoCo(128, 256, 0.07).cuda()
    b.load_state_dict(sd)
    assert b.index == 0                                  # the reference does not checkpoint `index` (SURVEY §5)
    np.testing.assert_array_equal(b.memory.cpu().numpy(), sd["memory"].numpy())
    np.testing.assert_array_equal(b._queue_bf16().float().cpu().numpy(), O.bf16_round(sd["memory"].numpy()))


def test_shufflebn_single_rank_roundtrip(golden_dir):
    """W = 1: the reference still permutes within the batch (SURVEY §8e)."""
    from moco_b200.util import DistributedShufle
    g = np.load(os.path.join(golden_dir, "shuffle.npz"))
    x = torch.from_numpy(g["w1_n8_e3_r0_x"]).cuda()
    xs, binds = DistributedShufle.forward_shuffle(x, 3)
    np.testing.assert_array_equal(xs.cpu().numpy(), g["w1_n8_e3_r0_x_shuf"])
    np.testing.assert_array_equal(binds.cpu().numpy(), g["w1_n8_e3_r0_binds"])
    assert binds.dtype == torch.int64 and binds.is_cuda
    feat = torch.from_numpy(g["w1_n8_e3_r0_feat"]).cuda()
    f_all, f_loc = DistributedShufle.backward_shuffle(feat, binds, return_local=True)
    np.testing.assert_array_equal(f_all.cpu().numpy(), g["w1_n8_e3_r0_feat_all"])
    np.testing.assert_array_equal(f_loc.cpu().numpy(), g["w1_n8_e3_r0_feat_local"])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_shufflebn_full_size_images_roundtrip(dtype):
    """BASELINE batch (256 x 3 x 224 x 224) through the bulk-async gather; properties: it is the oracle's
    permutation, and backward(forward(x)) == x."""
    from moco_b200.util import DistributedShufle
    n, epoch = 256, 11
    x = torch.randn(n, 3, 224, 224, device="cuda").to(dtype)
    xs, binds = DistributedShufle.forward_shuffle(x, epoch)
    fwd, bwd = O.get_shuffle_ids(n, epoch)
    np.testing.assert_array_equal(binds.cpu().numpy(), bwd)
    assert torch.equal(xs, x[torch.from_numpy(fwd).cuda()])
    back = DistributedShufle.backward_shuffle(xs, binds, return_local=False)
    assert torch.equal(back, x)


@pytest.mark.parametrize("mode", ["auto_one_pass", "two_pass"])
def test_sharded_queue_world1_matches_oracle(mode):
    """ShardedMemoryMoCo at world_size 1 (one shard == the whole ring): same loss / prob / dq / FIFO as the
    reference's replicated MemoryMoCo, with the one-sweep shard kernel (default at T = 0.07) and the two-pass
    kernels.  (world_size > 1: tests/test_gpu_multi.py.)"""
    from moco_b200 import _lib
    from moco_b200.NCE import ShardedMemoryMoCo
    rng = np.random.default_rng(11)
    N, C, K, T = 64, 128, 4096 + 77, 0.07
    mem = rand_unit(rng, K, C)
    mod = ShardedMemoryMoCo(C, K, T)
    mod.memory.copy_(torch.from_numpy(mem))
    mod = mod.cuda()
    if mode == "two_pass":
        mod.kernel_flags = _lib.NCE_TWO_PASS
    orc = O.MemoryMoCoOracle(mem, T)
    for _ in range(3):
        q, k = rand_unit(rng, N, C), rand_unit(rng, N, C)
        pre = orc.memory.copy()
        out = orc.logits(q, k)
        dq = O.nce_backward_dq(q, k, pre, T)
        orc.enqueue(k)
        qt = torch.from_numpy(q).cuda().requires_grad_(True)
        loss, prob = mod.forward_loss(qt, torch.from_numpy(k).cuda(), torch.from_numpy(k).cuda())
        loss.backward()
        assert abs(float(loss) - O.nce_softmax_loss(out)) < 2e-4
        assert abs(float(prob) - O.prob_metric(out)) < 1e-3 * O.prob_metric(out)
        assert np.abs(qt.grad.cpu().numpy() - dq).max() / np.abs(dq).max() < 5e-3
        assert mod.index == orc.index
    np.testing.assert_array_equal(mod.full_memory().cpu().numpy(), orc.memory)


@pytest.mark.parametrize("W", [2, 8])
def test_enqueue_shard_windows_reassemble_the_ring(W):
    """moco_queue_enqueue_shard on W disjoint row windows == the reference's index_copy_ on the full ring
    (ring slot g -> rank g // (K/W), local row g % (K/W)); bit-exact incl. a wrap across the last/first shard."""
    from moco_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(W)
    K, C, n_all = 1024, 64, 96
    rows = K // W
    mem = rng.standard_normal((K, C)).astype(np.float32)
    orc = O.MemoryMoCoOracle(mem, 0.07, index=K - 40)
    shards_f = [torch.from_numpy(mem[r * rows:(r + 1) * rows].copy()).cuda() for r in range(W)]
    shards_b = [s.bfloat16() for s in shards_f]
    index = K - 40
    for _ in range(3):
        k_all = rng.standard_normal((n_all, C)).astype(np.float32)
        orc.enqueue(k_all)
        kt = torch.from_numpy(k_all).cuda()
        for r in range(W):
            rc = lib.moco_queue_enqueue_shard(shards_b[r].data_ptr(), shards_f[r].data_ptr(), kt.data_ptr(), 0, n_all, C,
                                              K, index, r * rows, rows, torch.cuda.current_stream().cuda_stream)
            assert rc == 0
        index = (index + n_all) % K
    np.testing.assert_array_equal(torch.cat(shards_f).cpu().numpy(), orc.memory)
    np.testing.assert_array_equal(torch.cat(shards_b).float().cpu().numpy(), O.bf16_round(orc.memory))


def test_cpu_tensors_fail_loudly():
    from moco_b200.NCE import MemoryMoCo
    mod = MemoryMoCo(64, 32, 0.07)          # never moved to CUDA
    with pytest.raises(RuntimeError, match="CUDA"):
        mod(torch.randn(4, 64), torch.randn(4, 64), torch.randn(4, 64))


def test_full_step_matches_cpu_reference_step():
    """One whole MoCo iteration (train.py:244-283) -- ShuffleBN permute, both encoders, head, backward, SGD,
    EMA, enqueue -- through MoCoStep on the GPU in fp32 vs. the CPU port of the reference step
    (oracle/cpu_step.py) from identical weights, queue and images.  Two steps, so the second one sees the
    enqueued keys and the updated encoders.  fp32 convs on GPU (cuDNN/TF32 off) vs CPU: loose tolerances."""
    from moco_b200 import encoders
    from moco_b200.NCE import MemoryMoCo
    from moco_b200.train_step import MoCoStep
    from oracle.cpu_step import CpuMoCoStep
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        N, C, K, T = 8, 128, 256, 0.07
        cpu = CpuMoCoStep("resnet18", C, K, T, batch=N, seed=0)
        # GPU twin from the same weights / queue (bf16-representable queue so both heads see the same negatives)
        cpu.contrast.memory[:] = O.bf16_round(cpu.contrast.memory)
        model = encoders.resnet18(low_dim=C)
        model.load_state_dict(cpu.model.state_dict())
        model_ema = encoders.resnet18(low_dim=C)
        model_ema.load_state_dict(cpu.model_ema.state_dict())
        contrast = MemoryMoCo(C, K, T)
        contrast.memory.copy_(torch.from_numpy(cpu.contrast.memory))
        model, model_ema, contrast = model.cuda(), model_ema.cuda(), contrast.cuda()
        opt = torch.optim.SGD(model.parameters(), lr=0.03 * N / 256, momentum=0.9, weight_decay=1e-4)
        step = MoCoStep(model, model_ema, contrast, opt, alpha=0.999, amp_dtype=None, overlap_shuffle=True)
        g = torch.Generator().manual_seed(5)
        for it in range(2):
            inputs = torch.randn(N, 6, 224, 224, generator=g)
            ref_loss, ref_prob = cpu.step(inputs, epoch=3)
            x1, x2 = torch.split(inputs.cuda(), [3, 3], dim=1)
            loss, prob = step(x1.contiguous(), x2.contiguous(), 3)
            assert abs(float(loss) - ref_loss) < 5e-3 * max(1.0, abs(ref_loss)), (it, float(loss), ref_loss)
            assert abs(float(prob) - ref_prob) < 2e-2 * ref_prob + 1e-6, (it, float(prob), ref_prob)
            assert contrast.index == cpu.contrast.index
        # the queue now holds the same keys in the same ring slots (bf16 working copy ~ fp32 keys)
        np.testing.assert_allclose(contrast.memory.cpu().numpy(), cpu.contrast.memory, atol=2e-3)
        # EMA encoder followed the same trajectory
        w_gpu = next(model_ema.parameters()).detach().cpu().numpy()
        w_cpu = next(cpu.model_ema.parameters()).detach().numpy()
        np.testing.assert_allclose(w_gpu, w_cpu, atol=1e-4)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


def test_nce_fwd_is_cuda_graph_capturable():
    """include/moco_b200.h promises the compute calls are CUDA-graph capturable: capture moco_nce_fwd (stats +
    combine + dq + dq_reduce), change q in place, replay, and compare with a direct call on the new q."""
    from moco_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(21)
    N, C, K, T = 256, 128, 16384, 0.07
    dev = torch.device("cuda")
    q = torch.from_numpy(rand_unit(rng, N, C)).to(dev).bfloat16()
    k = torch.from_numpy(rand_unit(rng, N, C)).to(dev).bfloat16()
    queue = torch.from_numpy(rand_unit(rng, K, C)).to(dev).bfloat16()
    f32 = dict(dtype=torch.float32, device=dev)

    def bufs():
        return dict(lse=torch.zeros(N, **f32), lr=torch.zeros(N, **f32), pr=torch.zeros(N, **f32),
                    lp=torch.zeros(2, **f32), dq=torch.zeros(N, C, **f32))
    wsb = lib.moco_nce_workspace_bytes(N, C, K)
    ws = torch.zeros(wsb + 256, dtype=torch.uint8, device=dev)
    wp = ws.data_ptr() + (-ws.data_ptr()) % 256

    def call(b):
        rc = lib.moco_nce_fwd(q.data_ptr(), k.data_ptr(), 1, queue.data_ptr(), N, C, K, 1.0 / T, None, b["lse"].data_ptr(),
                              b["lr"].data_ptr(), b["pr"].data_ptr(), b["lp"].data_ptr(), b["dq"].data_ptr(), wp, wsb, 0,
                              torch.cuda.current_stream().cuda_stream)
        assert rc == 0, lib.moco_last_error()
    a = bufs()
    call(a)                                   # first call outside capture (one-time kernel attribute setup)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        call(a)
    q.copy_(torch.from_numpy(rand_unit(rng, N, C)).to(dev).bfloat16())
    g.replay()
    torch.cuda.synchronize()
    b = bufs()
    call(b)
    torch.cuda.synchronize()
    for key in ("lse", "lr", "pr", "lp", "dq"):
        assert torch.equal(a[key], b[key]), key


# ------------------------------------------------------------------ EMA (moment_update, util.py:124-127)
@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["m999", "m99", "m0"])
def test_moment_update_matches_reference_bit_exact(golden_dir, tag):
    """moco_ema_update on the reference's own inputs: fp32 bit patterns of every EMA parameter after every step."""
    from moco_b200 import _lib
    from moco_b200.util import moment_update
    z = np.load(os.path.join(golden_dir, "ema.npz"))
    n, m = int(z[f"{tag}_n"][0]), float(z[f"{tag}_m"][0])

    class Bag(torch.nn.Module):
        def __init__(self, arrs):
            super().__init__()
            self.ps = torch.nn.ParameterList([torch.nn.Parameter(torch.from_numpy(a.copy())) for a in arrs])
    ema = Bag([z[f"{tag}_ema0_{i}"] for i in range(n)]).cuda()
    model = Bag([z[f"{tag}_s0_p_{i}"] for i in range(n)]).cuda()
    for s in range(int(z[f"{tag}_steps"][0])):
        with torch.no_grad():
            for i, p in enumerate(model.parameters()):
                p.copy_(torch.from_numpy(z[f"{tag}_s{s}_p_{i}"]))
        before = _lib.launches
        moment_update(model, ema, m)
        assert _lib.launches == before + 1                       # one launch for all tensors
        for i, p in enumerate(ema.parameters()):
            got = p.detach().cpu().numpy()
            np.testing.assert_array_equal(got.view(np.uint32), z[f"{tag}_s{s}_ema_{i}"].view(np.uint32))


@pytest.mark.gpu
def test_moment_update_resnet50_unaligned_and_vs_oracle():
    """Full-size (ResNet-50, 23.8 M parameters) EMA against the oracle, plus views at 4-byte-aligned offsets."""
    from moco_b200 import encoders
    from moco_b200.util import moment_update
    torch.manual_seed(5)
    model, ema = encoders.resnet50(low_dim=128).cuda(), encoders.resnet50(low_dim=128).cuda()
    p0 = [p.detach().cpu().numpy() for p in model.parameters()]
    e0 = [p.detach().cpu().numpy() for p in ema.parameters()]
    moment_update(model, ema, 0.999)
    want = O.moment_update(p0, e0, 0.999)
    for w, p in zip(want, ema.parameters()):
        np.testing.assert_array_equal(p.detach().cpu().numpy().view(np.uint32), w.view(np.uint32))
    for a, b in zip(p0, model.parameters()):                      # the query encoder is read-only
        np.testing.assert_array_equal(a, b.detach().cpu().numpy())

    # misaligned storage offsets (scalar path) and a tail shorter than one vector
    class Views(torch.nn.Module):
        def __init__(self, flat, sizes, off):
            super().__init__()
            self._flat = flat
            self._views = []
            for n in sizes:
                self._views.append(flat[off:off + n])
                off += n + 1
        def parameters(self, recurse=True):
            return iter(self._views)
    sizes = [1, 3, 8191, 8193, 20001]
    fa, fb = torch.randn(40000, device="cuda"), torch.randn(40000, device="cuda")
    ref_b = fb.clone()
    va, vb = Views(fa, sizes, 1), Views(fb, sizes, 3)
    want = O.moment_update([v.cpu().numpy() for v in va.parameters()], [v.cpu().numpy() for v in vb.parameters()], 0.99)
    moment_update(va, vb, 0.99)
    touched = torch.zeros(40000, dtype=torch.bool)
    off = 3
    for n, w, v in zip(sizes, want, vb.parameters()):
        np.testing.assert_array_equal(v.cpu().numpy().view(np.uint32), w.view(np.uint32))
        touched[off:off + n] = True
        off += n + 1
    assert torch.equal(fb.cpu()[~touched], ref_b.cpu()[~touched])     # nothing outside the views was written


@pytest.mark.gpu
def test_moment_update_channels_last_parameters():
    """bench.py / MoCoStep keep the encoders in channels_last: conv weights are dense but not default-contiguous."""
    from moco_b200 import encoders
    from moco_b200.util import moment_update
    torch.manual_seed(6)
    model = encoders.resnet18(low_dim=128).cuda().to(memory_format=torch.channels_last)
    ema = encoders.resnet18(low_dim=128).cuda().to(memory_format=torch.channels_last)
    assert any(not p.is_contiguous() for p in model.parameters())
    p0 = [p.detach().cpu().numpy() for p in model.parameters()]
    e0 = [p.detach().cpu().numpy() for p in ema.parameters()]
    moment_update(model, ema, 0.999)
    for w, p in zip(O.moment_update(p0, e0, 0.999), ema.parameters()):
        np.testing.assert_array_equal(p.detach().cpu().numpy().view(np.uint32), w.view(np.uint32))
    mixed = encoders.resnet18(low_dim=128).cuda()                 # NCHW vs NHWC strides differ: must refuse
    with pytest.raises(RuntimeError, match="equal strides"):
        moment_update(mixed, ema, 0.999)


# ------------------------------------------------------------------ input path (SURVEY 8 f3)
@pytest.mark.gpu
@pytest.mark.parametrize("src_dtype", [torch.float32, torch.bfloat16])
def test_crop_to_channels_last_bf16_bit_exact(src_dtype):
    """One kernel = crop selection + cast + NCHW->NHWC; bit-identical to torch's cast + layout change."""
    from moco_b200.util import crop_to_channels_last_bf16
    g = torch.Generator(device="cuda").manual_seed(9)
    six = torch.randn(5, 6, 24, 20, device="cuda", generator=g).to(src_dtype)          # H*W = 480, multiple of 8
    for sl in (slice(0, 3), slice(3, 6), slice(2, 3), slice(1, 5)):
        x = six[:, sl]                                                                  # a view: read in place
        got = crop_to_channels_last_bf16(x)
        want = x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        assert got.shape == x.shape and got.dtype == torch.bfloat16
        assert got.is_contiguous(memory_format=torch.channels_last)
        assert torch.equal(got.contiguous().view(torch.int16), want.contiguous().view(torch.int16))
    full = torch.randn(3, 3, 224, 224, device="cuda", generator=g)
    assert torch.equal(crop_to_channels_last_bf16(full),
                       full.to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
    with pytest.raises(ValueError, match="H\\*W"):
        crop_to_channels_last_bf16(torch.randn(2, 3, 5, 5, device="cuda"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        crop_to_channels_last_bf16(torch.randn(2, 3, 8, 8))


@pytest.mark.gpu
def test_forward_shuffle_channels_last_matches_oracle():
    """ShuffleBN forward permute with the fused bf16/NHWC publish (world 1): rows = oracle's permutation of the
    bf16-rounded crop; output is a channels_last tensor; un-shuffle of per-row features restores the order (S6)."""
    from moco_b200.util import DistributedShufle
    g = torch.Generator().manual_seed(21)
    six = torch.randn(16, 6, 16, 16, generator=g)
    for epoch in (1, 2, 7):
        want, bwd = O.forward_shuffle([O.bf16_round(six[:, 3:].numpy())], epoch)
        got, binds = DistributedShufle.forward_shuffle(six.cuda()[:, 3:], epoch, channels_last=True)
        assert got.dtype == torch.bfloat16 and got.is_contiguous(memory_format=torch.channels_last)
        np.testing.assert_array_equal(got.float().cpu().numpy(), want[0])
        np.testing.assert_array_equal(binds.cpu().numpy(), bwd)
        feat = got.float().reshape(16, -1)[:, :32].contiguous()
        _, local = DistributedShufle.backward_shuffle(feat, binds, return_local=True)
        np.testing.assert_array_equal(local.cpu().numpy(), O.bf16_round(six[:, 3:].numpy()).reshape(16, -1)[:, :32])


@pytest.mark.gpu
def test_step_with_fused_input_path_matches_plain_step():
    """MoCoStep(channels_last=True) feeds both encoders bf16 NHWC crops taken in place from the 6-channel batch; the
    plain step lets autocast / cuDNN do the same conversions.  Same values in, same losses out."""
    from moco_b200 import encoders
    from moco_b200.NCE import MemoryMoCo
    from moco_b200.train_step import MoCoStep
    losses = []
    for nhwc in (False, "nhwc", True):             # plain; bf16 NHWC crops; bf16 space-to-depth crops (StemConv's 4x4 form)
        torch.manual_seed(0)
        model = encoders.resnet18(low_dim=128).cuda().to(memory_format=torch.channels_last)
        ema = encoders.resnet18(low_dim=128).cuda().to(memory_format=torch.channels_last)
        ema.load_state_dict(model.state_dict())
        contrast = MemoryMoCo(128, 1024, 0.07).cuda()
        opt = torch.optim.SGD(model.parameters(), lr=0.03, momentum=0.9, weight_decay=1e-4)
        step = MoCoStep(model, ema, contrast, opt, channels_last=nhwc)
        g = torch.Generator(device="cuda").manual_seed(4)
        out = []
        for _ in range(3):
            batch = torch.randn(16, 6, 64, 64, device="cuda", generator=g)
            x1, x2 = torch.split(batch, [3, 3], dim=1)
            if not nhwc:
                x1, x2 = x1.contiguous(memory_format=torch.channels_last), x2.contiguous()
            loss, prob = step(x1, x2, 1)
            out.append((float(loss), float(prob)))
        losses.append(out)
    # identical values enter both encoders; the bound only leaves room for run-to-run cuDNN non-determinism in the
    # two later steps (a wrong crop or layout would move the loss by O(1))
    for (l0, p0), (l1, p1) in zip(losses[0], losses[1]):
        assert abs(l0 - l1) < 1e-2 * max(1.0, abs(l0)), (losses)
        assert abs(p0 - p1) < 5e-2 * max(p0, 1e-6) + 1e-6
    # space-to-depth crops: the first convolution is the same function but another cuDNN kernel (other summation
    # order), so its bf16 outputs differ in the last bit and two SGD steps amplify that
    for (l0, p0), (l2, p2) in zip(losses[0], losses[2]):
        assert abs(l0 - l2) < 3e-2 * max(1.0, abs(l0)), (losses)
        assert abs(p0 - p2) < 0.15 * max(p0, 1e-6) + 1e-6


@pytest.mark.parametrize("graph", [False, True])
def test_step_with_fused_normalize_and_graphed_tail_matches_plain_step(graph):
    """SURVEY 8 f2: MoCoStep(fuse_normalize=True[, graph_tail=True]) takes the encoders' RAW fc outputs, normalises
    inside the head's two kernels (forward for q / k / the enqueued keys, backward for q) and -- graph_tail -- replays
    the whole post-encoder tail from one captured CUDA graph with the ring position on the device.  Same math as the
    plain step (Normalize in torch, eager tail): same losses, same queue, same ring position."""
    from moco_b200 import encoders
    from moco_b200.NCE import MemoryMoCo
    from moco_b200.train_step import MoCoStep
    runs = []
    for fused in (False, True):
        torch.manual_seed(0)
        model = encoders.resnet18(low_dim=128).cuda()
        ema = encoders.resnet18(low_dim=128).cuda()
        ema.load_state_dict(model.state_dict())
        contrast = MemoryMoCo(128, 80, 0.07, device_index=fused and graph).cuda()      # K = 80, 16 keys/step: wraps
        # a small learning rate: the comparison is about the kernels, not about how fast seven SGD steps on a
        # 16-image batch amplify rounding-level differences
        opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4)
        step = MoCoStep(model, ema, contrast, opt, amp_dtype=None, fuse_normalize=fused, graph_tail=fused and graph)
        g = torch.Generator(device="cuda").manual_seed(4)
        out, w_first = [], None
        for it in range(7):
            batch = torch.randn(16, 6, 64, 64, device="cuda", generator=g)
            x1, x2 = torch.split(batch, [3, 3], dim=1)
            loss, prob = step(x1.contiguous(), x2.contiguous(), 1)
            out.append((float(loss), float(prob)))
            if it == 1:          # after the first step the graphed run takes eagerly and the first one it replays
                w_first = model.fc.weight.detach().cpu().numpy().copy()
        torch.cuda.synchronize()
        runs.append((out, contrast.memory.cpu().numpy().copy(), contrast.sync_index() if fused and graph else contrast.index,
                     w_first))
    (o0, m0, i0, w0), (o1, m1, i1, w1) = runs
    assert i0 == i1 == (7 * 16) % 80
    # same values in, same losses out; the later steps only leave room for the amplification of rounding-level
    # differences by seven SGD steps on a tiny batch (a wrong gradient or ring slot moves the loss by O(1))
    for it, ((l0, p0), (l1, p1)) in enumerate(zip(o0, o1)):
        tol = 1e-2 if it < 3 else 3e-2
        assert abs(l0 - l1) < tol * max(1.0, abs(l0)), (it, o0, o1)
        assert abs(p0 - p1) < 5 * tol * max(p0, 1e-6) + 1e-6, (it, o0, o1)
    # the queue holds normalised keys in the same slots; the trained weights followed the same trajectory
    np.testing.assert_allclose(m0, m1, atol=5e-3)
    np.testing.assert_allclose(np.linalg.norm(m1, axis=1), 1.0, atol=1e-3)
    # two SGD steps in, the head's weights (which see the gradient through the normalisation first) still agree
    # closely: the backward of Normalize inside the tail kernel is the one autograd applies in the plain run
    assert np.abs(w0 - w1).max() < 2e-2 * np.abs(w0).max(), np.abs(w0 - w1).max() / np.abs(w0).max()


def test_normalize_falls_back_to_torch_where_the_kernels_do_not_fuse_it():
    """feat_dim 256 runs on nce_head256_kernel, which takes q already normalised: forward_loss(normalize=True)
    then normalises in torch (same definition as resnet.py:30-33) -- same result contract, three more launches."""
    from moco_b200.NCE import MemoryMoCo
    rng = np.random.default_rng(31)
    N, C, K, T = 48, 256, 700, 0.07
    xq = (rng.standard_normal((N, C)) * 2.5).astype(np.float32)
    xk = (rng.standard_normal((N, C)) * 0.7).astype(np.float32)
    memory = rand_unit(rng, K, C)
    loss, prob, dxq, qh, kh = O.head_with_normalize(xq, xk, memory, T, True)
    mod = MemoryMoCo(C, K, T)
    mod.memory.copy_(torch.from_numpy(memory))
    mod = mod.cuda()
    xt = torch.from_numpy(xq).cuda().requires_grad_(True)
    l, p = mod.forward_loss(xt, torch.from_numpy(xk).cuda(), torch.from_numpy(xk).cuda(), normalize=True)
    l.backward()
    assert abs(float(l) - loss) < 2e-4 * max(1.0, abs(loss)) and abs(float(p) - prob) < 1e-3 * prob + 1e-9
    assert np.abs(xt.grad.cpu().numpy() - dxq).max() / np.abs(dxq).max() < 5e-3
    np.testing.assert_allclose(mod.memory[:N].cpu().numpy(), kh, atol=2e-7)


def test_peer_wait_status_block_is_clean_and_standalone_enqueue_keeps_the_device_index():
    from moco_b200.NCE import MemoryMoCo
    from moco_b200.util import ShuffleContext
    assert ShuffleContext.last_timeout() is None
    m = MemoryMoCo(64, 40, 0.07, device_index=True).cuda()
    m.index = 33                                          # host assignment (as the reference allows) is honoured
    keys = torch.nn.functional.normalize(torch.randn(16, 64, device="cuda"), dim=1)
    q = torch.nn.functional.normalize(torch.randn(16, 64, device="cuda"), dim=1).requires_grad_(True)
    m.forward_loss(q, keys, keys)                         # fused step: wraps 33..39, 0..8
    assert m.index == 9 and m.sync_index() == 9
    m.enqueue(keys)                                       # stand-alone enqueue
    assert m.index == 25 and m.sync_index() == 25
    exp = torch.zeros(40, dtype=torch.bool)
    exp[torch.arange(33, 33 + 32) % 40] = True
    got = (m.memory.cpu().norm(dim=1) - 1).abs() < 1e-3  # rows holding unit-norm keys
    init_norms_are_not_one = True
    assert bool((got[exp]).all()) and init_norms_are_not_one
