"""Generate golden fixtures by RUNNING THE UNMODIFIED REFERENCE (bl0/moco).

Run in the build container only (``/root/reference`` does not exist on the
GPU box):

    python tests/golden/gen_golden.py

It imports ``moco.NCE`` / ``moco.util`` read-only from ``/root/reference`` with
the CPU shims SURVEY.md §8c lists (identity ``.cuda()``, gloo instead of nccl;
no reference file is modified or copied), feeds seeded inputs through
``MemoryMoCo`` / ``NCESoftmaxLoss`` / ``DistributedShufle`` and writes the
inputs AND the reference's outputs to ``tests/golden/*.npz``.  The committed
fixtures are what pins ``oracle/moco_oracle.py`` (and through it the CUDA path).
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))


def _shim():
    sys.path.insert(0, REF)
    torch.Tensor.cuda = lambda self, *a, **k: self          # Contrast.py:32, util.py:104-108
    torch.nn.Module.cuda = lambda self, *a, **k: self


def bf16r(x):
    return x.to(torch.bfloat16).to(torch.float32)


# ------------------------------------------------------------------ shuffle ids
def gen_shuffle_ids():
    from moco.util import DistributedShufle
    out = {}
    for bsz, epoch in [(8, 7), (32, 1), (64, 2), (256, 1), (2048, 1), (2048, 200), (4096, 13), (6, 0)]:
        fwd, bwd = DistributedShufle.get_shuffle_ids(bsz, epoch)
        out[f"fwd_{bsz}_{epoch}"] = fwd.numpy()
        out[f"bwd_{bsz}_{epoch}"] = bwd.numpy()
    np.savez_compressed(os.path.join(OUT, "shuffle_ids.npz"), **out)


# ------------------------------------------------------------------ contrast head
def gen_contrast():
    from moco.NCE import MemoryMoCo, NCESoftmaxLoss
    cases = {
        # name: (N, C, K, all_size, T, start_index, steps)
        "c1head": (32, 128, 1024, 32, 0.07, 0, 3),
        "wrap": (8, 64, 40, 16, 0.07, 0, 4),          # K not a multiple of all_size: wraps mid-batch at step 3
        "c256": (16, 256, 512, 32, 0.2, 0, 2),
        "ragged": (5, 128, 77, 10, 0.1, 0, 3),
    }
    out = {}
    for name, (N, C, K, A, T, idx0, steps) in cases.items():
        torch.manual_seed(1000 + sorted(cases).index(name))
        contrast = MemoryMoCo(C, K, T)
        contrast.index = idx0
        crit = NCESoftmaxLoss()
        out[f"{name}_meta"] = np.array([N, C, K, A, steps], dtype=np.int64)
        out[f"{name}_T"] = np.array([T], dtype=np.float64)
        # make the initial queue bf16-representable so GPU(bf16) and oracle(fp32) agree exactly
        contrast.memory.copy_(bf16r(contrast.memory))
        out[f"{name}_memory0"] = contrast.memory.numpy().copy()
        written = set()
        for s in range(steps):
            q = bf16r(F.normalize(torch.randn(N, C), dim=1)).requires_grad_(True)
            k = bf16r(F.normalize(torch.randn(N, C), dim=1))
            k_all = bf16r(F.normalize(torch.randn(A, C), dim=1))
            k_all[:min(N, A)] = k[:min(N, A)]                   # this rank's keys lead k_all (rank 0 view)
            index_before = contrast.index
            logits = contrast(q, k, k_all)                      # reference forward (+enqueue)
            loss = crit(logits)
            prob = F.softmax(logits, dim=1)[:, 0].mean()       # train.py:264
            loss.backward()                                     # train.py:273
            out[f"{name}_s{s}_q"] = q.detach().numpy().copy()
            out[f"{name}_s{s}_k"] = k.numpy().copy()
            out[f"{name}_s{s}_k_all"] = k_all.numpy().copy()
            out[f"{name}_s{s}_logits"] = logits.detach().numpy().copy()
            out[f"{name}_s{s}_loss"] = np.array([loss.item()], dtype=np.float64)
            out[f"{name}_s{s}_prob"] = np.array([prob.item()], dtype=np.float64)
            out[f"{name}_s{s}_dq"] = q.grad.numpy().copy()
            out[f"{name}_s{s}_index"] = np.array([index_before, contrast.index], dtype=np.int64)
            written.update((index_before + np.arange(A)) % K)
        # keep fixtures small: the final queue is stored as the ring slots the reference wrote (every other row is
        # memory0, asserted here); tests/helpers.py:load_contrast_golden rebuilds `<name>_memory_final`
        final, rows = contrast.memory.numpy(), np.array(sorted(written), dtype=np.int64)
        kept = np.setdiff1d(np.arange(K), rows)
        assert np.array_equal(final[kept], out[f"{name}_memory0"][kept])
        out[f"{name}_memory_final_rows"] = rows
        out[f"{name}_memory_final_vals"] = final[rows].copy()
    # state_dict keys (Contrast.py:15,18)
    sd = MemoryMoCo(128, 16, 0.07).state_dict()
    out["state_dict_keys"] = np.array(sorted(sd.keys()))
    out["state_dict_params"] = sd["params"].numpy()
    # two files, each under 1 MB: the BASELINE configs[0] head shape on its own
    big = {k: v for k, v in out.items() if k.startswith("c1head_")}
    np.savez_compressed(os.path.join(OUT, "contrast_c1head.npz"), **big)
    np.savez_compressed(os.path.join(OUT, "contrast.npz"), **{k: v for k, v in out.items() if k not in big})


# ------------------------------------------------------------------ Normalize -> head (SURVEY 8 f2)
def gen_normalize():
    """The reference's own `Normalize` layer (moco/models/resnet.py:24-33) in front of its head, differentiated down
    to the RAW encoder output: what moco_nce_step(normalize=1) fuses."""
    from moco.NCE import MemoryMoCo, NCESoftmaxLoss
    from moco.models.resnet import Normalize
    out = {}
    for ci, (name, (N, C, K, A, T)) in enumerate({"n128": (32, 128, 1024, 32, 0.07), "n64": (24, 64, 320, 48, 0.1)}.items()):
        torch.manual_seed(2000 + ci)
        contrast = MemoryMoCo(C, K, T)
        contrast.memory.copy_(bf16r(contrast.memory))
        l2 = Normalize(2)
        xq = (torch.randn(N, C) * 3.0).requires_grad_(True)
        xk = torch.randn(N, C) * 0.5
        xk_all = torch.randn(A, C) * 2.0
        xk_all[:min(N, A)] = xk[:min(N, A)]
        out[f"{name}_meta"] = np.array([N, C, K, A], dtype=np.int64)
        out[f"{name}_T"] = np.array([T], dtype=np.float64)
        out[f"{name}_memory0"] = contrast.memory.numpy().copy()
        q, k, k_all = l2(xq), l2(xk), l2(xk_all)
        logits = contrast(q, k, k_all)
        loss = NCESoftmaxLoss()(logits)
        prob = F.softmax(logits, dim=1)[:, 0].mean()
        loss.backward()
        for key, val in dict(xq=xq.detach(), xk=xk, xk_all=xk_all, q=q.detach(), k=k, dxq=xq.grad,
                             memory_final=contrast.memory).items():
            out[f"{name}_{key}"] = val.numpy().copy()
        out[f"{name}_loss"] = np.array([loss.item()], dtype=np.float64)
        out[f"{name}_prob"] = np.array([prob.item()], dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "normalize.npz"), **out)


# ------------------------------------------------------------------ ShuffleBN over gloo
def _shuffle_worker(rank, world, n, epoch, port, ret):
    _shim()
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from moco.util import DistributedShufle
    g = torch.Generator().manual_seed(100 + rank)
    x = torch.randn(n, 3, 4, 4, generator=g)                    # "images" (small spatial dims)
    x_shuf, binds = DistributedShufle.forward_shuffle(x, epoch)
    # a stand-in "key encoder": per-row features that depend only on the row content
    feat = x_shuf.reshape(n, -1)[:, :16].contiguous()
    feat_all, feat_local = DistributedShufle.backward_shuffle(feat, binds, return_local=True)
    ret[rank] = dict(x=x.numpy(), x_shuf=x_shuf.numpy(), binds=binds.numpy(),
                     feat=feat.numpy(), feat_all=feat_all.numpy(), feat_local=feat_local.numpy())
    dist.barrier()
    dist.destroy_process_group()


def gen_shuffle():
    out = {}
    port = 29611
    for world, n, epoch in [(1, 8, 3), (2, 4, 7), (4, 6, 2)]:
        mgr = mp.Manager()
        ret = mgr.dict()
        mp.spawn(_shuffle_worker, args=(world, n, epoch, port, ret), nprocs=world, join=True)
        port += 1
        tag = f"w{world}_n{n}_e{epoch}"
        for r in range(world):
            for key, val in ret[r].items():
                out[f"{tag}_r{r}_{key}"] = val
    np.savez_compressed(os.path.join(OUT, "shuffle.npz"), **out)


# ------------------------------------------------------------------ EMA (moment_update)
def gen_ema():
    from moco.util import moment_update
    torch.manual_seed(77)

    def make():
        # odd sizes on purpose: 1-element, non-multiple-of-4 and > one kernel chunk (8192 elements)
        return torch.nn.Sequential(torch.nn.Conv2d(3, 7, 3), torch.nn.BatchNorm2d(7), torch.nn.Linear(131, 67),
                                   torch.nn.Linear(1, 1), torch.nn.Linear(95, 33, bias=False))
    out = {}
    for tag, m, steps in [("m999", 0.999, 3), ("m99", 0.99, 2), ("m0", 0.0, 1)]:
        model, model_ema = make(), make()
        out[f"{tag}_m"] = np.array([m], dtype=np.float64)
        out[f"{tag}_steps"] = np.array([steps], dtype=np.int64)
        for i, p in enumerate(model_ema.parameters()):
            out[f"{tag}_ema0_{i}"] = p.detach().numpy().copy()
        for s in range(steps):
            with torch.no_grad():
                for p in model.parameters():                    # a different "trained" model every step
                    p.copy_(torch.randn_like(p) * 0.05)
            for i, p in enumerate(model.parameters()):
                out[f"{tag}_s{s}_p_{i}"] = p.detach().numpy().copy()
            moment_update(model, model_ema, m)                  # reference util.py:124-127
            for i, p in enumerate(model_ema.parameters()):
                out[f"{tag}_s{s}_ema_{i}"] = p.detach().numpy().copy()
        out[f"{tag}_n"] = np.array([len(list(model.parameters()))], dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "ema.npz"), **out)


# ------------------------------------------------------------------ encoder-side ops (BN group, max-pool, conv1)
def gen_encoder_ops():
    """Tensors captured INSIDE the reference's own modules (moco/models/resnet.py): the stem
    (conv1 -> bn1 -> relu -> maxpool, :155-158) and one Bottleneck with a downsample branch (:83-104), forward values
    and autograd gradients, fp32 on CPU."""
    from moco.models.resnet import ResNet, Bottleneck
    import torch.nn as nn
    out = {}
    torch.manual_seed(11)
    net = ResNet(Bottleneck, [1, 1, 1, 1], low_dim=16)
    net.train()
    with torch.no_grad():
        net.bn1.weight.copy_(torch.rand(64) + 0.5)
        net.bn1.bias.copy_(torch.randn(64) * 0.2)
    x = torch.randn(4, 3, 32, 32)
    cap = {}

    def keep(name, clone=False):
        def hook(m, i, o):                        # returns None: the module's output is left alone
            o.retain_grad()
            cap[name] = o
            if clone:
                cap[name + "_val"] = o.detach().clone()
        return hook
    h1 = net.conv1.register_forward_hook(keep("conv1"))
    y = net(x, layer=1)                                                   # conv1 -> bn1 -> relu -> maxpool
    h1.remove()
    dp = torch.randn_like(y)
    rm0, rv0 = torch.zeros(64), torch.ones(64)
    y.backward(dp)
    out.update(stem_x=x.numpy(), stem_w=net.conv1.weight.detach().numpy(), stem_conv1=cap["conv1"].detach().numpy(),
               stem_gamma=net.bn1.weight.detach().numpy(), stem_beta=net.bn1.bias.detach().numpy(),
               stem_pooled=y.detach().numpy(), stem_dpooled=dp.numpy(), stem_dconv1=cap["conv1"].grad.numpy(),
               stem_dgamma=net.bn1.weight.grad.numpy(), stem_dbeta=net.bn1.bias.grad.numpy(),
               stem_running_mean=net.bn1.running_mean.numpy().copy(), stem_running_var=net.bn1.running_var.numpy().copy(),
               stem_running_mean0=rm0.numpy(), stem_running_var0=rv0.numpy())
    # one Bottleneck whose residual comes from a downsample branch, so that the residual's gradient is observable
    torch.manual_seed(12)
    ds = nn.Sequential(nn.Conv2d(32, 64, kernel_size=1, stride=1, bias=False), nn.BatchNorm2d(64))
    blk = Bottleneck(32, 16, stride=1, downsample=ds)
    blk.train()
    with torch.no_grad():
        blk.bn3.weight.copy_(torch.rand(64) + 0.5)
        blk.bn3.bias.copy_(torch.randn(64) * 0.2)
    xb = torch.randn(3, 32, 6, 6)
    cap.clear()
    h3 = blk.conv3.register_forward_hook(keep("conv3"))
    hd = ds.register_forward_hook(keep("res", clone=True))
    yb = blk(xb)
    h3.remove(); hd.remove()
    dyb = torch.randn_like(yb)
    yb.backward(dyb)
    out.update(blk_conv3=cap["conv3"].detach().numpy(), blk_res=cap["res_val"].numpy(), blk_gamma=blk.bn3.weight.detach().numpy(),
               blk_beta=blk.bn3.bias.detach().numpy(), blk_out=yb.detach().numpy(), blk_dout=dyb.numpy(),
               blk_dconv3=cap["conv3"].grad.numpy(), blk_dres=cap["res"].grad.numpy(),
               blk_dgamma=blk.bn3.weight.grad.numpy(), blk_dbeta=blk.bn3.bias.grad.numpy(),
               blk_running_mean=blk.bn3.running_mean.numpy().copy(), blk_running_var=blk.bn3.running_var.numpy().copy())
    np.savez_compressed(os.path.join(OUT, "encoder_ops.npz"), **out)


# ------------------------------------------------------------------ the reference's training loop (drop-in test)
def gen_dropin():
    """Three steps of the reference's own ``train.train_moco`` (train.py:231-293) with its own head, ShuffleBN and
    EMA: ResNet-18, 16 synthetic 224 x 224 images per step, K = 256, fp32 on CPU in a gloo group of one.
    tests/dropin_train_py.py repeats the run with this project's modules on the GPU and compares with what is stored
    here: the learning rate of every step, the averaged loss / prob, the ring position, the final queue, and the query
    and EMA encoders' ``fc`` weights."""
    import argparse
    import logging
    import tempfile
    import types
    import warnings
    stub = types.ModuleType("termcolor")                        # moco/logger.py imports it; not installed
    stub.colored = lambda s, *a, **k: s
    sys.modules.setdefault("termcolor", stub)
    store = os.path.join(tempfile.mkdtemp(prefix="moco_golden_"), "store")
    dist.init_process_group("gloo", init_method=f"file://{store}", rank=0, world_size=1)
    import train
    from moco.lr_scheduler import get_scheduler
    from moco.models.resnet import resnet18
    from moco.NCE import MemoryMoCo, NCESoftmaxLoss
    from moco.util import moment_update
    train.logger = logging.getLogger("moco_golden")            # a module global only train.py's __main__ defines
    train.logger.setLevel(logging.WARNING)
    steps, N, K = 3, 16, 256
    args = argparse.Namespace(batch_size=N, nce_k=K, nce_t=0.07, alpha=0.999, base_learning_rate=0.03, lr_scheduler="cosine",
                              warmup_epoch=1, warmup_multiplier=100, lr_decay_epochs=[120, 160, 200], lr_decay_rate=0.1,
                              weight_decay=1e-4, momentum=0.9, amp_opt_level="O0", epochs=200, start_epoch=1,
                              print_freq=10 ** 9, local_rank=0, model_width=1)
    torch.manual_seed(0)
    model, model_ema = resnet18(), resnet18()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        moment_update(model, model_ema, 0)                      # train.py:133
    contrast = MemoryMoCo(128, K, 0.07)                         # train.py:181
    with torch.no_grad():                                       # bf16-representable queue: both heads see the same negatives
        contrast.memory.copy_(bf16r(contrast.memory))
    optimizer = torch.optim.SGD(model.parameters(), lr=N / 256 * args.base_learning_rate, momentum=0.9, weight_decay=1e-4)
    scheduler = get_scheduler(optimizer, steps, args)
    lrs = []
    sgd_step = optimizer.step

    def step_and_record(*a, **k):                              # the learning rate each SGD step used
        lrs.append(optimizer.param_groups[0]["lr"])
        return sgd_step(*a, **k)
    optimizer.step = step_and_record
    ddp = torch.nn.parallel.DistributedDataParallel(model, broadcast_buffers=False)    # train.py:198
    g = torch.Generator().manual_seed(7)
    # 224 x 224: the reference's AvgPool2d(7) (resnet.py:124) needs a 7 x 7 final map; the batch is kept small instead
    loader = [(torch.randn(N, 6, 224, 224, generator=g), None) for _ in range(steps)]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        loss, prob = train.train_moco(1, loader, ddp, model_ema, contrast, NCESoftmaxLoss(), optimizer, scheduler, args)
    dist.destroy_process_group()
    np.savez_compressed(os.path.join(OUT, "dropin.npz"),
                        meta=np.array([steps, N, K], dtype=np.int64), lrs=np.array(lrs, dtype=np.float64),
                        loss=np.array([loss], dtype=np.float64), prob=np.array([prob], dtype=np.float64),
                        index=np.array([contrast.index], dtype=np.int64), memory=contrast.memory.numpy().copy(),
                        fc=model.fc.weight.detach().numpy().copy(), ema_fc=model_ema.fc.weight.detach().numpy().copy())


GENERATORS = {"encoder_ops": gen_encoder_ops, "ema": gen_ema, "shuffle_ids": gen_shuffle_ids, "contrast": gen_contrast,
              "normalize": gen_normalize, "shuffle": gen_shuffle, "dropin": gen_dropin}


if __name__ == "__main__":
    _shim()
    # --only-<name> (e.g. --only-encoder-ops, --only-dropin) regenerates just those fixtures
    only = [a[len("--only-"):].replace("-", "_") for a in sys.argv[1:] if a.startswith("--only-")]
    for name in only or GENERATORS:
        GENERATORS[name]()
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(OUT, f)))
