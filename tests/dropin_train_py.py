"""Runs the reference's training loop (train.train_moco, train.py:231-293) on the GPU with exactly the import swap
INTEGRATION.md section 1 prescribes -- MemoryMoCo / NCESoftmaxLoss / DistributedShufle / moment_update from moco_b200 --
and compares it with the reference's own run from the same seeds (tests/golden/dropin.npz, written by
tests/golden/gen_golden.py:gen_dropin).  Prints one JSON line.
Test helper (tests/test_gpu_dropin.py runs it in its own process: it owns a process group and the CUDA device).

The loop body is train_moco's, line for line.  The encoders are moco_b200.encoders.resnet18, which under the same seed
holds exactly the parameters of the reference's moco.models.resnet.resnet18 (same layers, same initialisation, same
random draws) and computes the same function in fp32.  The reference's warm-up schedule (moco/lr_scheduler.py) is
replayed from the learning rates its run recorded."""
import json
import os
import sys
import tempfile
import warnings

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "dropin.npz")


def run(lrs, steps: int, N: int, K: int):
    from moco_b200 import encoders
    from moco_b200.NCE import MemoryMoCo, NCESoftmaxLoss
    from moco_b200.util import DistributedShufle, moment_update, set_bn_train
    torch.manual_seed(0)
    model, model_ema = encoders.resnet18().cuda(), encoders.resnet18().cuda()
    moment_update(model, model_ema, 0)                          # train.py:133
    contrast = MemoryMoCo(128, K, 0.07).cuda()                  # train.py:181
    with torch.no_grad():                                       # bf16-representable initial queue: both heads see the same negatives
        contrast.memory.copy_(contrast.memory.bfloat16().float())
    criterion = NCESoftmaxLoss().cuda()
    optimizer = torch.optim.SGD(model.parameters(), lr=lrs[0], momentum=0.9, weight_decay=1e-4)
    ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[0], broadcast_buffers=False)     # train.py:198
    g = torch.Generator().manual_seed(7)
    loader = [torch.randn(N, 6, 224, 224, generator=g) for _ in range(steps)]
    ddp.train()                                                 # train.py:234-235
    set_bn_train(model_ema)
    losses, probs = [], []
    for i, inputs in enumerate(loader):
        for group in optimizer.param_groups:                    # what the reference's scheduler set for this step
            group["lr"] = lrs[i]
        x1, x2 = torch.split(inputs, [3, 3], dim=1)             # train.py:250-254
        x1, x2 = x1.cuda(non_blocking=True), x2.cuda(non_blocking=True)
        feat_q = ddp(x1)                                        # train.py:256-260
        with torch.no_grad():
            x2_shuffled, backward_inds = DistributedShufle.forward_shuffle(x2, 1)
            feat_k = model_ema(x2_shuffled)
            feat_k_all, feat_k = DistributedShufle.backward_shuffle(feat_k, backward_inds, return_local=True)
        out = contrast(feat_q, feat_k, feat_k_all)              # train.py:262-264
        loss = criterion(out)
        prob = F.softmax(out, dim=1)[:, 0].mean()
        optimizer.zero_grad()                                   # train.py:267-275
        loss.backward()
        optimizer.step()
        moment_update(model, model_ema, 0.999)                  # train.py:277
        losses.append(loss.item())                              # train.py:280-281 (equal batches: the meters' mean)
        probs.append(prob.item())
    torch.cuda.synchronize()
    return {"loss_avg": float(np.mean(losses)), "prob_avg": float(np.mean(probs)), "index": int(contrast.index),
            "memory": contrast.memory.detach().float().cpu().numpy(), "fc": model.fc.weight.detach().float().cpu().numpy(),
            "ema_fc": model_ema.fc.weight.detach().float().cpu().numpy()}


def main():
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    ref = np.load(GOLDEN)
    steps, N, K = (int(v) for v in ref["meta"])
    torch.cuda.set_device(0)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.deterministic = True
    with tempfile.TemporaryDirectory(prefix="moco_dropin_") as tmp:
        dist.init_process_group("nccl", init_method=f"file://{os.path.join(tmp, 'store')}", rank=0, world_size=1,
                                device_id=torch.device("cuda", 0))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            new = run([float(v) for v in ref["lrs"]], steps, N, K)
        dist.destroy_process_group()
    out = {"ref_loss": float(ref["loss"][0]), "new_loss": new["loss_avg"], "ref_prob": float(ref["prob"][0]),
           "new_prob": new["prob_avg"], "ref_index": int(ref["index"][0]), "new_index": new["index"],
           "memory_max_abs_diff": float(np.abs(ref["memory"] - new["memory"]).max()),
           "fc_rel_diff": float(np.abs(ref["fc"] - new["fc"]).max() / np.abs(ref["fc"]).max()),
           "ema_fc_rel_diff": float(np.abs(ref["ema_fc"] - new["ema_fc"]).max() / np.abs(ref["ema_fc"]).max())}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
