"""GPU bring-up lab: runs each kernel variant in its own subprocess (a trap in one
kernel must not poison the others) with a timeout, checks it against a torch
fp32 reference computed on the same GPU and prints one JSON line per case.

    python tools/gpu_lab.py            # all cases
    python tools/gpu_lab.py tc1_c2     # one case, in-process
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FLAGS = {"auto": 0, "simt": 1, "tc2": 2, "tc1": 4, "op": 4 | 1024, "tp": 4 | 512}
# name: (N, C, K, T, flagname, want_logits, timing_iters)
NCE_CASES = {
    "simt_small": (32, 128, 1024, 0.07, "simt", True, 0),
    "tc1_small": (32, 128, 1024, 0.07, "tc1", True, 0),
    "tc2_small": (32, 128, 1024, 0.07, "tc2", True, 0),
    "tc1_ragged": (200, 192, 1000, 0.1, "tc1", True, 0),
    "tc2_ragged": (200, 192, 1000, 0.1, "tc2", True, 0),
    "tc1_c2": (256, 128, 16384, 0.07, "tc1", False, 20),
    "tc2_c2": (256, 128, 16384, 0.07, "tc2", False, 20),
    "tc1_c3": (256, 128, 65536, 0.07, "tc1", False, 20),
    "tc2_c3": (256, 128, 65536, 0.07, "tc2", False, 20),
    "tc1_c5": (512, 256, 262144, 0.07, "tc1", False, 10),
    "tc2_c5": (512, 256, 262144, 0.07, "tc2", False, 10),
    "tc1_c3_dense": (256, 128, 65536, 0.07, "tc1", True, 5),
    "tc1_c4": (2048, 128, 16384, 0.07, "tc1", False, 20),
    "tc1_ragged2": (300, 64, 5000, 0.1, "tc1", True, 0),
    # one sweep for loss + dq ("op") vs statistics pass + dq pass ("tp")
    "op_small": (32, 128, 1024, 0.07, "op", False, 0),
    "op_ragged": (200, 192, 1000, 0.1, "op", False, 0),
    "op_ragged2": (300, 64, 5000, 0.1, "op", False, 0),
    "op_c2": (256, 128, 16384, 0.07, "op", False, 20),
    "op_c3": (256, 128, 65536, 0.07, "op", False, 20),
    "op_c4": (2048, 128, 16384, 0.07, "op", False, 20),
    "op_c5": (512, 256, 262144, 0.07, "op", False, 10),
    "tp_small": (32, 128, 1024, 0.07, "tp", False, 0),
    "tp_ragged": (200, 192, 1000, 0.1, "tp", False, 0),
    "tp_c64": (100, 64, 777, 0.07, "tp", False, 0),
    "op_c64": (100, 64, 777, 0.07, "op", False, 0),
    "tp_c4": (2048, 128, 16384, 0.07, "tp", False, 20),
    "tp_c2": (256, 128, 16384, 0.07, "tp", False, 20),
    "tp_c3": (256, 128, 65536, 0.07, "tp", False, 20),
    "tp_c5": (512, 256, 262144, 0.07, "tp", False, 10),
}


def run_nce(name):
    import torch
    import torch.nn.functional as F
    from moco_b200 import _lib
    N, C, K, T, flagname, want_logits, iters = NCE_CASES[name]
    lib = _lib.load()
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    q = F.normalize(torch.randn(N, C, device=dev, generator=g), dim=1).bfloat16()
    k = F.normalize(torch.randn(N, C, device=dev, generator=g), dim=1).bfloat16()
    queue = F.normalize(torch.randn(K, C, device=dev, generator=g), dim=1).bfloat16()
    f32 = dict(dtype=torch.float32, device=dev)
    logits = torch.zeros(N, K + 1, **f32) if want_logits else None
    lse, loss_rows, prob_rows = (torch.zeros(N, **f32) for _ in range(3))
    loss_prob = torch.zeros(2, **f32)
    dq = torch.zeros(N, C, **f32)
    wsb = lib.moco_nce_workspace_bytes(N, C, K)
    ws = torch.zeros(wsb + 256, dtype=torch.uint8, device=dev)
    ws_ptr = ws.data_ptr() + (-ws.data_ptr()) % 256
    stream = torch.cuda.current_stream().cuda_stream

    def call(with_dq=True):
        code = lib.moco_nce_fwd(q.data_ptr(), k.data_ptr(), 1, queue.data_ptr(), N, C, K, 1.0 / T,
                                logits.data_ptr() if logits is not None else None, lse.data_ptr(),
                                loss_rows.data_ptr(), prob_rows.data_ptr(), loss_prob.data_ptr(),
                                dq.data_ptr() if with_dq else None, ws_ptr, wsb, FLAGS[flagname], stream)
        if code != 0:
            raise RuntimeError(f"moco_nce_fwd -> {code}: {lib.moco_last_error().decode()}")

    call()
    torch.cuda.synchronize()
    # torch fp32 reference on the same (bf16-representable) inputs
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    qf = q.float().requires_grad_(True)
    kf, mf = k.float(), queue.float()
    ref = torch.cat([(qf * kf).sum(-1, keepdim=True), qf @ mf.t()], 1) / T
    ref_loss = F.cross_entropy(ref, torch.zeros(N, dtype=torch.long, device=dev))
    ref_prob = F.softmax(ref, 1)[:, 0].mean()
    ref_loss.backward()
    ref_lse = torch.logsumexp(ref.detach(), 1)
    torch.backends.cuda.matmul.allow_tf32 = prev
    out = {"case": name, "N": N, "C": C, "K": K}
    if want_logits:
        out["logits_max_abs_err"] = float((logits - ref.detach()).abs().max())
        out["logits_rel_err"] = float((logits - ref.detach()).abs().max() / ref.detach().abs().max())
    out["lse_max_abs_err"] = float((lse - ref_lse).abs().max())
    out["loss"] = float(loss_prob[0]); out["ref_loss"] = float(ref_loss)
    out["prob"] = float(loss_prob[1]); out["ref_prob"] = float(ref_prob)
    dq_ref = qf.grad
    out["dq_rel_err"] = float((dq - dq_ref).abs().max() / dq_ref.abs().max())
    ok = out["lse_max_abs_err"] < 2e-3 and abs(out["loss"] - out["ref_loss"]) < 2e-3 and out["dq_rel_err"] < 2e-2
    if want_logits:
        ok = ok and out["logits_rel_err"] < 1e-3
    out["ok"] = bool(ok)
    if iters:
        for with_dq, tag in ((False, "fwd_us"), (True, "fwd_dq_us")):
            for _ in range(3):
                call(with_dq)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                call(with_dq)
            e1.record()
            torch.cuda.synchronize()
            out[tag] = e0.elapsed_time(e1) * 1e3 / iters
        # per-kernel device time via the library's profiling hook (events right around one kernel)
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(iters)]
        for e4 in ev:
            for e in e4:
                e.record()
        for i in range(iters):
            lib.moco_prof_set_events(1, ev[i][0].cuda_event, ev[i][1].cuda_event)
            lib.moco_prof_set_events(2, ev[i][2].cuda_event, ev[i][3].cuda_event)
            call(True)
        lib.moco_prof_set_events(1, None, None)
        lib.moco_prof_set_events(2, None, None)
        torch.cuda.synchronize()
        out["stats_kernel_us"] = sum(e[0].elapsed_time(e[1]) for e in ev) * 1e3 / iters
        out["dq_kernel_us"] = sum(e[2].elapsed_time(e[3]) for e in ev) * 1e3 / iters
        if out["stats_kernel_us"] > 1.0:
            out["stats_tflops"] = 2.0 * N * C * K / (out["stats_kernel_us"] * 1e-6) / 1e12
        else:                                   # one-pass mode: no statistics kernel ran
            del out["stats_kernel_us"]
        out["dq_tflops"] = 4.0 * N * C * K / (out["dq_kernel_us"] * 1e-6) / 1e12
        import ctypes
        win = ctypes.c_float()
        lib.moco_prof_sweep_window(ws_ptr, 148, ctypes.byref(win), stream)
        out["sweep_device_window_us"] = float(win.value)
    return out


def run_enqueue(name):
    import torch
    from moco_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda:0")
    res = {"case": name, "ok": True}
    for (K, C, n_all, index, dt) in [(40, 64, 16, 32, torch.float32), (1024, 128, 256, 1000, torch.bfloat16),
                                     (77, 100, 10, 70, torch.float32), (65536, 128, 2048, 65000, torch.float32)]:
        qf = torch.randn(K, C, device=dev)
        qb = qf.bfloat16()
        k_all = torch.randn(n_all, C, device=dev).to(dt)
        ref_f, ref_b = qf.clone(), qb.clone()
        ids = (torch.arange(n_all, device=dev) + index) % K
        ref_f[ids] = k_all.float()
        ref_b[ids] = k_all.bfloat16()
        code = lib.moco_queue_enqueue(qb.data_ptr(), qf.data_ptr(), k_all.data_ptr(), 0 if dt == torch.float32 else 1,
                                      n_all, C, K, index, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        good = code == 0 and torch.equal(qf, ref_f) and torch.equal(qb, ref_b)
        res["ok"] = res["ok"] and bool(good)
        res[f"K{K}_C{C}"] = bool(good)
    return res


def run_gather(name):
    import ctypes
    import torch
    from moco_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda:0")
    res = {"case": name, "ok": True}
    stream = torch.cuda.current_stream().cuda_stream
    for tag, shape, flags in [("small", (256, 128), 0), ("img_bulk", (64, 3, 224, 224), 0), ("img_ldg", (64, 3, 224, 224), 1),
                              ("img_bf16_bulk", (256, 3, 224, 224), 0)]:
        dt = torch.bfloat16 if "bf16" in tag else torch.float32
        x = torch.randn(*shape, device=dev).to(dt)
        n = shape[0]
        perm = torch.randperm(n, device=dev)
        out = torch.empty_like(x)
        row_bytes = x[0].numel() * x.element_size()
        table = (ctypes.c_void_p * 1)(x.data_ptr())
        code = lib.moco_shuffle_gather(table, 1, n, perm.data_ptr(), n, row_bytes, out.data_ptr(), flags, stream)
        torch.cuda.synchronize()
        good = code == 0 and torch.equal(out, x[perm])
        res[tag] = bool(good)
        res["ok"] = res["ok"] and bool(good)
        if good:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(3):
                lib.moco_shuffle_gather(table, 1, n, perm.data_ptr(), n, row_bytes, out.data_ptr(), flags, stream)
            e0.record()
            for _ in range(10):
                lib.moco_shuffle_gather(table, 1, n, perm.data_ptr(), n, row_bytes, out.data_ptr(), flags, stream)
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 100
            res[tag + "_us"] = us
            res[tag + "_GBps"] = 2 * n * row_bytes / (us * 1e-6) / 1e9
    return res


def run_module(name):
    """End-to-end through the Python modules against the golden fixture."""
    import torch
    from moco_b200.NCE import MemoryMoCo, NCESoftmaxLoss
    from tests.helpers import load_contrast_golden
    g = load_contrast_golden(os.path.join(ROOT, "tests", "golden"))
    res = {"case": name, "ok": True}
    for cname in ["c1head", "wrap", "c256", "ragged"]:
        N, C, K, A, steps = (int(v) for v in g[f"{cname}_meta"])
        T = float(g[f"{cname}_T"][0])
        m = MemoryMoCo(C, K, T)
        m.memory.copy_(torch.from_numpy(g[f"{cname}_memory0"]))
        m = m.cuda()
        crit = NCESoftmaxLoss()
        worst = 0.0
        for s in range(steps):
            q = torch.from_numpy(g[f"{cname}_s{s}_q"]).cuda().requires_grad_(True)
            k = torch.from_numpy(g[f"{cname}_s{s}_k"]).cuda()
            k_all = torch.from_numpy(g[f"{cname}_s{s}_k_all"]).cuda()
            out = m(q, k, k_all)
            loss = crit(out)
            loss.backward()
            ref = torch.from_numpy(g[f"{cname}_s{s}_logits"]).cuda()
            e1 = float((out.detach() - ref).abs().max() / ref.abs().max())
            e2 = abs(float(loss) - float(g[f"{cname}_s{s}_loss"][0]))
            dq_ref = torch.from_numpy(g[f"{cname}_s{s}_dq"]).cuda()
            e3 = float((q.grad - dq_ref).abs().max() / dq_ref.abs().max())
            worst = max(worst, e1, e2, e3)
            assert m.index == int(g[f"{cname}_s{s}_index"][1])
        mem_ok = bool(torch.equal(m.memory.cpu(), torch.from_numpy(g[f"{cname}_memory_final"])))
        res[cname] = {"worst_err": worst, "memory_bit_exact": mem_ok}
        res["ok"] = res["ok"] and worst < 2e-3 and mem_ok
    return res


CASES = {**{n: run_nce for n in NCE_CASES}, "enqueue": run_enqueue, "gather": run_gather, "module": run_module}


def main():
    if len(sys.argv) == 2 and sys.argv[1] != "--all":
        name = sys.argv[1]
        print(json.dumps(CASES[name](name)))
        return
    order = ["enqueue", "gather", "simt_small", "tc1_small", "tc2_small", "tc1_ragged", "tc2_ragged", "s4_ragged",
             "tc1_ragged2", "module", "tc1_c2", "tc2_c2", "tc1_c3", "nomc_c3", "tc2_c3", "tc1_c4", "s4_c4",
             "tc1_c5", "nomc_c5", "s4_c5", "tc2_c5", "tc1_c3_dense"]
    if len(sys.argv) > 2:
        order = sys.argv[1:]
    for name in order:
        t0 = time.time()
        try:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), name], capture_output=True, text=True,
                               timeout=180)
            line = p.stdout.strip().splitlines()[-1] if p.stdout.strip() else ""
            if p.returncode != 0 or not line.startswith("{"):
                print(json.dumps({"case": name, "ok": False, "rc": p.returncode,
                                  "stderr": p.stderr[-1500:], "stdout": p.stdout[-500:]}))
            else:
                print(line)
        except subprocess.TimeoutExpired:
            print(json.dumps({"case": name, "ok": False, "error": "timeout"}))
        sys.stdout.flush()


if __name__ == "__main__":
    main()
