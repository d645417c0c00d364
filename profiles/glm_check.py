"""GPU check of the fused GLM likelihood kernels through the C ABI: accuracy of every variant against an
fp64 torch evaluation of the same inputs, and device time (CUDA events around graph replays, L2 flushed
between replays).  Usage: python profiles/glm_check.py [--quick]"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pyro_b200 import _native as N  # noqa: E402

VARIANTS = {"tc_default": 0, "tc_3xtf32": N.B2_FLAG_GLM_3XTF32, "fp32_simt": N.B2_FLAG_GLM_FP32}


def run(X, y, W, b, flags):
    n, D = X.shape
    P = W.shape[0]
    dev = X.device
    total = torch.empty((), dtype=torch.float32, device=dev)
    sum_p = torch.empty(P, dtype=torch.float32, device=dev)
    dW = torch.empty(P, D, dtype=torch.float32, device=dev)
    db = torch.empty(P, dtype=torch.float32, device=dev)
    need = int(N.lib().b2_glm_workspace(n, D, P))
    ws = N.workspace(dev, need, tag="glm_check")

    def call():
        N.check(N.lib().b2_glm_bernoulli_logits(
            X.data_ptr(), y.data_ptr(), W.data_ptr(), b.data_ptr() if b is not None else None,
            n, D, P, 1.0, 1.0, 1.0, int(flags), sum_p.data_ptr(), total.data_ptr(), dW.data_ptr(),
            db.data_ptr(), ws.data_ptr(), ws.numel(), N.stream_ptr(dev)), "b2_glm_bernoulli_logits")
    return call, (total, sum_p, dW, db)


def reference(X, y, W, b):
    Xd, yd, Wd = X.double(), y.double(), W.double()
    logits = Wd @ Xd.t()
    if b is not None:
        logits = logits + b.double()[:, None]
    lp = yd * logits - torch.nn.functional.softplus(logits)
    g = yd - torch.sigmoid(logits)
    return lp.sum(1), g @ Xd, g.sum(1)


def main():
    quick = "--quick" in sys.argv
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    ok = True
    cases = [(300, 7, True), (4096, 64, True), (100000, 64, True), (1000003, 64, True), (5000, 100, False)]
    if quick:
        cases = cases[:3]
    for n, P, bias in cases:
        X = torch.randn(n, 32, device=dev)
        wt = torch.randn(32, device=dev) / 32 ** 0.5
        y = (torch.rand(n, device=dev) < torch.sigmoid(X @ wt + 0.5)).float()
        W = 0.3 * torch.randn(P, 32, device=dev) + wt
        b = (0.5 + 0.2 * torch.randn(P, device=dev)) if bias else None
        s_ref, dW_ref, db_ref = reference(X, y, W, b)
        for name, flags in VARIANTS.items():
            call, (total, sum_p, dW, db) = run(X, y, W, b, flags)
            try:
                call()
                torch.cuda.synchronize()
            except Exception as e:  # noqa: BLE001
                print("CASE n=%d P=%d %-10s FAILED: %s" % (n, P, name, e))
                ok = False
                continue
            e_sum = float(((sum_p.double() - s_ref).abs() / s_ref.abs().clamp_min(1.0)).max())
            e_dw = float((dW.double() - dW_ref).abs().max() / dW_ref.abs().max().clamp_min(1.0))
            e_db = float((db.double() - db_ref).abs().max() / db_ref.abs().max().clamp_min(1.0))
            e_tot = float((total.double() - s_ref.sum()).abs() / s_ref.sum().abs())
            print("CASE n=%d P=%d bias=%d %-10s rel err: sum_p %.2e total %.2e dW %.2e db %.2e"
                  % (n, P, bias, name, e_sum, e_tot, e_dw, e_db))
            if not (e_sum < 2e-5 and e_dw < 2e-4 and e_db < 2e-4):
                print("   ^^^ OUT OF TOLERANCE")
                ok = False
    # ---- timing at the BASELINE size ---------------------------------------------------------------------
    n, P = 1000000, 64
    X = torch.randn(n, 32, device=dev)
    y = (torch.rand(n, device=dev) < 0.5).float()
    W = 0.3 * torch.randn(P, 32, device=dev)
    b = torch.randn(P, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for name, flags in VARIANTS.items():
        call, _ = run(X, y, W, b, flags)
        try:
            for _ in range(3):
                call()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                call()
            ts = []
            for _ in range(10):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                g.replay()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) * 1e3)
            ts.sort()
            med = ts[len(ts) // 2]
            print("TIME %-10s N=1e6 P=64: median %.1f us (min %.1f) incl. finish kernel -> %.0f GB/s algorithmic, frac %.3f of 6576"
                  % (name, med, ts[0], 132e6 / med / 1e3, 132e6 / med / 1e3 / 6576.1))
        except Exception as e:  # noqa: BLE001
            print("TIME %-10s FAILED: %s" % (name, e))
            ok = False
    print("GLM_CHECK", "OK" if ok else "FAIL", time.strftime("%H:%M:%S"))


if __name__ == "__main__":
    main()
