"""Diagnostic (GPU box only): scn_conv_wgrad (tcgen05 path) vs a plain torch
gather + matmul of the same bf16 operands; prints the error structure so a descriptor / layout mistake is identifiable."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from sparseeventid_b200 import _lib as L
from sparseeventid_b200.scn import ops

torch.manual_seed(0)
dev = "cuda"


def case(n, K, cin, cout, density=0.3, n_in=None):
    n_in = n_in or n
    n_pad = ops.pad128(n)
    nbr = torch.full((K, n_pad), -1, dtype=torch.int32, device=dev)
    mask = torch.rand(K, n, device=dev) < density
    if K % 2 == 1:
        mask[K // 2] = True
    idx = torch.randint(0, n_in, (K, n), device=dev, dtype=torch.int32)
    nbr[:, :n] = torch.where(mask, idx, torch.full_like(idx, -1))
    x = torch.randn(n_in, cin, device=dev).bfloat16()
    d = torch.randn(n, cout, device=dev).bfloat16()
    dw = ops.conv_wgrad(x, d, nbr, n, cin, cout, L.PREC_BF16)
    torch.cuda.synchronize()
    ref = torch.zeros(K, cin, cout, device=dev)
    xf, df = x.float(), d.float()
    for k in range(K):
        j = nbr[k, :n].long()
        m = j >= 0
        ref[k] = xf[j[m]].t() @ df[m]
    err = (dw - ref).abs()
    rel = float(err.max() / ref.abs().max().clamp_min(1e-6))
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(5):
        ops.conv_wgrad(x, d, nbr, n, cin, cout, L.PREC_BF16)
    t1.record()
    torch.cuda.synchronize()
    us = t0.elapsed_time(t1) / 5 * 1e3
    pairs = int(mask.sum())
    print(f"n={n} K={K} {cin}->{cout} rel_max_err={rel:.3e} time={us:.1f}us TF={2.0 * pairs * cin * cout / us / 1e6:.1f}",
          flush=True)
    if rel > 1e-2:
        e = err
        print("  err by k (first 8):", [float(e[k].max()) for k in range(min(K, 8))])
        print("  err by cin chunk of 16:", [round(float(e[:, c:c + 16].max()), 3) for c in range(0, cin, 16)])
        print("  err by cout chunk of 16:", [round(float(e[:, :, c:c + 16].max()), 3) for c in range(0, cout, 16)])
        print("  dw[0,0,:8]", dw[0, 0, :8].tolist(), "\n  ref[0,0,:8]", ref[0, 0, :8].tolist())
        print("  dw[0,:8,0]", dw[0, :8, 0].tolist(), "\n  ref[0,:8,0]", ref[0, :8, 0].tolist())
    return rel


if __name__ == "__main__":
    shapes = [(200, 1, 64, 64), (1000, 3, 64, 64), (5000, 27, 32, 32), (5000, 27, 64, 64), (5000, 27, 96, 96),
              (5000, 27, 128, 128), (3000, 27, 160, 160), (3000, 27, 192, 192), (4000, 8, 32, 64), (4000, 8, 160, 192),
              (317485, 27, 64, 64), (150000, 27, 96, 96), (60000, 27, 128, 128), (500000, 27, 32, 32)]
    if len(sys.argv) > 1:
        shapes = shapes[: int(sys.argv[1])]
    bad = 0
    for (n, K, ci, co) in shapes:
        bad += case(n, K, ci, co) > 1e-2
    print("WGRAD_CHECK", "FAIL" if bad else "OK")
