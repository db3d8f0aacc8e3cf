"""Distance of every convolution launch of a bench step from its bounds (no GPU needed: reads the per-launch CUDA-event
records `bench.py --breakdown-json PATH` writes, committed as profiles/*_breakdown_n1.json).

For each (kind, K, Cin, Cout, rows) shape:
  hbm_us     compulsory HBM bytes / measured HBM peak          (features in + out once, weights, the int32 table)
  gather_us  bytes the kernel must pull through L2 to gather   (P pairs x row bytes; wgrad gathers x and dout)
             at --l2-tbs (default 8 TB/s: an ASSUMED B200 L2 figure, not measured here)
  tensor_us  2*P*Cin*Cout / measured sustained bf16 peak
and the ratio measured / max(bounds).

  python tools/conv_bounds.py profiles/r01d_breakdown_n1.json
"""
import argparse
import collections
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("breakdown")
    ap.add_argument("--l2-tbs", type=float, default=8.0)
    args = ap.parse_args()
    peaks = {"hbm_gbs": 6549.8, "bf16_tflops_sustained": 1354.4}
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        mp = json.load(open(p))
        peaks["hbm_gbs"] = mp.get("hbm_gbs", peaks["hbm_gbs"])
        peaks["bf16_tflops_sustained"] = mp.get("bf16_tflops_sustained", mp.get("bf16_tflops", peaks["bf16_tflops_sustained"]))
    hbm, tf, l2 = peaks["hbm_gbs"] * 1e9, peaks["bf16_tflops_sustained"] * 1e12, args.l2_tbs * 1e12
    recs = json.load(open(args.breakdown))["per_launch"]
    agg = collections.OrderedDict()
    for r in recs:
        if not r["kind"].startswith("conv"):
            continue
        key = (r["kind"], r["K"], r["n_in"], r["n_out"], r["rows_out"])
        a = agg.setdefault(key, [0, 0.0, r])
        a[0] += 1
        a[1] += r["ms"]
    print(f"{'kind':11s} {'K':>3s} {'Cin':>4s} {'Cout':>4s} {'rows':>7s} {'P/N':>5s} {'n':>2s} {'meas_us':>8s} {'hbm_us':>7s} "
          f"{'gather_us':>9s} {'tensor_us':>9s} {'x_bound':>7s}")
    tot = bound = 0.0
    for (kind, K, ci, co, ro), (n, ms, r) in agg.items():
        P, ri, eb = r["pairs"], r.get("rows_in", ro), 2
        by = ri * ci * eb + ro * co * eb + K * ci * co * (4 if kind == "conv_wgrad" else 2) + 4 * K * ro
        gather = P * (ci + co if kind == "conv_wgrad" else ci) * eb
        t = [by / hbm * 1e6, gather / l2 * 1e6, 2.0 * P * ci * co / tf * 1e6]
        us = ms / n * 1e3
        tot += ms
        bound += max(t) * n / 1e3
        print(f"{kind:11s} {K:3d} {ci:4d} {co:4d} {ro:7d} {P / ro:5.1f} {n:2d} {us:8.1f} {t[0]:7.1f} {t[1]:9.1f} {t[2]:9.1f} "
              f"{us / max(t):7.1f}")
    print(f"all convolutions: measured {tot:.2f} ms per step, sum of per-launch bounds {bound:.2f} ms "
          f"({tot / bound:.1f}x); peaks: HBM {hbm / 1e9:.0f} GB/s, bf16 {tf / 1e12:.0f} TFLOP/s, L2 {args.l2_tbs} TB/s (assumed)")


if __name__ == "__main__":
    main()
