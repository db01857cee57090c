"""Sweep of K~^-1 = V V^T: the DMMA GEMM against the emulated INT8 product (tools/bin/ozaki_check compare)
at n = 2048 .. 32768, on V = L^-T of a Matern-5/2 Gram.  The INT8 denominator is torch._int_mm at
8192^3 measured in the same run.  The smallest n where the emulated product wins sets kOzakiMinN
(pygp_b200/csrc/chol.cu).

    python tools/ozaki_sweep.py [--out FILE] [--sizes 2048,...] [--feed]

--feed times the residue products alone instead (tools/bin/ozaki_check feed): operands as laid out in HBM,
and the same items reading an L2-resident window.  If the resident run is much faster, the operand feed
limits the products.
"""

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def int8_tops():
    import torch
    a = torch.randint(-128, 128, (8192, 8192), dtype=torch.int8, device='cuda')
    b = torch.randint(-128, 128, (8192, 8192), dtype=torch.int8, device='cuda')
    for _ in range(3):
        torch._int_mm(a, b)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record()
    for _ in range(reps):
        torch._int_mm(a, b)
    e1.record()
    torch.cuda.synchronize()
    return 2 * 8192**3 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out')
    ap.add_argument('--sizes', default='2048,4096,8192,16384,32768')
    ap.add_argument('--feed', action='store_true')
    args = ap.parse_args()
    lines = []
    tops = int8_tops()
    lines.append('torch._int_mm 8192^3: %.1f INT8 TOP/s' % tops)
    for n in [int(s) for s in args.sizes.split(',')]:
        mode = 'feed' if args.feed else 'compare'
        p = subprocess.run([os.path.join(ROOT, 'tools', 'bin', 'ozaki_check'), mode, str(n), '3'],
                           capture_output=True, text=True)
        if p.returncode not in (0, 1):
            sys.exit(p.stdout + p.stderr)
        rec = json.loads(p.stdout.strip().splitlines()[-1])
        rec['products_frac_of_int_mm'] = rec['products_int8_tops'] / tops
        if args.feed:
            rec['resident_frac_of_int_mm'] = rec['resident_int8_tops'] / tops
        lines.append(json.dumps(rec))
    text = '\n'.join(lines) + '\n'
    sys.stdout.write(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
