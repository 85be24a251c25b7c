"""A downsampling block's input gradient: lbt_conv_i8_dgrad_block (one launch) against the two lbt_conv_i8_dgrad_strided
launches it replaces (1x1/2 shortcut, then the 3x3/2 main convolution with the shortcut's dX as addend), at ResNet-18's three
block shapes.  Each variant is captured into a CUDA graph of `reps` calls; the graphs are replayed alternately and timed
with CUDA events.  Prints one JSON line per shape: microseconds per call (median of the rounds), algorithmic bytes and ops,
the share of the larger data-sheet floor, and whether both outputs are equal.

    python benchmarks/dgrad_block_bench.py [--batch 256] [--rounds 7] [--reps 20]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lbt_b200 import _lib, dfxp as D, quantizer as Q  # noqa: E402

HBM_BPS = 7.7e12     # HGX B200 data sheet, one GPU
I8_OPS = 4.5e15      # dense 8-bit tensor rate, same source

SHAPES = [('stage2', 56, 64, 128), ('stage3', 28, 128, 256), ('stage4', 14, 256, 512)]   # block input H = W, Cin, Cout


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = 'unknown'
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--reps', type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('dgrad_block_bench: needs a GPU')
    name, pl = card()
    S8 = Q.MANT_S8
    rng = np.random.default_rng(0)
    for tag, H, Cin, Cout in SHAPES:
        N, W, s, k = a.batch, H, 2, 3
        OH, pt, _ = D.same_pad(H, k, s)
        OW, pl_, _ = D.same_pad(W, k, s)
        wm = torch.from_numpy(rng.integers(-128, 128, (k, k, Cin, Cout), dtype=np.int8)).cuda()
        perm = torch.tensor(D._class_perm(k, k, s, s), device='cuda')
        w2 = wm.view(k * k, Cin, Cout).index_select(0, perm).permute(1, 0, 2).reshape(Cin, k * k * Cout).contiguous()
        ws = torch.from_numpy(rng.integers(-128, 128, (Cin, Cout), dtype=np.int8)).cuda()
        g = torch.from_numpy(rng.integers(-128, 128, (N, OH, OW, Cout), dtype=np.int8)).cuda()
        gs = torch.from_numpy(rng.integers(-128, 128, (N, OH, OW, Cout), dtype=np.int8)).cuda()
        ib = torch.tensor([2, 1, 0, 1], dtype=torch.int32, device='cuda')
        dx_old = torch.empty(N, H, W, Cin, device='cuda')
        dx_s = torch.empty(N, H, W, Cin, device='cuda')
        dx_new = torch.empty(N, H, W, Cin, device='cuda')
        st = lambda: torch.cuda.current_stream().cuda_stream   # noqa: E731

        def old():
            _lib.call('lbt_conv_i8_dgrad_strided', gs.data_ptr(), S8, N, OH, OW, Cout, ws.data_ptr(), S8, Cout, Cin, 1, 1, s, s, 0, 0,
                      H, W, ib[2:3].data_ptr(), ib[3:4].data_ptr(), -13, dx_s.data_ptr(), Cin, None, st())
            _lib.call('lbt_conv_i8_dgrad_strided', g.data_ptr(), S8, N, OH, OW, Cout, w2.data_ptr(), S8, w2.stride(0), Cin, k, k, s, s,
                      pt, pl_, H, W, ib[0:1].data_ptr(), ib[1:2].data_ptr(), -14, dx_old.data_ptr(), Cin, dx_s.data_ptr(), st())

        def new():
            _lib.call('lbt_conv_i8_dgrad_block', g.data_ptr(), S8, N, OH, OW, Cout, w2.data_ptr(), S8, w2.stride(0), Cin, k, k, s, s,
                      pt, pl_, H, W, ib[0:1].data_ptr(), ib[1:2].data_ptr(), -14, gs.data_ptr(), S8, OH, OW, Cout, ws.data_ptr(), S8,
                      Cout, ib[2:3].data_ptr(), ib[3:4].data_ptr(), -13, dx_new.data_ptr(), Cin, None, st())

        graphs = {}
        for key, fn in (('old', old), ('new', new)):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    fn()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                for _ in range(a.reps):
                    fn()
            graphs[key] = gr
        times = {'old': [], 'new': []}
        for _ in range(a.rounds):
            for key in ('old', 'new'):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                graphs[key].replay()
                e1.record()
                torch.cuda.synchronize()
                times[key].append(e0.elapsed_time(e1) * 1e3 / a.reps)
        equal = bool(torch.equal(dx_old, dx_new))
        ops = 2 * N * OH * OW * Cin * (k * k * Cout + Cout)
        byts = {'new': g.numel() + gs.numel() + w2.numel() + ws.numel() + 4 * dx_new.numel(),
                'old': g.numel() + gs.numel() + w2.numel() + ws.numel() + 4 * dx_new.numel() * 3}
        floor = max(byts['new'] / HBM_BPS, ops / I8_OPS)
        bound = 'HBM' if byts['new'] / HBM_BPS >= ops / I8_OPS else 'tensor'
        row = dict(shape=tag, batch=N, H=H, Cin=Cin, Cout=Cout, card=name, power_limit=pl, equal=equal, ops=ops,
                   floor_us=round(floor * 1e6, 1), floor_bound=bound)
        for key in ('old', 'new'):
            med = statistics.median(times[key])
            row[key + '_us'] = round(med, 1)
            row[key + '_us_spread'] = round(max(times[key]) - min(times[key]), 1)
            row[key + '_bytes'] = byts[key]
            row[key + '_share_of_floor'] = round(floor * 1e6 / med, 3)
        row['speedup'] = round(row['old_us'] / row['new_us'], 2)
        print(json.dumps(row), flush=True)
    assert _lib.lib().lbt_conv_debug_error() == 0


if __name__ == '__main__':
    main()
