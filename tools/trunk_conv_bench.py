#!/usr/bin/env python
"""SimpleNN's trunk convolutions: the tcgen05 trunk kernel (dbaz_nn_trunk_conv) against cuDNN on the same folded weights,
per batch size of the adaptive ladder, one layer at a time (conv1 = padded 3x3, conv4 = unpadded) and for the whole
evaluator (FusedSimpleNN with and without the kernel).  CUDA events over graph replays; the card's name and power limit
are read in the same run.
    python tools/trunk_conv_bench.py [--board 3x3] [--games 4096]"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dotsboxesaz_b200 import engine
from dotsboxesaz_b200.dots_boxes.dots_boxes_nn import SimpleNN
from dotsboxesaz_b200.nn import FusedSimpleNN, _conv_add_relu, _conv_relu, trunk_conv_bias, trunk_conv_pack

ap = argparse.ArgumentParser()
ap.add_argument("--board", default="3x3")
ap.add_argument("--games", type=int, default=4096)
ap.add_argument("--ladder-steps", type=int, default=16)
args = ap.parse_args()
L, C = (int(v) for v in args.board.split("x"))
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30)
    print("gpu:", q.stdout.strip().splitlines()[torch.cuda.current_device()])
except Exception as e:  # the timings stand without it, but say so
    print("gpu: nvidia-smi unavailable (%s); device %s" % (e, torch.cuda.get_device_name()))
torch.manual_seed(0)
model = SimpleNN(board=(L, C)).eval()
eng = engine.Engine((L, C), n_games=args.games, max_nodes=16)
eng.LADDER_STEPS = args.ladder_steps
eng.leaf_states.copy_(eng.new_states(args.games))
plans = {"kernel": FusedSimpleNN(model, eng), "cudnn": FusedSimpleNN(model, eng, use_trunk=False)}
assert len(plans["kernel"].trunk) == 3 and plans["cudnn"].trunk is None
rows_list = sorted(set(eng._ladder(plans["kernel"])) | {64, 128, args.games})


def timed(fn, reps=4):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / (5 * reps) * 1e3


kp, cp = plans["kernel"], plans["cudnn"]
kp.TRUNK_MIN_ROWS = 0  # the kernel at every rung here, to show where the plan's threshold falls
x1 = torch.rand((args.games, L + 1, C + 1, 256), device=eng.device).to(torch.bfloat16)
kp.stem_out.copy_(x1)  # the trunk kernel's input buffer (conv1 reads the stem output)
xc = x1.permute(0, 3, 1, 2)
(w1, b1, z1, p1), (w4, b4, _, p4) = cp.convs[0], cp.convs[3]
# conv4 (unpadded) through the kernel too, on the same folded weights as the cuDNN plan's
t_in = torch.rand_like(kp.trunk_out)
t_in_c = t_in.permute(0, 3, 1, 2)
bpos4 = torch.zeros((256, L - 1, C - 1), device=eng.device)
plan4 = eng.nn_trunk_conv_plan(t_in, torch.empty((args.games, L - 1, C - 1, 256), dtype=torch.bfloat16, device=eng.device),
                               trunk_conv_pack(w4.float()), *trunk_conv_bias(b4.float(), bpos4, 0), 0)
real = sum(len(t) for t in engine.trunk_conv_taps(L + 1, C + 1, 1)[2])
print("conv1 taps: %d of %d in the board (%.1f %%)" % (real, 9 * (L + 1) * (C + 1), 100.0 * real / (9 * (L + 1) * (C + 1))))
print("| rows | conv1 kernel us | conv1 cuDNN us | conv4 kernel us | conv4 cuDNN us | evaluator kernel us | evaluator cuDNN us | evaluator speed-up |")
print("|---|---|---|---|---|---|---|---|")
for rows in rows_list:
    k1 = timed(lambda: eng.nn_trunk_conv(kp.trunk_plans[0], rows))
    c1 = timed(lambda: _conv_add_relu(xc[:rows], w1, z1[:rows], b1, p1))
    k4 = timed(lambda: eng.nn_trunk_conv(plan4, rows))
    c4 = timed(lambda: _conv_relu(t_in_c[:rows], w4, b4, p4))
    eng._batch_rows = rows
    ek, ec = timed(lambda: kp(eng)), timed(lambda: cp(eng))
    eng._batch_rows = None
    print("| %d | %.1f | %.1f | %.1f | %.1f | %.1f | %.1f | %.2fx |" % (rows, k1, c1, k4, c4, ek, ec, ec / ek), flush=True)
eng.close()
