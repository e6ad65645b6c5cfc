"""Clock64 timeline of one persistent CTA (blockIdx.x == 40) of attn_bwd_dq_cc_kernel through the debug hook (GPU box).

python tools/attn_timeline.py [debug mode: 16 = soft mbarrier timeouts]  -> per-tile stamps relative to the first one (cycles); column = global tile
index of the CTA (item * ntiles + tile).  Events (chexpert_b200/csrc/attn_cc.cu, TL_STAMP):
   0 S: loop top   1 S: K tile landed   2 S: slot free   3 S: issued+committed     4 G: loop top   5 G: dS ready   6 G: issued
   7 WG: waiting for S'   8 WG: S' ready   9 WG: S' in registers   10 WG: math done   11 WG: dS stored, arrived
  12 drain, per item (warpgroup 0): final wait begin / final seen / accumulator free / bulk store issued
  14 TMA: stage free
"""
import ctypes
import os
import sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import chexpert_b200 as cb  # noqa: E402
from chexpert_b200 import _lib  # noqa: E402
from bench import SHAPES    # noqa: E402

EV, COLS = 16, 96
cin, hin, cout, dk, dv = SHAPES['T1']
H = hin // 2
torch.manual_seed(0)
m = cb.AAConv2d(cin, cout, 3, 2, dk, dv, 8, True, (H, H), precision='bf16').cuda()
x = torch.relu(torch.randn(16, cin, hin, hin, device='cuda')).requires_grad_(True)
dy = torch.randn(16, cout, H, H, device='cuda')
buf = torch.zeros(EV * COLS, dtype=torch.int64, device='cuda')
lib = _lib.load()
if len(sys.argv) > 1:
    lib.aaconv_debug_set_mode(int(sys.argv[1]))
for it in range(3):
    m.zero_grad(set_to_none=True)
    x.grad = None
    y = m(x)
    if it == 2:
        lib.aaconv_debug_set_timeline(ctypes.c_void_p(buf.data_ptr()))
    y.backward(dy)
torch.cuda.synchronize()
lib.aaconv_debug_set_timeline(None)
lib.aaconv_debug_set_mode(0)
t = buf.cpu().reshape(EV, COLS)
t0 = int(t[t > 0].min())
names = ['TMA:free', 'S:top', 'S:landed', 'S:slot', 'S:issued', 'wg:wait', 'wg:S rdy', 'wg:in reg', 'wg:math', 'wg:arrive', 'G:top', 'G:dS rdy', 'G:issued']
order = [14, 0, 1, 2, 3, 7, 8, 9, 10, 11, 4, 5, 6]
print('tile ' + ' '.join(f'{n:>9s}' for n in names))
for j in range(0, 80):
    print(f'{j:4d} ' + ' '.join(f'{(int(t[e, j]) - t0) if t[e, j] > 0 else -1:9d}' for e in order))
print('drain per item (warpgroup 0): [wait final, final seen, accumulator free, store issued]')
for i in range(0, 4):
    print(i, [int(v) - t0 if v > 0 else -1 for v in t[12, i * 4:i * 4 + 4]])
