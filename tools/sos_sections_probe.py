import sys
from pathlib import Path

import numpy as np, torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from scipy.signal import butter, tf2sos
from waveforms_b200.dsp import sosfilt_device
x = torch.randn(256, 400000, dtype=torch.float64, device='cuda')
out = torch.empty_like(x)
for order in (4, 6, 8):
    sos = tf2sos(*butter(order, 0.3))
    f = lambda: sosfilt_device(sos, x, out=out, mode='scan')
    f(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5): f()
    b.record(); torch.cuda.synchronize()
    print('sections', len(sos), '%.3f ms' % (a.elapsed_time(b) / 5))
