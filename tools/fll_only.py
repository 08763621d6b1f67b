"""Time the FLL kernel alone: python tools/fll_only.py [channels] [samples] [taps] (CUDA events on the launching stream)."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import qpsk_modulator_demodulator_b200 as Q
C = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
L = int(sys.argv[2]) if len(sys.argv) > 2 else 4196
N = int(sys.argv[3]) if len(sys.argv) > 3 else 40
Q.set_device(0)
ts = torch.cuda.Stream(); torch.cuda.set_stream(ts); s = ts.cuda_stream
g = torch.Generator(device="cuda"); g.manual_seed(1)
x = (torch.rand(C, 2 * L, device="cuda", generator=g) - 0.5)
y = torch.empty_like(x)
f = Q.FLLBandEdgeFilter(4.0, 0.35, N, 0.01, channels=C)
for _ in range(3):
    f.process_dev(x.data_ptr(), y.data_ptr(), 2 * L, stream=s)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
reps = 5
e0.record(ts)
for _ in range(reps):
    f.process_dev(x.data_ptr(), y.data_ptr(), 2 * L, stream=s)
e1.record(ts); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / reps
print(json.dumps({"channels": C, "samples": L, "taps": N, "ms": ms, "cycles_per_sample_at_1965MHz": ms * 1e-3 * 1.965e9 / L,
                  "msamples_s": C * L / ms / 1e3}))
