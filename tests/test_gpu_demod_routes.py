"""GPU: each route of a DeModulate call launches the symbol stage as often as the call plan says (tests/symsync_dispatch.py
`route` / `chunks`): symsync_decode_kernel once per time chunk on the fused routes, decode_kernel once on the unfused ones.
The value tests pass whatever the chunk count, so only this pins the pipeline to its chunks."""
import ast
import os
import re
import subprocess
import sys

import pytest

import symsync_dispatch as sd

pytestmark = pytest.mark.gpu

# The profiler runs in a child process: once a torch.profiler session has been opened in the pytest process, the profiled
# tests of other files that run later in the same process recorded no kernels at all.
_CHILD = """
import sys
sys.path[:0] = {paths!r}
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
import qpsk_modulator_demodulator_b200 as Q
from symsync_dispatch import ROUTE_ROWS
Q.set_device({device})
calls = {{}}
for name, r in ROUTE_ROWS.items():
    C, L = r["channels"], r["L"]
    x = np.random.default_rng(1).standard_normal((C, 2 * L)).astype(np.float32)
    d = Q.QPSKDeModulator(r["fs"], r["rs"], 0.35, 10, use_fll=r.get("use_fll", False), channels=C)
    if r.get("eq"):
        d.set_equalizer(11, 0.01)
    if r.get("cs16"):
        x16 = np.clip(np.round(x * 8000.0), -32768, 32767).astype(np.int16)
        calls[name] = lambda d=d, x16=x16: d.DeModulateBytesCs16(x16, 1.0 / 8000.0, b"START", b"END")
    elif r.get("host"):
        calls[name] = lambda d=d, x=x: d.DeModulate(x)
    else:
        dx = torch.from_numpy(x).cuda()
        cap = d.bits_bound(2 * L)
        bits = torch.zeros((C, cap), dtype=torch.uint8, device="cuda")
        nb = torch.zeros(C, dtype=torch.int64, device="cuda")
        calls[name] = lambda d=d, dx=dx, L=L, cap=cap, bits=bits, nb=nb: d.demod_bits_dev(
            dx.data_ptr(), 2 * L, 2 * L, bits.data_ptr(), cap, nb.data_ptr())
mark = torch.zeros(1, device="cuda")
torch.cuda.synchronize()
# one profiler session; a fill kernel between two calls marks where one call's kernels end
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for call in calls.values():
        call()
        torch.cuda.synchronize()
        mark.fill_(1.0)
        torch.cuda.synchronize()
ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start)
names = [e.name for e in ev if not e.name.startswith("Memcpy") and not e.name.startswith("Memset")]
per_call, cur = [], []
for n in names:
    if "FillFunctor" in n:
        per_call.append(cur)
        cur = []
    else:
        cur.append(n)
assert len(per_call) == len(calls) and all(per_call), per_call
print("KERNELS", repr(dict(zip(calls, per_call))))
"""


@pytest.fixture(scope="module")
def launched(gpu):
    here = os.path.dirname(os.path.abspath(__file__))
    code = _CHILD.format(paths=[os.path.dirname(here), here], device=int(os.environ.get("LOCAL_RANK", "0")))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("KERNELS ")][-1]
    return ast.literal_eval(line[len("KERNELS "):])


@pytest.mark.parametrize("row", list(sd.ROUTE_ROWS))
def test_symbol_stage_runs_once_per_chunk(launched, row):
    route, chunks = sd.route(sd.ROUTE_ROWS[row])
    names = launched[row]
    n_symsync = sum(1 for n in names if sd.SYMSYNC_RE.search(n))
    n_decode = sum(1 for n in names if re.search(r"(?<!\w)decode_kernel", n))
    if route == "unfused":
        assert (n_symsync, n_decode) == (0, 1), (route, names)
    else:
        assert (n_symsync, n_decode) == (chunks, 0), (route, chunks, names)
