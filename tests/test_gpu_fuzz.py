"""A seeded slice of the randomised parity soaks (tools/fuzz_path.py, tools/fuzz_fll.py) in the GPU suite: random design
parameters, sizes, channel counts and chunkings through the C ABI against the oracle on the same chunks."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("tool,args,env", [("fuzz_path.py", ["16", "5"], {}), ("fuzz_fll.py", ["30", "5"], {}),
                                           # two lanes per stream (csrc/fll_pair.cu): 10 or 40 taps from 5120 streams
                                           ("fuzz_fll.py", ["40", "7"], {"FUZZ_SIZES": "10,40", "FUZZ_CHANNELS": "5120,5137"})])
def test_fuzz_slice(gpu, tool, args, env):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", tool)] + args, capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, **env))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "0 mismatching" in r.stdout
