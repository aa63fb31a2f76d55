"""Device sampler at the C-ABI, without a GPU: the new symbols are exported, the limits agree between the header and
the Python binding, and the single-op entry point refuses to run (no CPU fallback) when no device is visible."""
import os
import re
import subprocess
import sys
from pathlib import Path

from crowdllama_b200 import engine as eng

ROOT = Path(__file__).resolve().parents[1]

_NO_DEVICE_CHILD = r"""
import numpy as np
from crowdllama_b200 import engine as eng
sp = eng.ollama_default_sampling(seed=1)
try:
    eng.op_sample(np.zeros((1, 300), np.float32), [sp], [[5, 6]], [0])
except eng.EngineError as ex:
    assert ex.status == eng.CL_ERR_NO_DEVICE, ex
else:
    raise SystemExit("cl_op_sample ran without a device")
"""


def test_sampler_symbols_exported_and_declared():
    L = eng.lib()
    header = (ROOT / "include" / "clengine.h").read_text()
    for name in ("cl_op_sample", "cl_decode_sample_batch"):
        assert name in eng.EXPORTS
        assert hasattr(L, name)
        assert re.search(rf"\b{name}\(", header)


def test_sampler_limits_match_header():
    header = (ROOT / "include" / "clengine.h").read_text()
    top_k = int(re.search(r"#define CL_SAMPLE_MAX_TOP_K (\d+)", header).group(1))
    window = int(re.search(r"#define CL_SAMPLE_MAX_WINDOW (\d+)", header).group(1))
    assert (top_k, window) == (eng.SAMPLE_MAX_TOP_K, eng.SAMPLE_MAX_WINDOW)
    # the Ollama defaults (top_k 40, repeat_last_n 64) fit the device sampler
    sp = eng.ollama_default_sampling()
    assert 1 <= sp.top_k <= top_k and 0 < sp.repeat_last_n <= window


def test_op_sample_without_device_returns_no_device():
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHILD], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:] + r.stdout[-2000:]
