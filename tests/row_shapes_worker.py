"""Real-input envelopes at several row shapes, for comparing the channelizer's two-rows-per-thread form
(ACB_REAL_ROWS=2, read once per process) with the default four-rows form and the oracle.

Run as a script with ACB_REAL_ROWS=2 in its environment: prints one JSON line with a digest of every case's envelope
and the names of the channelizer kernels that ran.  tests/test_gpu_row_shapes.py imports the case definitions."""
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from acarsdec_b200 import api  # noqa: E402
from common import ragged_sizes, stream_envelope  # noqa: E402

FLAG_REAL = 2
# name: (K, taps, channels)
CASES = {
    "K200": (200, 200, 9),
    "K204": (204, 204, 17),
    "K2048": (2048, 2048, 17),
    "K200_taps21": (200, 21, 9),
}


def real_case(name: str):
    """(K, taps, x (1, n) float32, table (nch, 2*taps) float32, submit lengths, max_blocks), the same on every call."""
    K, taps, nch = CASES[name]
    rng = np.random.default_rng([K, taps, nch])
    nrows = 2 * 1024 + 517
    x = (rng.standard_normal((1, nrows * K + K // 2 + 1)) * 0.25).astype(np.float32)
    wf = (rng.standard_normal((nch, 2 * taps)) / taps).astype(np.float32)
    max_blocks = nrows // 1024 + 2
    return K, taps, x, wf, ragged_sizes(K, x.shape[1], (max_blocks * 1024 - 1) * K, seed=K + taps), max_blocks


def run_real(name: str) -> np.ndarray:
    """Stream 0's envelope (nout, nch) through a real-input context with the case's table."""
    K, taps, x, wf, sizes, max_blocks = real_case(name)
    with api.Context(K, 1, wf.shape[0], max_blocks, flags=FLAG_REAL, taps=taps if taps < K else 0) as ctx:
        ctx.set_wf(0, wf)
        env, _ = stream_envelope(ctx, ctx.submit_real, x, sizes)
    return env[0]


def digest(env: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(env, dtype=np.float32).tobytes()).hexdigest()


def main():
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    out = {}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for name in CASES:
            out[name] = digest(run_real(name))
    kernels = sorted({e.key for e in prof.key_averages() if "k_channelize" in e.key})
    print(json.dumps({"digests": out, "kernels": kernels}), flush=True)


if __name__ == "__main__":
    main()
