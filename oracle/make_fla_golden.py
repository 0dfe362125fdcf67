"""Generate tests/golden/fla_long_conv.npz from independent published code.

    python oracle/make_fla_golden.py [path/to/fla/modules/conv/long_conv.py]

`fla/modules/conv/long_conv.py` (flash-linear-attention, MIT) carries the same `fft_conv` and `PositionalEmbedding`
lineage as HyenaDNA's remote code (SURVEY §8c).  It is loaded by file path (default: the installed `fla` package):
importing the `fla` package would pull in its Triton kernels.  Recorded, on inputs drawn from numpy's seeded generator
(the same stream on every platform):
  * `fft_conv(u, k, None, gelu=False)` for u [2, 16, L], k [16, L] at L = 7, 600, 4 097 - the values at a fixed, seeded
    sample of flat positions (every position at L = 7), with the positions;
  * `PositionalEmbedding(emb_dim, max_seq_len).z` at the model's own table size - a seeded sample of its rows.
The first and last position are always in a sample.  `tests/test_oracle.py` checks the oracle against these values.
"""

from __future__ import annotations

import importlib.util
import sys
import sysconfig
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
OUT = ROOT / "tests" / "golden" / "fla_long_conv.npz"
CONV_LENGTHS = (7, 600, 4097)


def conv_inputs(L: int):
    """u [2, 16, L], k [16, L] (float32) of the checked convolution at length L."""
    rng = np.random.default_rng(11 + L)
    u = rng.standard_normal((2, 16, L), dtype=np.float32)
    k = rng.standard_normal((16, L), dtype=np.float32) * np.float32(0.1)
    return u, k


def sample_positions(n: int, k: int) -> np.ndarray:
    if n <= k:
        return np.arange(n, dtype=np.int32)
    idx = np.random.default_rng(n).choice(n, k, replace=False)
    return np.unique(np.concatenate([idx, [0, n - 1]])).astype(np.int32)


def main(path: Path) -> None:
    from chimeralm_b200.config import HyenaConfig

    spec = importlib.util.spec_from_file_location("_fla_long_conv", path)
    fla = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fla)
    out = {}
    for L in CONV_LENGTHS:
        u, k = conv_inputs(L)
        y = fla.fft_conv(torch.from_numpy(u), torch.from_numpy(k), None, gelu=False).numpy().reshape(-1)
        pos = sample_positions(y.size, 4096)
        out[f"conv_pos_{L}"], out[f"conv_{L}"] = pos, y[pos]
    cfg = HyenaConfig()
    z = fla.PositionalEmbedding(cfg.emb_dim, cfg.max_seq_len).z.detach().numpy()
    rows = sample_positions(z.shape[1], 2048)
    out["z_shape"], out["z_rows"], out["z"] = np.array(z.shape), rows, z[0, rows]
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT} ({OUT.stat().st_size} bytes)")


if __name__ == "__main__":
    main(Path(sys.argv[1]) if len(sys.argv) > 1
         else Path(sysconfig.get_paths()["purelib"]) / "fla" / "modules" / "conv" / "long_conv.py")
