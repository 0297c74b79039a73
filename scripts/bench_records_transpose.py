"""Times emei_records_transpose (time-major rollout records [T, n, ...] -> env-major [n, T, ...], DESIGN.md 4.4) against
torch's ``x.transpose(0, 1).contiguous()`` on the same tensor, for every observation-record width:

  16 bytes  float32 rows of 4 (cart-pole, inverted pendulum, charged ball)
  24 bytes  float32 rows of 6 (inverted double pendulum)
  32 bytes  float64 rows of 4
  48 bytes  float64 rows of 6 (inverted double pendulum in float64: the headline case)

at T = 1000 steps and n = 2^16 envs (3.1 GB each way at 48 bytes, far beyond the 126 MB L2, so every pass reads HBM).
Each line carries the bytes moved (read once + written once), the achieved rate, the time a copy of those bytes would
take at the data sheet's 7.7 TB/s (its share of the measured time), and torch's time and rate.  Both outputs are
compared bit for bit before timing.  Card name and power limit are read in the same run.

    python scripts/bench_records_transpose.py [--out profiles/r06_bench_records_transpose.jsonl]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from emei_b200 import _lib  # noqa: E402
from bench_autodiff import card, time_ms  # noqa: E402

HBM_DATASHEET_BPS = 7.7e12
T, N = 1000, 1 << 16
ROWS = ((torch.float32, 4), (torch.float32, 6), (torch.float64, 4), (torch.float64, 6))


def run(dtype, D, iters):
    dev = "cuda:0"
    x = torch.randn((T, N, D), dtype=dtype, device=dev)
    out = torch.empty((N, T, D), dtype=dtype, device=dev)
    elem = D * x.element_size()
    stream = torch.cuda.current_stream().cuda_stream

    def ours():
        _lib.call("emei_records_transpose", x.data_ptr(), out.data_ptr(), T, N, elem, stream)

    def theirs():
        return x.transpose(0, 1).contiguous()

    ours()
    same = bool(torch.equal(out, theirs()))
    ms = time_ms(ours, iters)
    ms_torch = time_ms(theirs, iters)
    nbytes = 2 * x.numel() * x.element_size()
    bound_ms = nbytes / HBM_DATASHEET_BPS * 1e3
    del x, out
    torch.cuda.empty_cache()
    return dict(what="records_transpose", dtype=str(dtype).split(".")[-1], D=D, elem_bytes=elem, T=T, n=N, bytes_moved=nbytes,
                ms=round(ms, 4), TBps=round(nbytes / ms / 1e9, 3), datasheet_bound_ms=round(bound_ms, 4),
                share_of_datasheet_hbm=round(bound_ms / ms, 3), torch_ms=round(ms_torch, 4),
                torch_TBps=round(nbytes / ms_torch / 1e9, 3), speedup_vs_torch=round(ms_torch / ms, 2), bit_identical_to_torch=same)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_bench_records_transpose.jsonl"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_records_transpose.py measures on a CUDA device; there is none")
    name, power = card()
    lines = [json.dumps(dict(card=name, power_limit_and_max_sm_clock=power, hbm_datasheet_Bps=HBM_DATASHEET_BPS))]
    print(lines[0], flush=True)
    for dtype, D in ROWS:
        lines.append(json.dumps(run(dtype, D, args.iters)))
        print(lines[-1], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
