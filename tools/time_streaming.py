"""Times streaming synthesis (HotPath.stream = vsg_infer_zp_window per chunk) against the one-pass vsg_infer_zp on the
shipped flow + decoder (random weights), and prints the card's name, power limit and maximum SM clock first.

For B = 1 x T = 4600 and B = 16 x T = 1000, chunks of 100 / 250 / 500 / 1000 frames, bf16 and bf16x3:
  * first chunk: wall time from the stream's start to its first chunk on the device (event after the first window);
  * streamed total: all windows of one pass, back to back on one stream, against the one-pass call;
  * launches per window (vsg_last_launch_count of an interior window);
  * workspace bytes of the stream (vsg_window_workspace_bytes) against one pass (vsg_workspace_bytes).
Each stream's concatenated output is checked against the one-pass waveform with torch.equal.  CUDA events after one
warm-up pass; L2 is not flushed between passes.

    python tools/time_streaming.py [--reps 3] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from visinger_b200 import _lib  # noqa: E402
from visinger_b200.configs import VISINGER_FLOW, VISINGER_GENERATOR  # noqa: E402
from visinger_b200.models.visinger import HotPath  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def ms(e0, e1):
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_streaming.py measures on a CUDA device; none is available")
    dev = torch.device("cuda:0")
    info = card()
    print(f"card: {info}", flush=True)
    rows = []
    for prec in ("bf16", "bf16x3"):
        hp = HotPath.random_init(VISINGER_FLOW, VISINGER_GENERATOR, dev, precision=prec, seed=1)
        code = _lib.precision_code(prec)
        for B, T in ((1, 4600), (16, 1000)):
            gen = torch.Generator().manual_seed(B * T)
            z_p = torch.randn(B, 192, T, generator=gen).to(dev)
            mask = torch.ones(B, 1, T, device=dev)
            g = (0.1 * torch.randn(B, 256, 1, generator=gen)).to(dev)
            ref, _ = hp.infer_zp(z_p, mask, g)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                hp.infer_zp(z_p, mask, g)
            e1.record()
            torch.cuda.synchronize()
            one_ms = ms(e0, e1) / a.reps
            one_ws = hp._pack().workspace_bytes(B, T, code)
            for n in (100, 250, 500, 1000):
                n_eff = min(n, T)
                chunks = list(hp.stream(z_p, mask, g, n_eff))     # warm-up + bit check
                exact = torch.equal(torch.cat(chunks, 2), ref)
                # launches of an interior window
                it = hp.stream(z_p, mask, g, n_eff)
                next(it)
                if T > n_eff:
                    next(it)
                launches = hp.last_launches
                del it
                first, total = [], []
                for _ in range(a.reps):
                    torch.cuda.synchronize()
                    s, f, t = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                    s.record()
                    it = hp.stream(z_p, mask, g, n_eff)
                    next(it)
                    f.record()
                    for _ in it:
                        pass
                    t.record()
                    torch.cuda.synchronize()
                    first.append(ms(s, f))
                    total.append(ms(s, t))
                row = dict(precision=prec, B=B, T=T, chunk=n_eff, windows=(T + n_eff - 1) // n_eff,
                           first_chunk_ms=round(min(first), 3), streamed_total_ms=round(min(total), 3),
                           one_pass_ms=round(one_ms, 3), total_over_one_pass=round(min(total) / one_ms, 3),
                           launches_per_window=launches,
                           workspace_bytes=hp._pack().window_workspace_bytes(B, T, n_eff, code), one_pass_workspace_bytes=one_ws,
                           bit_identical=exact)
                rows.append(row)
                print(json.dumps(row), flush=True)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(f"# card: {info}\n")
            for r in rows:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
