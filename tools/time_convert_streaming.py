"""Times streaming voice conversion (VISinger.voice_conversion_streaming = vsg_model_convert_window per chunk) against one
vsg_model_convert call, full hparams with seeded weights (win_length 1200), and prints the card's name, power limit and
maximum SM clock first.

For B = 1 x T = 4600 and B = 16 x T = 1000, chunks of 100 / 250 / 1000 frames, bf16 and bf16x3:
  * first chunk: device time from the stream's start to its first chunk (event after the first window);
  * streamed total: all windows of one pass, back to back on one stream, against the one-pass call;
  * launches per interior window (vsg_last_launch_count);
  * workspace bytes of the stream (vsg_convert_window_workspace_bytes) against one pass (vsg_convert_workspace_bytes).
Each stream's concatenated output is checked against the one-pass waveform with torch.equal.  CUDA events after one
warm-up pass, best of --reps; L2 is not flushed between passes.

    python tools/time_convert_streaming.py [--reps 3] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from model_inputs import full_hparams  # noqa: E402
from visinger_b200 import _lib  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def model(dev):
    from visinger_b200.models.visinger import VISinger
    hp = full_hparams()
    hp.update(num_spk=4, win_size=1200)
    torch.manual_seed(4321)
    m = VISinger(73, 117, 132, hp).eval()
    with torch.no_grad():
        for f in range(4):
            m.flow.flows[2 * f].post.weight.normal_(0, 0.05)
            m.flow.flows[2 * f].post.bias.normal_(0, 0.05)
    return m.to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_convert_streaming.py measures on a CUDA device; none is available")
    dev = torch.device("cuda:0")
    info = card()
    print(f"card: {info}", flush=True)
    m = model(dev)
    rows = []
    for prec in ("bf16", "bf16x3"):
        m.precision = prec
        code = _lib.precision_code(prec)
        pack = m._convert_pack(dev)
        for B, T in ((1, 4600), (16, 1000)):
            g = torch.Generator().manual_seed(B * T)
            t = torch.arange(T * pack.hop, dtype=torch.float64)
            f = 0.005 + 0.3 * torch.rand(B, 1, generator=g, dtype=torch.float64)
            wav = (0.4 * torch.sin(f * t) + 0.05 * torch.randn(B, T * pack.hop, generator=g, dtype=torch.float64)).float()
            wav = wav.to(dev)
            ln = torch.full((B,), T, dtype=torch.int32, device=dev)
            seeds = torch.arange(1, B + 1, dtype=torch.int64, device=dev)
            kw = dict(spk_id=[0] * B, tgt_spk_id=[1] * B, seeds=seeds)
            ref = m.voice_conversion(wav=wav, lengths=ln, **kw)["wav_out"]
            one = []
            for _ in range(a.reps):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                m.voice_conversion(wav=wav, lengths=ln, **kw)
                e1.record()
                torch.cuda.synchronize()
                one.append(e0.elapsed_time(e1))
            one_ms = min(one)
            one_ws = pack.convert_workspace_bytes(B, T, code)
            for n in (100, 250, 1000):
                n_eff = min(n, T)
                chunks = list(m.voice_conversion_streaming(wav, ln, chunk_frames=n_eff, **kw))   # warm-up + bit check
                exact = torch.equal(torch.cat(chunks, 1), ref)
                it = m.voice_conversion_streaming(wav, ln, chunk_frames=n_eff, **kw)
                next(it)
                if T > 2 * n_eff:
                    next(it)
                launches = m.last_launches
                del it
                first, total = [], []
                for _ in range(a.reps):
                    torch.cuda.synchronize()
                    s, f1, t1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                    s.record()
                    it = m.voice_conversion_streaming(wav, ln, chunk_frames=n_eff, **kw)
                    next(it)
                    f1.record()
                    for _ in it:
                        pass
                    t1.record()
                    torch.cuda.synchronize()
                    first.append(s.elapsed_time(f1))
                    total.append(s.elapsed_time(t1))
                row = dict(precision=prec, B=B, T=T, chunk=n_eff, windows=(T + n_eff - 1) // n_eff,
                           first_chunk_ms=round(min(first), 3), streamed_total_ms=round(min(total), 3),
                           one_pass_ms=round(one_ms, 3), total_over_one_pass=round(min(total) / one_ms, 3),
                           launches_per_window=launches,
                           workspace_bytes=pack.convert_window_workspace_bytes(B, T, n_eff, code),
                           one_pass_workspace_bytes=one_ws, bit_identical=exact)
                rows.append(row)
                print(json.dumps(row), flush=True)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(f"# card: {info}\n")
            for r in rows:
                fh.write(json.dumps(r) + "\n")
    if not all(r["bit_identical"] for r in rows):
        raise SystemExit("a stream differs from its one pass")


if __name__ == "__main__":
    main()
