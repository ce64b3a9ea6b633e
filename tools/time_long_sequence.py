"""Times the prior network on long utterances, on both sides of the 2048-frame switch of the bf16 attention (one launch at
T <= 2048, key chunks of 2048 plus a combine beyond).  Prints the card's name, power limit and maximum SM clock first.

  * a 4-layer bf16 RelativeEncoder at VISinger sizes (hidden 192, filter 768, 2 heads, kernel 9, window 4, per-frame
    condition as in the FramePriorNetwork), B = 1, T in {1024, 2048, 4096, 8192, 16384};
  * VISinger.forward_graphed in bf16 (full hparams, seeded weights) for one utterance of T in {1280, 4096, 16384} frames,
    in audio-s/s (hop 300 at 24 kHz), with the share of the prior network: eager prior() (through prior sampling) over
    the eager forward.

CUDA events after two warm-up calls; L2 is not flushed between repetitions (back-to-back inference on one utterance).

    python tools/time_long_sequence.py [--reps 5]"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import visinger_oracle as O  # noqa: E402  (weights generator only)
from model_inputs import full_model_mirror, synth_utterances  # noqa: E402
from visinger_b200.modules.rel_transformer import RelativeEncoder  # noqa: E402

FRAME_SEC = 300.0 / 24000.0


def timeit(fn, reps):
    fn()
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_long_sequence.py needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print(f"card: {q.stdout.strip() or q.stderr.strip()}", flush=True)
    dev = torch.device("cuda:0")

    sd = O.synth_rel_encoder_state_dict(O.rel_encoder_param_shapes(192, 768, 2, 4, 9, 4, 1), 5)
    enc = RelativeEncoder(192, 768, 2, 4, kernel_size=9, window_size=4, gin_channels=1)
    enc.load_state_dict(sd)
    enc = enc.to(dev).eval()
    enc.precision = "bf16"
    for T in (1024, 2048, 4096, 8192, 16384):
        gen = torch.Generator().manual_seed(T)
        x = torch.randn(1, 192, T, generator=gen).to(dev)
        g = torch.randn(1, 1, T, generator=gen).to(dev)
        mask = torch.ones(1, 1, T, device=dev)
        ms = timeit(lambda: enc(x, mask, g), a.reps)
        path = "one launch" if T <= 2048 else f"{(T + 2047) // 2048} key chunks + combine"
        print(f"RelativeEncoder bf16, 4 layers, B=1 T={T} ({path}): {ms:.3f} ms, {ms / T * 1e3:.2f} us/frame", flush=True)

    m = full_model_mirror(precision="bf16").to(dev)
    for T in (1280, 4096, 16384):
        batch = synth_utterances(seed=T, n=1, lengths=[T])
        d = {k: v.to(dev) for k, v in batch.items()}
        args = (d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"])
        noise = torch.randn(1, 192, T, generator=torch.Generator().manual_seed(1)).to(dev)
        ms_g = timeit(lambda: m.forward_graphed(*args, spk_id=d["spk_ids"], noise=noise), a.reps)
        ms_e = timeit(lambda: m(*args, spk_id=d["spk_ids"], infer=True, noise=noise), a.reps)
        with torch.no_grad():
            ms_p = timeit(lambda: m.prior(*args, spk_id=d["spk_ids"], noise=noise, sample=True), a.reps)
        audio = T * FRAME_SEC
        print(f"VISinger.forward_graphed bf16, B=1 T={T} ({audio:.1f} s audio): {ms_g:.2f} ms, {audio / (ms_g * 1e-3):.0f} "
              f"audio-s/s; eager forward {ms_e:.2f} ms, eager prior network {ms_p:.2f} ms ({ms_p / ms_e:.1%} of it)",
              flush=True)
        del m.__dict__["_fw_graphs"]
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
