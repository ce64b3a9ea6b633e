#!/usr/bin/env python
"""bench.py -- audio-seconds synthesised per wall-second on the VISinger inference hot path.

    python bench.py --gpus N --steps K --warmup W [--precision bf16|fp32] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (models/visinger.py:107-111 of the reference: prior sampling ->
ResidualCouplingBlock reverse -> HiFi-GAN Generator) over one batch of synthetic input: B=16 utterances
x T=1000 latent frames = 200 s of 24 kHz audio per GPU per step (BASELINE.json configs[1]+[2], the shapes
the metric's roofline is quoted on), random weights of config/models/visinger.yaml shape.

  value     device-resident throughput: inputs already in HBM, CUDA events around K steps, max over ranks
  e2e       the same through the public module API with pinned HOST buffers: H2D of (mu_p, logs_p, noise,
            mask, g) and D2H of the waveform inside the timed region, every step
  roofline  decoder convolutions (the dominant kernels): algorithmic FLOPs (SURVEY.md 8d:
            333 911 680 FLOP per latent frame) / CUDA-event time of the generator region
  cpu_baseline  the oracle port of the reference's CPU path on this box's host cores (rank 0, N=1 only)
  parity_mode   (N=1) the same workload in bf16x3 -- the tensor-core mode that meets the fp32 tolerances (decoder on two
            bf16 planes per value, flow on three; no CUDA-core convolution) -- with its measured distance to the CPU
            oracle on a full-length utterance
  bf16      (N=1) the headline mode's distance to the CPU oracle on the same full-length utterance: relative L2,
            max-abs and the reference's own log-mel L1 (MelSpectrogramFixed, utils/audio/mel_processing.py:28-38)
  full_model  (N=1) BASELINE.json configs[3]: the whole VISinger.forward(infer=True) -- native transformer stacks of the prior
            network, length regulator, fused frame-prior head, flow, decoder -- on 64 mixed-length utterances, host
            tokens -> host waveforms, with the bf16 mode's distance to the fp32 mode on the same padded batch
  sharded   BASELINE.json configs[4]: 512 mixed-length utterances (log-normal lengths, seed 1234) -> length buckets over
            the whole list -> LPT assignment of the batches to ranks -> per-rank serving loop -> pinned host results;
            strong scaling (fixed total work), with padding overhead and per-rank imbalance

Multi-GPU: utterances are independent, so ranks shard by utterance with no collective on the data path
(weak scaling: every rank runs the same per-GPU batch); torch.distributed is used only for the barrier
and the max-over-ranks of the device-measured time.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FRAME_SEC = 300.0 / 24000.0                 # hop_size / sample_rate (preprocess.yaml:9,11)
DEC_FLOP_PER_FRAME = 333_911_680            # SURVEY.md 8(d) / Appendix A.2
FLOW_FLOP_PER_FRAME = 14_155_776            # SURVEY.md 8(d) / Appendix A.1
METRIC = "audio-sec synthesized per wall-sec"
UNIT = "audio-s/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("VSG_BENCH_PRECISION", "bf16"), choices=["bf16", "bf16x3", "fp32"])
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels directly instead of replaying a CUDA graph")
    ap.add_argument("--l2-mb", type=int, default=-1, help="L2-resident batch tiling target (MB per tensor; 0 = off)")
    ap.add_argument("--no-pdl", action="store_true", help="disable programmatic dependent launch of the conv kernels")
    ap.add_argument("--no-fuse", action="store_true", help="disable the fused ResBlock pair kernel")
    ap.add_argument("--no-merge-ups", action="store_true", help="one launch per polyphase of the transposed convs")
    ap.add_argument("--no-split-n", action="store_true", help="keep N = 256 tiles whole (no 2 x 128 split)")
    ap.add_argument("--one-epi-set", action="store_true", help="a single set of 4 epilogue warps per CTA")
    ap.add_argument("--generic-epilogue", action="store_true", help="never use the signature-specialised kernels")
    ap.add_argument("--no-parity-mode", action="store_true", help="skip the bf16x3 timing / parity block")
    ap.add_argument("--no-sharded", action="store_true", help="skip the 512-utterance sharded sweep (configs[4])")
    ap.add_argument("--no-full-model", action="store_true", help="skip the 64-utterance full-model leg (configs[3])")
    ap.add_argument("--no-chain-streams", action="store_true", help="run the resblock chains of a stage one after the other")
    ap.add_argument("--two-streams", action="store_true", help="store raw and activated copies of the resblock stream")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each tensor of `arrays` as out_dir/<name>.npy in float32.  Should they hold more than DUMP_BYTES in all,
    each is cut to the same fraction of its elements: a fixed sample (seed 0) of its flat indices, in index order, 1-D."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_BYTES - 4096 * len(arrays)           # room for the .npy headers
    for name, a in arrays.items():
        if total > budget:
            idx = np.random.default_rng(0).choice(a.size, a.size * budget // total, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_sustained=d.get("bf16_tflops_sustained", 1390.4), bf16_burst=d.get("bf16_tflops", 1674.5),
                    hbm=d.get("hbm_gbs", 6549.8), src="measured (MEASURED_PEAKS.json)")
    return dict(bf16_sustained=1400.0, bf16_burst=1590.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(sm)}


REF_DIR = os.path.join(ROOT, "baseline", "_ref")     # vendored by __graft_entry__.build() (git-ignored; travels with gpurun)


def bench_weights_and_inputs(B, T, rank=0):
    """The workload both arms run: random-init weights of config/models/visinger.yaml shape (torch default init through
    the module mirrors' constructors, seed 1234, `post` re-randomised) and the seeded inputs of `rank`."""
    import torch
    from visinger_b200.configs import VISINGER_FLOW as FLOW_FULL, VISINGER_GENERATOR as GEN_FULL
    from visinger_b200.models.visinger import HotPath
    hp = HotPath.random_init(FLOW_FULL, GEN_FULL, "cpu", precision="fp32", seed=1234)
    gen_in = torch.Generator().manual_seed(rank)
    x = torch.randn(B, 192, T, generator=gen_in)                 # prior mean
    g = 0.1 * torch.randn(B, 256, 1, generator=gen_in)           # speaker embedding
    mask = torch.ones(B, 1, T)                                   # full-length utterances
    logs = torch.full_like(x, -1.0)
    noise = torch.randn(x.shape, generator=torch.Generator().manual_seed(100 + rank))
    return hp, (x, logs, noise, mask, g)


class CpuHotPath:
    """The reference's CPU implementation of the path for one batch: the REAL reference modules when the vendored copy
    (baseline/_ref) is present -- `ResidualCouplingBlock` (modules/visinger/flow.py:15) and `Generator`
    (modules/visinger/decoder.py:13) driven exactly as models/visinger.py:107-111 drives them -- else the oracle port."""

    def __init__(self, state_dict):
        import torch
        self.kind = "port"
        self.sd = {k: v.detach().cpu() for k, v in state_dict.items()}
        if os.path.isdir(os.path.join(REF_DIR, "modules", "visinger")):
            import warnings
            warnings.filterwarnings("ignore")
            sys.path.insert(0, REF_DIR)
            try:
                from modules.visinger.flow import ResidualCouplingBlock      # the unmodified reference
                from modules.visinger.decoder import Generator
                self.flow = ResidualCouplingBlock(192, 192, 5, 1, 4, gin_channels=256).eval()       # models/visinger.py:65
                self.dec = Generator(192, "1", [3, 7, 11], [[1, 3, 5]] * 3, [5, 5, 3, 2, 2], 512, [11, 11, 7, 4, 4],
                                     gin_channels=256).eval()                                      # models/visinger.py:67-69
                self.flow.load_state_dict({k[5:]: v for k, v in self.sd.items() if k.startswith("flow.")})
                self.dec.load_state_dict({k[8:]: v for k, v in self.sd.items() if k.startswith("decoder.")})
                self.kind = "reference"
            finally:
                sys.path.remove(REF_DIR)

    def __call__(self, mu, logs, noise, mask, g):
        import torch
        with torch.no_grad():
            if self.kind == "reference":
                z_p = (mu + noise * torch.exp(logs)) * mask                          # models/visinger.py:107
                z_q = self.flow(z_p, mask, g=g, reverse=True) * mask                 # :109
                return self.dec(z_q * mask, g=g).squeeze(1), z_q                     # :111
            from oracle import visinger_oracle as O
            return O.infer_hot_path(self.sd, mu, logs, noise, mask, g)


def cpu_hot_path_time(cpu, inputs, reps, threads):
    import torch
    torch.set_num_threads(threads)
    times, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = cpu(*inputs)
        times.append(time.perf_counter() - t0)
    return times, out


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (the vendored reference modules when
    present, else the oracle port) on all host threads, same weights and inputs as the B200 arm; each step a bounded
    sample of the arm's workload (one of its B utterances)."""
    import torch
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    Ts = args.frames
    hp, inputs = bench_weights_and_inputs(args.batch, Ts)
    cpu = CpuHotPath(hp.state_dict())
    one = [t[:1].contiguous() for t in inputs]
    times, (wav, z_q) = cpu_hot_path_time(cpu, one, args.warmup + args.steps, cores)
    times = times[args.warmup:]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"wav": wav, "z_q": z_q})
    audio = Ts * FRAME_SEC
    tot = sum(times)
    val = audio * len(times) / tot
    t1, _ = cpu_hot_path_time(cpu, one, 1, 1)                    # the reference's own launcher pins OMP_NUM_THREADS=1 (tasks/runs/run.py:3)
    what = "the unmodified reference modules (baseline/_ref)" if cpu.kind == "reference" else "oracle port of the reference CPU path"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"hot path (prior sample -> flow reverse -> HiFi-GAN generator), {what}; bounded sample per "
                                   f"step: utterance 0 of the B={args.batch} x T={Ts} workload ({audio:.1f} s audio), same weights "
                                   "and inputs as the B200 arm",
                       "threads": cores},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": cpu.kind,
                             "sample": f"{args.steps} steps of 1 utterance x T={Ts} frames ({audio:.1f} s audio each), fp32, all host threads",
                             "one_thread": {"value": audio / t1[0], "unit": UNIT, "cores": 1,
                                            "sample": "1 step of the same utterance with torch.set_num_threads(1) "
                                                      "(the reference launcher's OMP_NUM_THREADS=1, tasks/runs/run.py:3)"}},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def sharded_leg(hp, dev, rank, world, barrier, max_over_ranks, n_utt=512, frames_per_batch=16000):
    """BASELINE.json configs[4] through the hot path: 512 synthetic utterances with the CSD-like length distribution of
    SURVEY.md 8(d) (seed 1234) are length-bucketed over the whole list (utils/commons/dataset_utils.py:69-118) and the
    batches assigned to the ranks longest-first on their padded size (reference analogue: the rank slicing of
    tasks/base.py:130-133; visinger_b200.sharding.plan_sharded_batches), then run through the per-rank serving loop.  Timed from "padded batches in pinned host memory" (what the reference's collater
    hands over) to "all int16 / fp32 results in pinned host memory"; device time, max over ranks."""
    import numpy as np
    import torch
    from visinger_b200.sharding import HostBatchRunner, plan_sharded_batches
    rng = np.random.default_rng(1234)
    lengths = np.clip(np.round(80 * rng.lognormal(np.log(5.6), 0.45, n_utt)), 120, 1280).astype(int).tolist()
    plans = plan_sharded_batches(lengths, world, frames_per_batch, 64)      # length buckets first, then LPT of the batches
    loads = [sum(lengths[i] for b in pl for i in b) for pl in plans]
    padded = [sum(len(b) * max(lengths[i] for i in b) for b in pl) for pl in plans]
    gen = torch.Generator().manual_seed(4000 + rank)
    pool = torch.randn(3, 192 * 1280 * 64 // 8, generator=gen)       # one pool of random values, sliced per batch (host time)
    batches, lens = [], []
    for b in plans[rank]:
        T, B = max(lengths[i] for i in b), len(b)
        n = B * 192 * T
        mu, noise = (pool[k, :1].expand(n) if n > pool.shape[1] else pool[k, :n] for k in (0, 1))
        mask = torch.zeros(B, 1, T)
        for r, i in enumerate(b):
            mask[r, :, :lengths[i]] = 1
        batches.append({"mu_p": mu.reshape(B, 192, T).contiguous().pin_memory(),
                        "logs_p": torch.full((B, 192, T), -1.0).pin_memory(),
                        "noise": noise.reshape(B, 192, T).contiguous().pin_memory(), "mask": mask.pin_memory(),
                        "g": (0.1 * pool[2, :B * 256]).reshape(B, 256, 1).contiguous().pin_memory()})
        lens.append(torch.tensor([lengths[i] * 300 for i in b], dtype=torch.int32).pin_memory())
    res = {}
    for pcm in (False, True):
        runner = HostBatchRunner(hp, dev, n_streams=2, pcm=pcm)
        outs = runner.alloc_outputs(batches)
        runner.run(batches, outs, lens)          # warm-up: workspaces grow to the largest batch, lazy module load
        runner.wait()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        runner.run(batches, outs, lens)
        e1.record()
        barrier()
        res["int16" if pcm else "fp32"] = (max_over_ranks(e0.elapsed_time(e1)), sum(o.numel() * o.element_size() for o in outs))
        finite = all(bool(torch.isfinite(o).all()) for o in outs) if not pcm else all(int(o.abs().max()) == 32767 for o in outs)
        assert finite, "sharded leg produced a non-finite / un-normalised result"
    audio = sum(lengths) * FRAME_SEC
    ms, d2h = res["fp32"]
    ms16, d2h16 = res["int16"]
    return {"workload": f"{n_utt} utterances, T_i = clip(round(80 * LogNormal(ln 5.6, 0.45)), 120, 1280) frames (seed 1234), "
                        f"{audio:.0f} s audio in total; length-sorted buckets of <= {frames_per_batch} padded frames (smaller with more "
                        "ranks: ~6 batches per rank) -> LPT assignment of the batches to ranks -> HotPath.infer per batch on 2 "
                        "streams -> pinned host results",
            "scaling": "strong", "value": audio / (ms * 1e-3), "unit": UNIT, "ms": ms,
            "value_int16_output": audio / (ms16 * 1e-3), "ms_int16_output": ms16,
            "d2h_bytes_rank0": d2h, "d2h_bytes_rank0_int16": d2h16,
            "batches_per_rank": [len(pl) for pl in plans],
            "padding_overhead": sum(padded) / sum(loads),
            "imbalance_max_over_mean": max(padded) / (sum(padded) / len(padded)),
            "efficiency_bound": sum(loads) / (len(padded) * max(padded)),
            "timed": "padded batches in pinned host memory -> results in pinned host memory, CUDA events, max over ranks"}


def full_model_leg(dev, mel_l1=None, steps=3, n_utt=64, frames_per_batch=16000):
    """BASELINE.json configs[3]: full infer on 64 mixed-length synthetic utterances (note / lyric token tensors of the
    collater, SURVEY.md 8(d) length distribution, seed 1234) on one GPU.  Utterances are length-sorted into buckets of
    <= 16000 padded frames (the reference sorts by length too: base_config.yaml:15); each bucket is one
    VISinger.forward_graphed call (the whole forward from one CUDA graph per bucket shape).  Timed from pinned host token
    tensors to pinned host waveforms, CUDA events.  Parity: the fp32 mode of this model is pinned to the reference's
    whole-model golden by tests/test_model_mirror.py; the leg reports the bf16 mode's distance to it on the identical padded
    batch (the shortest bucket, so the 260 ms/16k-frame fp32 kernels stay within seconds)."""
    import numpy as np
    import torch
    from model_inputs import full_hparams, synth_utterances
    from visinger_b200.models.visinger import VISinger
    rng = np.random.default_rng(1234)
    lengths = np.clip(np.round(80 * rng.lognormal(np.log(5.6), 0.45, n_utt)), 120, 1280).astype(int).tolist()
    order = sorted(range(n_utt), key=lambda i: -lengths[i])
    buckets, cur = [], []
    for i in order:
        if cur and (len(cur) + 1) * lengths[cur[0]] > frames_per_batch:
            buckets.append(cur)
            cur = []
        cur.append(i)
    buckets.append(cur)
    torch.manual_seed(1234)
    m = VISinger(73, 117, 132, full_hparams(), precision="bf16").eval()
    for name, prm in m.named_parameters():       # the reference zero-initialises flow `post` (flow.py:63-64): make it non-trivial
        if ".post." in name:
            torch.nn.init.normal_(prm, std=0.05)
    m = m.to(dev)
    host, noises, outs = [], [], []
    for k, b in enumerate(buckets):
        hb = synth_utterances(seed=100 + k, n=len(b), lengths=[lengths[i] for i in b])
        host.append({kk: v.pin_memory() for kk, v in hb.items()})
        T = hb["mel2ph"].shape[1]
        noises.append(torch.randn(len(b), 192, T, generator=torch.Generator().manual_seed(200 + k)).to(dev))
        outs.append(torch.empty(len(b), T * 300, dtype=torch.float32).pin_memory())

    def run_all():
        for hb, nz, o in zip(host, noises, outs):
            d = {kk: v.to(dev, non_blocking=True) for kk, v in hb.items()}
            r = m.forward_graphed(d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"], spk_id=d["spk_ids"], noise=nz)
            o.copy_(r["wav_out"], non_blocking=True)

    with torch.no_grad():
        run_all()                                 # captures one graph per bucket shape
        run_all()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            run_all()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        # parity on the identical padded batch: bf16 vs the fp32 mode of the same model (shortest bucket)
        hb = host[-1]
        d = {kk: v.to(dev) for kk, v in hb.items()}
        w16 = m(d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"], spk_id=d["spk_ids"], infer=True, noise=noises[-1])["wav_out"]
        m.precision = "fp32"
        w32 = m(d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"], spk_id=d["spk_ids"], infer=True, noise=noises[-1])["wav_out"]
        n0 = lengths[buckets[-1][0]] * 300        # valid samples of the bucket's first utterance
        a, r = w16[0, :n0].cpu(), w32[0, :n0].cpu()
        finite = all(bool(torch.isfinite(o).all()) for o in outs)
    assert finite, "full-model leg produced a non-finite waveform"
    audio = sum(lengths) * FRAME_SEC
    padded = sum(len(b) * lengths[b[0]] for b in buckets)
    del m
    torch.cuda.empty_cache()
    return {"workload": f"VISinger.forward(infer=True), {n_utt} utterances, T_i = clip(round(80 * LogNormal(ln 5.6, 0.45)), 120, 1280) "
                        f"frames (seed 1234, {audio:.0f} s audio), length-sorted into {len(buckets)} buckets of <= {frames_per_batch} "
                        "padded frames, one CUDA graph per bucket; pinned host tokens -> pinned host waveforms",
            "value": audio / (ms * 1e-3), "unit": UNIT, "ms": ms, "padding_overhead": padded / sum(lengths),
            "precision_mode": "bf16 (prior network: native bf16 encoder kernels; hot path: tcgen05)",
            "bf16_vs_fp32_mode": {"rel_l2": float((a - r).norm() / r.norm()), "max_abs": float((a - r).abs().max()),
                                  "mel_l1": mel_l1(a[None], r[None]) if mel_l1 is not None else None,
                                  "ref_max_abs": float(r.abs().max()),
                                  "on": f"utterance 0 of the last bucket ({len(buckets[-1])} x {lengths[buckets[-1][0]]} frames), the "
                                        "identical padded batch and noise in both modes"}}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    # this arm never touches oracle/: random-init weights come from the module mirrors themselves
    from visinger_b200.configs import VISINGER_FLOW as FLOW_FULL, VISINGER_GENERATOR as GEN_FULL
    from visinger_b200.models.visinger import HotPath
    import visinger_b200

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, T = args.batch, args.frames
    audio_per_step = B * T * FRAME_SEC

    hp_cpu, (x, logs, noise, mask, g) = bench_weights_and_inputs(B, T, rank)
    hp = HotPath(hp_cpu.flow, hp_cpu.decoder, precision=args.precision).to(dev).eval()
    if args.l2_mb >= 0 or args.no_pdl or args.no_fuse or args.no_merge_ups or args.no_split_n or args.two_streams or args.generic_epilogue or args.no_chain_streams:
        from visinger_b200 import _lib
        _lib.set_tc_options(halo_mode=1 | (256 if args.no_pdl else 0) | (512 if args.no_fuse else 0) |
                            (1024 if args.no_merge_ups else 0) | (2048 if args.no_split_n else 0) | (4096 if args.two_streams else 0) | (8192 if args.generic_epilogue else 0) | (16384 if args.no_chain_streams else 0), l2_tensor_mb=args.l2_mb)

    host = [t.pin_memory() for t in (x, logs, noise, mask, g)]
    devin = [t.to(dev) for t in host]
    wav_host = torch.empty(B, T * 300, dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * 4 for t in host)
    d2h = wav_host.numel() * 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, after=None):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        if after is not None:
            after()            # joins the side streams of the pipelined e2e loop into the timing stream
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    graph = None if args.no_graph else hp.graph(B, T, dev)
    if graph is not None:
        for dst, src in zip((graph.mu_p, graph.logs_p, graph.noise, graph.mask, graph.g), devin):
            dst.copy_(src)

    last = {}                  # (wav, z_q) of the latest resident step, for --dump-outputs

    def step_resident():
        if graph is not None:
            last["out"] = graph.replay()
        else:
            last["out"] = hp.infer(*devin)

    # e2e: the public serving loop (HotPath.pipeline): every step uploads its inputs from pinned host memory and
    # downloads its waveform into pinned host memory; copies of neighbouring steps overlap the kernels (3 streams)
    pipe = None if args.no_graph else hp.pipeline(B, T, dev)

    def step_e2e():
        if pipe is not None:
            pipe.submit(*host)
        else:
            wav, _ = hp.infer(*[t.to(dev, non_blocking=True) for t in host])
            wav_host.copy_(wav.view(B, -1), non_blocking=True)

    # the decoder region on its own (roofline): one CUDA graph, like the step it is a part of
    dec_graph = None
    if graph is not None:
        for _ in range(2):
            hp.decode(devin[0], devin[4])
        torch.cuda.synchronize()
        dec_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(dec_graph):
            dec_keep = hp.decode(devin[0], devin[4])     # noqa: F841  (keeps the captured output alive)

    def step_decoder():
        if dec_graph is not None:
            dec_graph.replay()
        else:
            hp.decode(devin[0], devin[4])

    for _ in range(max(args.warmup, 3)):
        step_resident()
    launches_per_step = graph.launches if graph is not None else hp.last_launches
    sampler = ClockSampler(local)
    sampler.start()
    ms = timed(step_resident, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("wav", "z_q"), last["out"])))
    for _ in range(3):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps, after=pipe.flush if pipe is not None else None)
    for _ in range(2):
        step_decoder()
    ms_dec = timed(step_decoder, args.steps)
    sampler.stop_flag = True        # clocks are sampled across all three timed regions (resident, e2e, decoder)
    sampler.join()

    # CPU leg (N=1): the reference's CPU path on utterance 0 of the batch -- timed (cpu_baseline) and, because it runs the
    # same weights and inputs, also the CHECKER of this run: the bf16 mode's relative L2 / max-abs / log-mel L1 and the
    # bf16x3 mode's max-abs error against it, on a full-length utterance.
    cpu_line, bf16_report, parity = None, None, None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import visinger_oracle as O          # checker + baseline only; never on the product path
        cores = len(os.sched_getaffinity(0))
        cpu = CpuHotPath(hp_cpu.state_dict())
        one = [t[:1].contiguous() for t in (x, logs, noise, mask, g)]
        ts, (wav_ref, z_ref) = cpu_hot_path_time(cpu, one, 4, cores)
        t1, _ = cpu_hot_path_time(cpu, one, 1, 1)
        cpu_line = {"value": T * FRAME_SEC / min(ts[1:]), "unit": UNIT, "cores": cores, "kind": cpu.kind,
                    "sample": f"utterance 0 of the {B} (T={T} frames, {T * FRAME_SEC:.1f} s audio), best of 3 after 1 warm-up, "
                              "fp32, " + ("the unmodified reference modules (baseline/_ref)" if cpu.kind == "reference"
                                          else "oracle port of the reference CPU path") + " on all host threads",
                    "one_thread": {"value": T * FRAME_SEC / t1[0], "unit": UNIT, "cores": 1,
                                   "sample": "1 pass of the same utterance with torch.set_num_threads(1) (tasks/runs/run.py:3)"}}
        sub = [t[:1].contiguous() for t in devin]
        if args.precision == "bf16":
            w16, z16 = hp.infer(*sub)
            w16, z16 = w16.cpu().squeeze(1), z16.cpu()
            bf16_report = {"rel_l2": float((w16 - wav_ref).norm() / wav_ref.norm()), "max_abs": float((w16 - wav_ref).abs().max()),
                           "mel_l1": O.mel_l1(w16, wav_ref), "z_rel_l2": float((z16 - z_ref).norm() / z_ref.norm()),
                           "ref_max_abs": float(wav_ref.abs().max()),
                           "vs": f"CPU {cpu.kind} (fp32) on utterance 0 of the batch, T={T}: waveform relative L2, max-abs, "
                                 "L1 of log-mel spectrograms (MelSpectrogramFixed, utils/audio/mel_processing.py:28-38)"}
        if args.precision == "bf16" and not args.no_parity_mode:
            # the mode that meets north_star's fp32 tolerances (waveform <= 1e-4, z <= 1e-5) on the tensor-core kernels
            hp3 = HotPath(hp.flow, hp.decoder, precision="bf16x3")       # same modules, own weight pack
            wav3, z3 = hp3.infer(*sub)
            err3, errz = float((wav3.cpu().squeeze(1) - wav_ref).abs().max()), float((z3.cpu() - z_ref).abs().max())
            mel3 = O.mel_l1(wav3.cpu().squeeze(1), wav_ref)
            for _ in range(2):
                hp3.infer(*devin)
            k3 = max(3, min(args.steps, 5))
            ms3 = timed(lambda: hp3.infer(*devin), k3)
            parity = {"precision": "bf16x3", "value": audio_per_step * k3 / (ms3 * 1e-3), "unit": UNIT, "ms_per_step": ms3 / k3,
                      "wav_max_abs_err": err3, "z_max_abs_err": errz, "mel_l1": mel3,
                      "meets_fp32_tolerance": bool(err3 <= 1e-4 and errz <= 1e-5),
                      "arithmetic": "tcgen05 throughout: decoder on two bf16 planes per value (3 MMAs per product), flow on "
                                    "three (6 plane products, small-first: the tensor pipe's fp32 accumulation truncates)",
                      "vs": f"CPU {cpu.kind} (fp32) on utterance 0 of the batch, T={T}"}
            del hp3
            torch.cuda.empty_cache()

    sharded = None
    if args.precision == "bf16" and not args.no_sharded:
        sharded = sharded_leg(hp, dev, rank, world, barrier, max_over_ranks)
    full_model = None
    if args.precision == "bf16" and not args.no_full_model and world == 1 and (B, T) == (16, 1000):
        # (the mel metric is the checker's -- oracle/ -- and only available when the cpu_baseline leg imported it)
        full_model = full_model_leg(dev, mel_l1=None if args.no_cpu_baseline else __import__("oracle.visinger_oracle", fromlist=["mel_l1"]).mel_l1)

    if rank == 0:
        pk = peaks()
        value = world * audio_per_step * args.steps / (ms * 1e-3)
        e2e_value = world * audio_per_step * args.steps / (ms_e2e * 1e-3)
        dec_tflops = DEC_FLOP_PER_FRAME * B * T * args.steps / (ms_dec * 1e-3) / 1e12
        traffic, traffic_launches = None, 0   # DRAM bytes of the decoder's conv kernels per pass, from the committed ncu capture
        tp = os.path.join(ROOT, "profiles", "r2_decoder_traffic.json")
        if os.path.exists(tp) and args.precision == "bf16" and (B, T) == (16, 1000):
            tj = json.load(open(tp))
            traffic, traffic_launches = tj["traffic_bytes"], tj["launches"]
        peak = pk["bf16_sustained"]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "bf16x3": "bf16x3 (split-bf16 pairs, fp32 accumulate)", "fp32": "f32"}[args.precision],
            "data": "synthetic",
            "config": {"workload": f"hot path: prior sample -> ResidualCouplingBlock.reverse -> HiFi-GAN Generator; "
                                   f"B={B} utterances x T={T} latent frames ({audio_per_step:.0f} s audio) per GPU per step; "
                                   "config/models/visinger.yaml shapes, random weights",
                       "precision_mode": args.precision, "sharding": f"by utterance, {world} replica(s), no collective",
                       "l2": "no explicit flush: each step streams >1 GB of activations, far beyond the 126 MB L2",
                       "launch": "direct" if graph is None else "one CUDA graph per step",
                       "e2e_path": "HotPath.pipeline: pinned host inputs -> H2D -> graph -> D2H -> pinned host waveform, "
                                   "double-buffered on 3 streams (every step's copies are inside the timed region)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": sampler.summary(),
            "roofline": {"bound": "tensor", "achieved": dec_tflops, "peak": peak, "unit": "TFLOP/s",
                         "frac": dec_tflops / peak, "frac_of_burst_peak": dec_tflops / pk["bf16_burst"], "traffic": traffic,
                         "traffic_note": f"dram__bytes_read.sum + dram__bytes_write.sum over the {traffic_launches} conv_tc / rp_tc / "
                                         "conv_post launches of one decoder pass (profiles/r2_decoder_traffic.json)",
                         "kernel": "decoder convolutions (vsg_generator_forward region, replayed as one CUDA graph like the step)",
                         "algorithmic": f"{DEC_FLOP_PER_FRAME} FLOP/frame x {B * T} frames",
                         "ms": ms_dec / args.steps, "peak_source": pk["src"] + ", sustained bf16"},
        }
        if bf16_report is not None:
            line["bf16"] = bf16_report
        if parity is not None:
            line["parity_mode"] = parity
        if sharded is not None:
            line["sharded"] = sharded
        if full_model is not None:
            line["full_model"] = full_model
        if cpu_line is not None:
            line["cpu_baseline"] = cpu_line
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
