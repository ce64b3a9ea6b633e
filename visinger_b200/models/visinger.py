"""Host-side mirror of the reference's `models/visinger.py` inference branch (lines 105-111).

`HotPath` owns a `ResidualCouplingBlock` (as `.flow`) and a `Generator` (as `.decoder`) -- the
attribute names and state-dict prefixes of the reference `VISinger` module -- packs both into ONE
VsgPack and runs prior sampling -> flow reverse -> decoder through a single `vsg_infer` call
(include/visinger_b200.h), i.e. exactly models/visinger.py:107-111.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from copy import deepcopy

from .. import _lib
from ..modules.rel_transformer import RelativeEncoder, SinusoidalPositionalEmbedding
from ..modules.visinger._packing import PackedModuleMixin
from ..modules.visinger.flow import ResidualCouplingBlock
from ..modules.visinger.decoder import Generator
from ..modules.visinger.encoder import (DEFAULT_MAX_TARGET_POSITIONS, Embedding, FramePriorNetwork, PosteriorEncoder,
                                        TextEncoder)
from ..modules.visinger.encoder import PhonemePredictor, PitchPredictor


class HotPath(PackedModuleMixin, nn.Module):
    """models/visinger.py:105-111 as one fused native call."""

    def __init__(self, flow: ResidualCouplingBlock, decoder: Generator, precision: str = "fp32"):
        super().__init__()
        if flow.channels != decoder.initial_channel:
            raise ValueError("flow channels must equal the decoder's initial_channel")
        if flow.gin_channels != decoder.gin_channels:
            raise ValueError(f"flow.gin_channels ({flow.gin_channels}) must equal decoder.gin_channels "
                             f"({decoder.gin_channels}): both are conditioned on the same speaker embedding "
                             "(models/visinger.py:109,111)")
        self.flow = flow
        self.decoder = decoder
        self.precision = precision
        self.last_launches = 0

    @classmethod
    def from_configs(cls, flow_cfg, gen_cfg, flow_sd, gen_sd, device, precision="fp32"):
        flow = ResidualCouplingBlock(flow_cfg["channels"], flow_cfg["hidden"], flow_cfg["kernel_size"],
                                     flow_cfg["dilation_rate"], flow_cfg["n_layers"], n_flows=flow_cfg["n_flows"],
                                     gin_channels=flow_cfg["gin"])
        dec = Generator(gen_cfg["initial_channel"], gen_cfg["resblock"], gen_cfg["rk"], gen_cfg["rd"], gen_cfg["ur"],
                        gen_cfg["uic"], gen_cfg["uk"], gin_channels=gen_cfg["gin"])
        flow.load_state_dict(flow_sd)
        dec.load_state_dict(gen_sd)
        return cls(flow, dec, precision).to(device).eval()

    @classmethod
    def random_init(cls, flow_cfg, gen_cfg, device, precision="fp32", seed=0, post_std=0.05):
        """Randomly initialised hot path of the given architecture (benchmarks, smoke runs without a checkpoint).
        PyTorch's default initialisation of the mirrors, except that the coupling layers' `post` convolutions -- which the
        reference zero-initialises (flow.py:63-64), making an untrained flow the identity -- get N(0, post_std) weights so
        that every kernel of the flow computes on non-trivial data."""
        with torch.random.fork_rng(devices=[]):
            torch.manual_seed(seed)
            flow = ResidualCouplingBlock(flow_cfg["channels"], flow_cfg["hidden"], flow_cfg["kernel_size"],
                                         flow_cfg["dilation_rate"], flow_cfg["n_layers"], n_flows=flow_cfg["n_flows"],
                                         gin_channels=flow_cfg["gin"])
            dec = Generator(gen_cfg["initial_channel"], gen_cfg["resblock"], gen_cfg["rk"], gen_cfg["rd"], gen_cfg["ur"],
                            gen_cfg["uic"], gen_cfg["uk"], gin_channels=gen_cfg["gin"])
            for name, prm in flow.named_parameters():
                if ".post." in name:
                    nn.init.normal_(prm, std=post_std)
        return cls(flow, dec, precision).to(device).eval()

    # -- packing: both modules in one pack, reference checkpoint prefixes ------------------------
    def _vsg_config(self):
        c = self.decoder._vsg_config()
        f = self.flow._vsg_config()
        for name in ("flow_channels", "flow_hidden", "flow_kernel_size", "flow_dilation_rate", "flow_n_layers",
                     "flow_n_flows", "flow_gin"):
            setattr(c, name, getattr(f, name))
        return c

    def _vsg_prefixes(self):
        return "flow.", "decoder."

    # -- models/visinger.py:107-111 --------------------------------------------------------------
    @torch.no_grad()
    def infer(self, mu_p, logs_p, noise, mask, g):
        """(mu_p, logs_p, noise) [B, C, T], mask [B, 1, T], g [B, gin, 1] -> (wav [B, 1, T*hop], z_q [B, C, T])."""
        for n, t in (("mu_p", mu_p), ("logs_p", logs_p), ("noise", noise), ("mask", mask)):
            _lib.require_cuda(t, n)
        B, C, T = mu_p.shape
        if C != self.flow.channels:
            raise RuntimeError(f"expected {self.flow.channels} channels, got {C}")
        if logs_p.shape != mu_p.shape or noise.shape != mu_p.shape or mask.numel() != B * T:
            raise RuntimeError("mu_p, logs_p, noise must share a shape and mask must be [B, 1, T]")
        use_g = self._check_g(g, B)
        pack = self._pack()
        prec = _lib.precision_code(self.precision)
        a = [_lib.as_f32c(t) for t in (mu_p, logs_p, noise, mask)]
        gc = _lib.as_f32c(g) if use_g else None
        dev = mu_p.device
        wav = torch.empty(B, 1, T * self.decoder.hop_size, dtype=torch.float32, device=dev)
        z_q = torch.empty(B, C, T, dtype=torch.float32, device=dev)
        if B == 0 or T == 0:
            return wav, z_q
        with torch.cuda.device(dev):
            ws = _lib.workspace(dev, pack.workspace_bytes(B, T, prec))
            rc = _lib.lib().vsg_infer(pack.handle, a[0].data_ptr(), a[1].data_ptr(), a[2].data_ptr(), a[3].data_ptr(),
                                      gc.data_ptr() if use_g else None, wav.data_ptr(), z_q.data_ptr(), B, T, prec,
                                      ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev))
        _lib.check(rc, "vsg_infer")
        self.last_launches = _lib.last_launch_count()
        return wav, z_q

    @torch.no_grad()
    def infer_zp(self, z_p, mask, g):
        """models/visinger.py:109-111 from an already sampled z_p [B, C, T] (what the native frame-prior head emits):
        z_q = flow(z_p, reverse) * mask; wav = decoder(z_q).  Returns (wav [B, 1, T*hop], z_q)."""
        _lib.require_cuda(z_p, "z_p")
        _lib.require_cuda(mask, "mask")
        B, C, T = z_p.shape
        if C != self.flow.channels or mask.numel() != B * T:
            raise RuntimeError(f"expected z_p [B, {self.flow.channels}, T] and mask [B, 1, T]")
        use_g = self._check_g(g, B)
        pack = self._pack()
        prec = _lib.precision_code(self.precision)
        zc, mc = _lib.as_f32c(z_p), _lib.as_f32c(mask)
        gc = _lib.as_f32c(g) if use_g else None
        dev = z_p.device
        wav = torch.empty(B, 1, T * self.decoder.hop_size, dtype=torch.float32, device=dev)
        z_q = torch.empty(B, C, T, dtype=torch.float32, device=dev)
        if B == 0 or T == 0:
            return wav, z_q
        with torch.cuda.device(dev):
            ws = _lib.workspace(dev, pack.workspace_bytes(B, T, prec))
            rc = _lib.lib().vsg_infer_zp(pack.handle, zc.data_ptr(), mc.data_ptr(), gc.data_ptr() if use_g else None,
                                         wav.data_ptr(), z_q.data_ptr(), B, T, prec, ws.data_ptr(), ws.numel(),
                                         _lib.stream_ptr(dev))
        _lib.check(rc, "vsg_infer_zp")
        self.last_launches = _lib.last_launch_count()
        return wav, z_q

    @torch.no_grad()
    def stream(self, z_p, mask, g, chunk_frames: int):
        """`infer_zp`'s waveform in pieces: a generator of wav chunks [B, 1, n * hop], n = chunk_frames (the last chunk
        may be shorter), one `vsg_infer_zp_window` call each.  The concatenated chunks equal `infer_zp(z_p, mask, g)[0]`
        bit for bit, in every precision.  One workspace of `vsg_window_workspace_bytes` -- independent of T -- serves the
        whole stream.  z_p, mask and g must stay unchanged until the stream is exhausted."""
        _lib.require_cuda(z_p, "z_p")
        _lib.require_cuda(mask, "mask")
        B, C, T = z_p.shape
        if C != self.flow.channels or mask.numel() != B * T:
            raise RuntimeError(f"expected z_p [B, {self.flow.channels}, T] and mask [B, 1, T]")
        if chunk_frames < 1:
            raise RuntimeError("chunk_frames must be >= 1")
        use_g = self._check_g(g, B)
        pack = self._pack()
        prec = _lib.precision_code(self.precision)
        zc, mc = _lib.as_f32c(z_p), _lib.as_f32c(mask)
        gc = _lib.as_f32c(g) if use_g else None
        dev, hop = z_p.device, self.decoder.hop_size
        n = min(chunk_frames, T)
        ws = torch.empty(max(pack.window_workspace_bytes(B, T, n, prec), 1), dtype=torch.uint8, device=dev) if T else None
        for t0 in range(0, T, n):
            t1 = min(T, t0 + n)
            wav = torch.empty(B, 1, (t1 - t0) * hop, dtype=torch.float32, device=dev)
            if B:
                with torch.cuda.device(dev):
                    rc = _lib.lib().vsg_infer_zp_window(pack.handle, zc.data_ptr(), mc.data_ptr(),
                                                        gc.data_ptr() if use_g else None, wav.data_ptr(), (t1 - t0) * hop,
                                                        None, B, T, t0, t1, prec, ws.data_ptr(), ws.numel(),
                                                        _lib.stream_ptr(dev))
                _lib.check(rc, "vsg_infer_zp_window")
                self.last_launches = _lib.last_launch_count()
            yield wav

    @torch.no_grad()
    def decode_window(self, z, g, t0: int, t1: int):
        """Frames [t0, t1) of `decode(z, g)` (vsg_generator_forward_window): wav [B, 1, (t1 - t0) * hop], bit for bit."""
        _lib.require_cuda(z, "z")
        B, _, T = z.shape
        pack = self._pack()
        prec = _lib.precision_code(self.precision)
        zc = _lib.as_f32c(z)
        use_g = self._check_g(g, B)
        gc = _lib.as_f32c(g) if use_g else None
        hop = self.decoder.hop_size
        wav = torch.empty(B, 1, max(t1 - t0, 0) * hop, dtype=torch.float32, device=z.device)
        with torch.cuda.device(z.device):
            ws = _lib.workspace(z.device, pack.window_workspace_bytes(B, T, max(t1 - t0, 1), prec))
            rc = _lib.lib().vsg_generator_forward_window(pack.handle, zc.data_ptr(), gc.data_ptr() if use_g else None,
                                                         wav.data_ptr(), max(t1 - t0, 0) * hop, B, T, t0, t1, prec,
                                                         ws.data_ptr(), ws.numel(), _lib.stream_ptr(z.device))
        _lib.check(rc, "vsg_generator_forward_window")
        self.last_launches = _lib.last_launch_count()
        return wav

    def _check_g(self, g, B: int) -> bool:
        """The reference broadcasts g [B, gin, 1] over time (models/visinger.py:84); anything else would be misread
        as B*gin floats through the raw pointer, so it is rejected here.  Returns whether g is used."""
        gin = self.flow.gin_channels
        if gin == 0:
            return False
        if g is None:
            raise RuntimeError("g is required (gin_channels != 0)")
        _lib.require_cuda(g, "g")
        if g.numel() != B * gin or g.shape[0] != B:
            raise RuntimeError(f"g must be [B={B}, gin={gin}, 1]; got {tuple(g.shape)}")
        return True

    # -- CUDA-graph replay of the whole path -----------------------------------------------------
    @torch.no_grad()
    def graph(self, B: int, T: int, device=None) -> "HotPathGraph":
        """Capture prior sampling -> flow reverse -> decoder for a fixed (B, T) into one CUDA graph.

        The run calls of the C ABI neither allocate nor synchronise, so the ~300-1200 kernel launches of one
        pass (more with L2-resident batch tiling) replay from a single cudaGraphLaunch.  Inputs are written into
        the graph's static buffers (`.mu_p, .logs_p, .noise, .mask, .g`), outputs read from `.wav, .z_q`."""
        dev = torch.device(device) if device is not None else next(self.parameters()).device
        self._pack()
        # the graph bakes the pack's device pointers in: key on the parameter identity / version the pack was built from,
        # so load_state_dict / .to() / remove_weight_norm get a fresh capture instead of stale (or freed) weights
        key = (B, T, _lib.precision_code(self.precision), str(dev), self._vsg_key)
        cache = self.__dict__.setdefault("_graphs", {})
        for k in [k for k in cache if k[4] != self._vsg_key]:
            del cache[k]
        if key not in cache:
            cache[key] = HotPathGraph(self, B, T, dev)
        return cache[key]

    @torch.no_grad()
    def pipeline(self, B: int, T: int, device=None, depth: int = 2, run_streams: int = 1) -> "HotPathPipeline":
        """Double-buffered serving loop for host-resident requests (see HotPathPipeline)."""
        dev = torch.device(device) if device is not None else next(self.parameters()).device
        return HotPathPipeline(self, B, T, dev, depth, run_streams)

    def decode(self, z, g):
        """Generator only, through the shared pack (used by bench.py for the decoder roofline)."""
        _lib.require_cuda(z, "z")
        B, _, T = z.shape
        pack = self._pack()
        prec = _lib.precision_code(self.precision)
        zc = _lib.as_f32c(z)
        use_g = self._check_g(g, B)
        gc = _lib.as_f32c(g) if use_g else None
        wav = torch.empty(B, 1, T * self.decoder.hop_size, dtype=torch.float32, device=z.device)
        with torch.cuda.device(z.device):
            ws = _lib.workspace(z.device, pack.workspace_bytes(B, T, prec))
            rc = _lib.lib().vsg_generator_forward(pack.handle, zc.data_ptr(), gc.data_ptr() if use_g else None,
                                                  wav.data_ptr(), B, T, prec, ws.data_ptr(), ws.numel(),
                                                  _lib.stream_ptr(z.device))
        _lib.check(rc, "vsg_generator_forward")
        self.last_launches = _lib.last_launch_count()
        return wav


class HotPathGraph:
    """A captured (B, T)-shaped pass of `HotPath`: static input/output/workspace buffers + one torch.cuda.CUDAGraph."""

    def __init__(self, hp: HotPath, B: int, T: int, device: torch.device):
        C, gin = hp.flow.channels, hp.flow.gin_channels
        f32 = dict(dtype=torch.float32, device=device)
        self.mu_p = torch.zeros(B, C, T, **f32)
        self.logs_p = torch.zeros(B, C, T, **f32)
        self.noise = torch.zeros(B, C, T, **f32)
        self.mask = torch.ones(B, 1, T, **f32)
        self.g = torch.zeros(B, max(gin, 1), 1, **f32)
        self.wav = torch.empty(B, 1, T * hp.decoder.hop_size, **f32)
        self.z_q = torch.empty(B, C, T, **f32)
        pack = hp._pack()
        prec = _lib.precision_code(hp.precision)
        self._ws = torch.empty(pack.workspace_bytes(B, T, prec), dtype=torch.uint8, device=device)  # private: pointers are baked
        self._pack = pack                      # keeps the device weights alive for as long as the graph exists
        self._gin, self._B = gin, B
        L = _lib.lib()

        def run():
            rc = L.vsg_infer(pack.handle, self.mu_p.data_ptr(), self.logs_p.data_ptr(), self.noise.data_ptr(),
                             self.mask.data_ptr(), self.g.data_ptr() if gin else None, self.wav.data_ptr(),
                             self.z_q.data_ptr(), B, T, prec, self._ws.data_ptr(), self._ws.numel(),
                             _lib.stream_ptr(device))
            _lib.check(rc, "vsg_infer")

        with torch.cuda.device(device):
            side = torch.cuda.Stream(device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):      # warm-up outside capture (one-time function attributes, lazy module load)
                run()
            torch.cuda.current_stream(device).wait_stream(side)
            torch.cuda.synchronize(device)
            self.launches = _lib.last_launch_count()
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                run()

    def replay(self):
        self._graph.replay()
        return self.wav, self.z_q

    def check_g(self, g) -> None:
        if self._gin and (g is None or g.numel() != self._B * self._gin):
            raise RuntimeError(f"g must be [B={self._B}, gin={self._gin}, 1] (gin_channels != 0)")

    def __call__(self, mu_p, logs_p, noise, mask, g=None):
        self.check_g(g)
        self.mu_p.copy_(mu_p, non_blocking=True)
        self.logs_p.copy_(logs_p, non_blocking=True)
        self.noise.copy_(noise, non_blocking=True)
        self.mask.copy_(mask, non_blocking=True)
        if g is not None:
            self.g.copy_(g, non_blocking=True)
        return self.replay()


class HotPathPipeline:
    """Serving loop around `HotPathGraph` for host-resident requests: the host->device copy of request i+1 and the
    device->host copy of waveform i-1 overlap the kernels of request i.

    `depth` graph instances (own static inputs, outputs and workspace) and three streams -- upload, run, download --
    chained with events per slot:  upload(i) waits for run(i - depth) (the graph that last read this slot's inputs),
    run(i) waits for upload(i) and download(i - depth) (the copy that last read this slot's waveform), download(i)
    waits for run(i).  Inputs must be pinned host tensors (or device tensors); `result(ticket)` blocks until that
    request's waveform is in its pinned host buffer.  Nothing here is specific to a benchmark: it is the loop a
    synthesis server would run."""

    def __init__(self, hp: "HotPath", B: int, T: int, device: torch.device, depth: int = 2, run_streams: int = 1):
        # run_streams > 1: consecutive requests replay on alternating streams, so the kernels of two requests are in
        # flight together (the latency-bound flow launches and the tails of one request's persistent decoder kernels
        # are filled by the other's CTAs); use depth >= 2 * run_streams so the copies still overlap
        self.device = torch.device(device)
        self.B, self.T, self.depth = B, T, depth
        self.slots = [HotPathGraph(hp, B, T, self.device) for _ in range(depth)]
        hop = hp.decoder.hop_size
        self.wav_host = [torch.empty(B, T * hop, dtype=torch.float32).pin_memory() for _ in range(depth)]
        with torch.cuda.device(self.device):
            self.s_up, self.s_run, self.s_down = (torch.cuda.Stream(self.device) for _ in range(3))
            self.s_runs = [self.s_run] + [torch.cuda.Stream(self.device) for _ in range(max(1, run_streams) - 1)]
        self._ran = [None] * depth       # event: graph of this slot finished
        self._down = [None] * depth      # event: waveform of this slot is in host memory
        self._n = 0

    def submit(self, mu_p, logs_p, noise, mask, g=None) -> int:
        """Enqueue one request; returns a ticket for `result`."""
        s = self._n % self.depth
        slot = self.slots[s]
        slot.check_g(g)
        cur = torch.cuda.current_stream(self.device)
        with torch.cuda.stream(self.s_up):
            self.s_up.wait_stream(cur)             # inputs produced on the caller's stream (device tensors) are complete
            if self._ran[s] is not None:
                self.s_up.wait_event(self._ran[s])
            slot.mu_p.copy_(mu_p, non_blocking=True)
            slot.logs_p.copy_(logs_p, non_blocking=True)
            slot.noise.copy_(noise, non_blocking=True)
            slot.mask.copy_(mask, non_blocking=True)
            if g is not None:
                slot.g.copy_(g, non_blocking=True)
            up = self.s_up.record_event()
        s_run = self.s_runs[self._n % len(self.s_runs)]
        with torch.cuda.stream(s_run):
            s_run.wait_event(up)
            if self._down[s] is not None:
                s_run.wait_event(self._down[s])
            slot.replay()
            self._ran[s] = s_run.record_event()
        with torch.cuda.stream(self.s_down):
            self.s_down.wait_event(self._ran[s])
            self.wav_host[s].copy_(slot.wav.view(self.B, -1), non_blocking=True)
            self._down[s] = self.s_down.record_event()
        self._n += 1
        return self._n - 1

    def result(self, ticket: int) -> torch.Tensor:
        """Pinned host waveform [B, T*hop] of request `ticket` (valid until `depth` more requests are submitted)."""
        if ticket < self._n - self.depth or ticket >= self._n:
            raise RuntimeError("ticket is no longer (or not yet) held by the pipeline")
        s = ticket % self.depth
        self._down[s].synchronize()
        return self.wav_host[s]

    def flush(self) -> None:
        """Make the caller's current stream wait for every outstanding request (upload, kernels and download)."""
        cur = torch.cuda.current_stream(self.device)
        for ev in self._down:
            if ev is not None:
                cur.wait_event(ev)


class VISinger(nn.Module):
    """Drop-in for the reference `VISinger` (models/visinger.py:18-135) on the inference branch.

    Same constructor `VISinger(ph_dict_size, pitch_size, dur_size, hparams, out_dims=None)`, same child names and
    state-dict keys (reference checkpoints load with `load_state_dict`), same
    `forward(text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed=None, spk_id=None, f0=None, uv=None, mel=None,
    infer=False, **kwargs) -> dict` with keys `wav_out` [B, T*hop] and `f0_pred`.

    The prior network runs on the native kernels too: the `RelativeEncoder` stacks of the text encoder, pitch predictor
    and frame prior (`vsg_relenc_forward`), the length regulator with its data-dependent frame positions
    (`vsg_length_regulate`) and the fused frame-prior head (`vsg_frame_prior_forward`: encoder -> proj -> prior sampling);
    from `z_p` on -- flow reverse, HiFi-GAN decoder (models/visinger.py:107-111) -- one `vsg_infer_zp` call.  What stays in
    PyTorch in `forward` is token-rate glue: three embedding lookups, one Linear(576 -> 192), the speaker embedding and the
    1x1 head of the pitch predictor.  `forward_native` runs the same model, glue included, as one `vsg_model_forward`
    call.  `voice_conversion` takes audio (or a linear spectrogram) through the posterior encoder and the flow to another
    speaker's voice as one `vsg_model_convert` call; `spectrogram` is its linear spectrogram alone.  `infer=False`
    (training) is out of scope and raises.

    Extra keyword arguments (not in the reference): `noise` injects the prior noise instead of
    `torch.randn_like(mu_p)` (CPU and CUDA generators differ, so parity tests need it); `precision` selects
    "fp32" | "bf16" | "bf16x3" for the native path.

    Supported lengths: utterances of any number of latent frames T up to T * hop <= 2^29 samples, in all three modes.
    The prior network has no frame cap of its own: the length regulator works in fixed chunks of frames, and the bf16
    attention splits the keys into chunks of 2048 frames beyond T = 2048 (a workspace of about
    ceil(T / 2048) * B * T * hidden * 4 bytes per encoder).
    """

    def __init__(self, ph_dict_size, pitch_size, dur_size, hparams, out_dims=None, precision="fp32"):
        super().__init__()
        self.hparams = deepcopy(hparams)
        hp = hparams
        self.enc_layers = hp["enc_layers"]
        self.dec_blocks = hp["dec_blocks"]
        self.hidden_size = H = hp["hidden_size"]
        self.use_pos_embed = hp["use_pos_embed"]
        self.segment_size = hp["segment_size"]
        self.out_dims = hp["num_mel_bins"] if out_dims is None else out_dims
        self.precision = precision
        if hp["use_spk_id"]:
            self.spk_id_proj = Embedding(hp["num_spk"], hp["gin_channels"])
        if hp["use_spk_embed"]:
            self.spk_embed_proj = nn.Linear(256, hp["gin_channels"], bias=True)
        self.text_encoder = TextEncoder(ph_dict_size, pitch_size, dur_size, H, hp["ffn_filter_channels"], hp["num_heads"],
                                        self.enc_layers, hp["ffn_kernel_size"], hp["p_dropout"], True)
        self.embed_positions = SinusoidalPositionalEmbedding(H, 0, init_size=DEFAULT_MAX_TARGET_POSITIONS)
        if hp["use_pitch_embed"]:
            self.pitch_predictor = PitchPredictor(H, hp["ffn_filter_channels"], hp["num_heads"],
                                                  n_layers=hp["pitch_predictor_layers"], kernel_size=hp["ffn_kernel_size"],
                                                  p_dropout=hp["p_dropout"], gin_channels=hp["gin_channels"], out_dim=2)
        if hp["use_phoneme_pred"]:
            self.phoneme_predictor = PhonemePredictor(ph_dict_size, H, hp["ffn_filter_channels"], hp["num_heads"],
                                                      n_layers=hp["phoneme_predictor_layers"],
                                                      kernel_size=hp["ffn_kernel_size"], p_dropout=hp["p_dropout"])
        self.frame_prior = FramePriorNetwork(H, hp["ffn_filter_channels"], hp["num_heads"], hp["frame_prior_layers"],
                                             hp["ffn_kernel_size"], p_dropout=hp["p_dropout"], gin_channels=1)
        self.posterior_encoder = PosteriorEncoder(hp["num_linear_bins"], H, H, 5, 1, 16, gin_channels=hp["gin_channels"])
        self.flow = ResidualCouplingBlock(H, H, 5, 1, 4, gin_channels=hp["gin_channels"])
        self.decoder = Generator(H, hp["dec_blocks"], hp["dec_kernel_size"], hp["dec_dilation_sizes"], hp["upsample_rates"],
                                 hp["initial_upsample_channels"], hp["upsample_kernel_sizes"],
                                 gin_channels=hp["gin_channels"])
        # the fused native path shares the flow / decoder modules (and hence their parameters) without re-registering them
        object.__setattr__(self, "_hot", HotPath(self.flow, self.decoder, precision))

    def forward(self, text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed=None, spk_id=None, f0=None, uv=None,
                mel=None, infer=False, noise=None, **kwargs):
        if not infer:
            raise NotImplementedError("visinger_b200.VISinger implements forward(infer=True); training stays with the reference")
        with torch.no_grad():
            ret = {}
            self._hot.precision = self.precision
            if mel2ph.is_cuda and getattr(self, "fused_prior_head", True):
                # frame prior network + proj + prior sampling in one native call (vsg_frame_prior_forward), then
                # flow + decoder from z_p (vsg_infer_zp): mu_p / logs_p never round-trip through PyTorch
                z_p, mask, spk_emb = self.prior(text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed, spk_id, f0, uv, ret,
                                                noise=noise, sample=True)
                wav, z_q = self._hot.infer_zp(z_p, mask, spk_emb)
            else:
                mu_p, logs_p, mask, spk_emb = self.prior(text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed, spk_id,
                                                         f0, uv, ret)
                if noise is None:
                    noise = torch.randn_like(mu_p)
                wav, z_q = self._hot.infer(mu_p, logs_p, noise, mask, spk_emb)          # models/visinger.py:107-111
            ret["wav_out"] = wav.squeeze(1)
            ret["z_q"] = z_q
            return ret

    def forward_streaming(self, text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed=None, spk_id=None, f0=None,
                          uv=None, chunk_frames: int = 250, noise=None):
        """`forward(..., infer=True)`'s waveform as a stream: a generator of fp32 chunks [B, 1, n * hop] of chunk_frames
        latent frames each (the last may be shorter).  The prior network (global attention) runs once, on the first
        `next()`; flow and decoder then run window by window (`HotPath.stream`, vsg_infer_zp_window), every chunk bit
        for bit the same samples as the one-pass waveform, with a workspace that does not grow with the length.
        The chunks are float.  Peak-normalised int16 (`save_wav` with norm, utils/audio/io.py:8-14) needs the whole
        utterance's peak; a stream converts each chunk on its own with vsg_wav_to_int16(norm = 0)
        (`utils.audio.io.wav_to_int16(chunk, norm=False)`)."""
        if not mel2ph.is_cuda:
            raise RuntimeError("forward_streaming runs on the native path: inputs must be CUDA tensors")
        with torch.no_grad():
            self._hot.precision = self.precision
            z_p, mask, spk_emb = self.prior(text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed, spk_id, f0, uv, {},
                                            noise=noise, sample=True)
        yield from self._hot.stream(z_p, mask, spk_emb, chunk_frames)

    def forward_graphed(self, text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed=None, spk_id=None, noise=None):
        """`forward(..., infer=True)` replayed from one CUDA graph per input shape (prior network + prior sampling + flow +
        decoder: ~600 eager launches and ~12 ms of CPU issue time at B=16 x T=1000 become one cudaGraphLaunch).
        The first call with a new (shape, precision) captures; later calls copy the inputs into the graph's static
        buffers and replay.  The returned tensors are the graph's static outputs: valid until the next call with the
        same shape.  Without `noise` the prior noise comes from the CUDA generator inside the graph (fresh per replay).
        The hot path's scratch buffer is allocated during capture, i.e. in the graph's private memory pool."""
        ins = {"text_tokens": text_tokens, "pitch_tokens": pitch_tokens, "dur_tokens": dur_tokens, "mel2ph": mel2ph,
               "spk_embed": spk_embed, "spk_id": spk_id, "noise": noise}
        ins = {k: v for k, v in ins.items() if v is not None}
        for k, v in ins.items():
            _lib.require_cuda(v, k)
        # weight identity is part of the key (the graph bakes device pointers of the pack and of every prior-network
        # parameter in); the entry also holds the pack so that the weights it replays from cannot be freed under it
        wkey = tuple((p.data_ptr(), p._version) for p in self.parameters())
        key = (self.precision, wkey) + tuple((k, tuple(v.shape), v.dtype) for k, v in ins.items())
        cache = self.__dict__.setdefault("_fw_graphs", {})
        for k in [k for k in cache if k[1] != wkey]:
            del cache[k]
        if key not in cache:
            static = {k: v.clone() for k, v in ins.items()}
            dev = mel2ph.device
            with torch.cuda.device(dev):
                side = torch.cuda.Stream(dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):          # warm-up outside capture: weight pack, workspaces, cuDNN plans
                    for _ in range(2):
                        self.forward(infer=True, **static)
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    out = self.forward(infer=True, **static)
            cache[key] = (graph, static, out, self._hot._pack())
        graph, static, out, _pack = cache[key]
        for k, v in ins.items():
            static[k].copy_(v, non_blocking=True)
        graph.replay()
        return out

    def _model_config(self) -> "_lib.VsgModelConfig":
        hp = self.hparams
        te = self.text_encoder
        return _lib.VsgModelConfig(
            te.ph_emb.num_embeddings, te.pitch_emb.num_embeddings, te.dur_emb.num_embeddings, self.hidden_size,
            hp["ffn_filter_channels"], hp["num_heads"], hp["ffn_kernel_size"], te.text_encoder.window_size,
            self.enc_layers, hp["pitch_predictor_layers"] if hp["use_pitch_embed"] else 0, hp["frame_prior_layers"],
            int(bool(self.use_pos_embed)), int(bool(hp["use_pitch_embed"])), int(bool(hp["use_spk_id"])),
            int(bool(hp["use_spk_embed"])), hp["num_spk"] if hp["use_spk_id"] else 0,
            self.spk_embed_proj.in_features if hp["use_spk_embed"] else 0, self._hot._vsg_config())

    def _model_pack(self, device) -> "_lib.ModelPack":
        """The whole-model pack (vsg_model_pack_create), rebuilt when a parameter's storage or version changes."""
        wkey = (str(device),) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        cached = self.__dict__.get("_native_pack")
        if cached is None or cached[0] != wkey:
            pack = _lib.ModelPack(self._model_config(), dict(self.state_dict()), "", device)
            self.__dict__["_native_pack"] = cached = (wkey, pack)
        return cached[1]

    @property
    def win_length(self) -> int:
        """Hann window length of the linear spectrogram: hparams["win_size"], else n_fft = 2 * (num_linear_bins - 1)."""
        return int(self.hparams.get("win_size", 2 * (self.posterior_encoder.in_channels - 1)))

    def _convert_pack(self, device) -> "_lib.ConvertPack":
        """The voice-conversion pack (vsg_convert_pack_create), rebuilt like `_model_pack`."""
        wkey = (str(device), self.win_length) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        cached = self.__dict__.get("_native_convert_pack")
        if cached is None or cached[0] != wkey:
            pack = _lib.ConvertPack(self._model_config(), dict(self.state_dict()), "", self.win_length, device)
            self.__dict__["_native_convert_pack"] = cached = (wkey, pack)
        return cached[1]

    @torch.no_grad()
    def spectrogram(self, wav, lengths):
        """The linear spectrogram the posterior encoder reads (vsg_spectrogram): wav CUDA [B, T * hop], lengths CUDA int
        [B] latent frames per utterance -> fp32 [B, num_linear_bins, T].  VITS's spectrogram_torch of each utterance on
        its own (reflect padding about the utterance's ends, periodic Hann window of `win_length`, sqrt(|X|^2 + 1e-6)),
        masked beyond lengths.  bf16 precision: the bf16 values the posterior consumes."""
        _lib.require_cuda(lengths, "lengths")
        pack = self._convert_pack(wav.device)
        return pack.spectrogram(wav, lengths, _lib.precision_code(self.precision))

    @torch.no_grad()
    def voice_conversion(self, wav=None, lengths=None, spk_id=None, spk_embed=None, tgt_spk_id=None, tgt_spk_embed=None,
                         spec=None, noise=None, seeds=None):
        """Audio to audio in one library call (vsg_model_convert), VITS's voice_conversion on this model's modules:
        spectrogram -> posterior encoder under the source speaker -> flow -> flow reverse and decoder under the target
        speaker.  Give `wav` [B, T * hop] or a precomputed `spec` [B, num_linear_bins, T], and `lengths` (int [B], valid
        latent frames).  spk_id / spk_embed describe the source speaker, tgt_spk_id / tgt_spk_embed the target, as the
        model's configuration requires (ids are read on the host).  The posterior noise is `noise` [B, H, T], else drawn
        on the device from `seeds` (int64 [B]), else from seeds taken from torch's default CPU generator.
        Returns {"wav_out": [B, T * hop], "z": z_hat [B, H, T], "spec": the spectrogram the posterior read}."""
        pack, a, hosts, B, T = self._convert_inputs(wav, spec, lengths, spk_id, spk_embed, tgt_spk_id, tgt_spk_embed, noise,
                                                    seeds)
        dev, H = pack.device, self.hidden_size
        prec = _lib.precision_code(self.precision)
        wav_out = torch.empty(B, T * pack.hop, dtype=torch.float32, device=dev)
        z = torch.empty(B, H, T, dtype=torch.float32, device=dev)
        spec_out = torch.empty(B, pack.bins, T, dtype=torch.float32, device=dev) if wav is not None else None
        ptr = lambda k: a[k].data_ptr() if k in a else None   # noqa: E731
        hptr = lambda k: hosts[k].data_ptr() if k in hosts else None   # noqa: E731
        with torch.cuda.device(dev):
            ws = _lib.workspace(dev, pack.convert_workspace_bytes(B, T, prec))
            rc = _lib.lib().vsg_model_convert(
                pack.handle, ptr("wav"), ptr("spec"), ptr("lengths"), hptr("spk_id"), ptr("spk_embed"), hptr("tgt_spk_id"),
                ptr("tgt_spk_embed"), ptr("noise"), ptr("seeds"), wav_out.data_ptr(),
                spec_out.data_ptr() if spec_out is not None else None, z.data_ptr(), B, T, prec, ws.data_ptr(), ws.numel(),
                _lib.stream_ptr(dev))
        _lib.check(rc, "vsg_model_convert")
        self.last_launches = _lib.last_launch_count()
        return {"wav_out": wav_out, "z": z, "spec": spec_out if spec_out is not None else spec}

    @torch.no_grad()
    def voice_conversion_streaming(self, wav, lengths, spk_id=None, spk_embed=None, tgt_spk_id=None, tgt_spk_embed=None,
                                   noise=None, seeds=None, chunk_frames: int = 250):
        """`voice_conversion(wav, ...)["wav_out"]` as a stream: a generator of fp32 chunks [B, n * hop] of chunk_frames
        latent frames each (the last may be shorter), one vsg_model_convert_window call each.  The concatenated chunks
        equal the one-pass waveform bit for bit, in every precision, and one workspace of
        `convert_window_workspace_bytes` -- independent of the length -- serves the whole stream.  Inputs are validated as
        `voice_conversion` validates them; without `noise` and `seeds`, seeds are drawn once up front, so every window
        draws the one pass's noise.  `wav`, `lengths` and `noise` are read in place: they must stay unchanged until the
        generator is exhausted."""
        if chunk_frames < 1:
            raise RuntimeError("chunk_frames must be >= 1")
        pack, a, hosts, B, T = self._convert_inputs(wav, None, lengths, spk_id, spk_embed, tgt_spk_id, tgt_spk_embed, noise,
                                                    seeds)
        dev, hop = pack.device, pack.hop
        prec = _lib.precision_code(self.precision)
        n = min(chunk_frames, T)
        ptr = lambda k: a[k].data_ptr() if k in a else None   # noqa: E731
        hptr = lambda k: hosts[k].data_ptr() if k in hosts else None   # noqa: E731
        ws = torch.empty(max(pack.convert_window_workspace_bytes(B, T, n, prec), 1), dtype=torch.uint8, device=dev) \
            if T else None
        for t0 in range(0, T, n):
            t1 = min(T, t0 + n)
            out = torch.empty(B, (t1 - t0) * hop, dtype=torch.float32, device=dev)
            if B:
                with torch.cuda.device(dev):
                    rc = _lib.lib().vsg_model_convert_window(
                        pack.handle, ptr("wav"), ptr("lengths"), hptr("spk_id"), ptr("spk_embed"), hptr("tgt_spk_id"),
                        ptr("tgt_spk_embed"), ptr("noise"), ptr("seeds"), out.data_ptr(), (t1 - t0) * hop, None, B, T, t0,
                        t1, prec, ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev))
                _lib.check(rc, "vsg_model_convert_window")
                self.last_launches = _lib.last_launch_count()
            yield out

    def _convert_inputs(self, wav, spec, lengths, spk_id, spk_embed, tgt_spk_id, tgt_spk_embed, noise, seeds):
        """The checks and conversions of voice_conversion's arguments: (pack, device arguments by name, host speaker ids by
        name, B, T).  Draws seeds from torch's default CPU generator when neither noise nor seeds is given."""
        hp = self.hparams
        if (wav is None) == (spec is None):
            raise RuntimeError("give exactly one of wav and spec")
        src = wav if wav is not None else spec
        ins = {"wav" if wav is not None else "spec": src, "lengths": lengths}
        if hp["use_spk_embed"]:
            ins["spk_embed"], ins["tgt_spk_embed"] = spk_embed, tgt_spk_embed
        if noise is not None:
            ins["noise"] = noise
        elif seeds is not None:
            ins["seeds"] = seeds
        for k, v in ins.items():
            if v is None:
                raise RuntimeError(f"{k} is required by this model's configuration")
            _lib.require_cuda(v, k)
        dev = src.device
        pack = self._convert_pack(dev)
        B, H = src.shape[0], self.hidden_size
        if wav is not None:
            if wav.dim() != 2 or wav.shape[1] % pack.hop:
                raise RuntimeError(f"expected wav [B, T * {pack.hop}], got {tuple(wav.shape)}")
            T = wav.shape[1] // pack.hop
        else:
            if spec.dim() != 3 or spec.shape[1] != pack.bins:
                raise RuntimeError(f"expected spec [B, {pack.bins}, T], got {tuple(spec.shape)}")
            T = spec.shape[2]
        shapes = {"lengths": (B,), "noise": (B, H, T), "seeds": (B,)}
        if hp["use_spk_embed"]:
            shapes["spk_embed"] = shapes["tgt_spk_embed"] = (B, self.spk_embed_proj.in_features)
        for k, shape in shapes.items():
            if k in ins and tuple(ins[k].shape) != shape:
                raise RuntimeError(f"expected {k} of shape {shape}, got {tuple(ins[k].shape)}")
        for k, v in ins.items():
            if v.device != dev:
                raise RuntimeError(f"{k} is on {v.device}, {'wav' if wav is not None else 'spec'} on {dev}")
        hosts = {}
        if hp["use_spk_id"]:
            for k, v in (("spk_id", spk_id), ("tgt_spk_id", tgt_spk_id)):
                if v is None:
                    raise RuntimeError(f"{k} is required by this model's configuration")
                hosts[k] = torch.as_tensor(v).to("cpu", torch.int64).contiguous().reshape(-1)
                if hosts[k].numel() != B:
                    raise RuntimeError(f"expected {k} of shape ({B},), got {tuple(torch.as_tensor(v).shape)}")
        if "noise" not in ins and "seeds" not in ins:
            ins["seeds"] = torch.randint(0, 2 ** 62, (B,), dtype=torch.int64).to(dev)
        a = {k: v.to(torch.int32).contiguous() if k == "lengths" else v.to(torch.int64).contiguous() if k == "seeds"
             else _lib.as_f32c(v) for k, v in ins.items()}
        return pack, a, hosts, B, T

    @torch.no_grad()
    def forward_native(self, text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed=None, spk_id=None, f0=None, uv=None,
                       noise=None, seeds=None):
        """`forward(..., infer=True)` as ONE library call (vsg_model_forward): token front end, the three RelativeEncoder
        stacks, length regulator, speaker condition, pitch head, frame prior, flow and decoder, with no PyTorch op in
        between.  Same inputs and result keys (`wav_out` [B, T*hop], `f0_pred` [B, T, 2] with the pitch predictor, `z_q`
        [B, H, T]).  The prior noise is `noise` [B, H, T] if given, else drawn on the device from `seeds` (int64 [B], one
        Philox stream per utterance: vsg_normal_noise), else from seeds taken from torch's default CPU generator.
        `spk_id` is read on the host (the library range-checks it before it launches anything)."""
        hp = self.hparams
        ins = {"text_tokens": text_tokens, "pitch_tokens": pitch_tokens, "dur_tokens": dur_tokens, "mel2ph": mel2ph}
        if hp["use_spk_embed"]:
            ins["spk_embed"] = spk_embed
        if hp["use_pitch_embed"] and (f0 is not None or uv is not None):
            ins["f0"], ins["uv"] = f0, uv
        if noise is not None:
            ins["noise"] = noise
        elif seeds is not None:
            ins["seeds"] = seeds
        for k, v in ins.items():
            if v is None:
                raise RuntimeError(f"{k} is required by this model's configuration")
            _lib.require_cuda(v, k)
        if text_tokens.dim() != 2 or mel2ph.dim() != 2 or mel2ph.shape[0] != text_tokens.shape[0]:
            raise RuntimeError("expected tokens [B, T_ph] and mel2ph [B, T]")
        B, T_ph = text_tokens.shape
        T, H = mel2ph.shape[1], self.hidden_size
        shapes = {"pitch_tokens": (B, T_ph), "dur_tokens": (B, T_ph), "f0": (B, T), "uv": (B, T), "noise": (B, H, T),
                  "seeds": (B,)}
        if hp["use_spk_embed"]:
            shapes["spk_embed"] = (B, self.spk_embed_proj.in_features)
        for k, shape in shapes.items():
            if k in ins and tuple(ins[k].shape) != shape:
                raise RuntimeError(f"expected {k} of shape {shape}, got {tuple(ins[k].shape)}")
        dev = mel2ph.device
        for k, v in ins.items():
            if v.device != dev:
                raise RuntimeError(f"{k} is on {v.device}, mel2ph on {dev}")
        spk_host = None
        if hp["use_spk_id"]:
            if spk_id is None:
                raise RuntimeError("spk_id is required by this model's configuration")
            spk_host = torch.as_tensor(spk_id).to("cpu", torch.int64).contiguous().reshape(-1)
            if spk_host.numel() != B:
                raise RuntimeError(f"expected spk_id of shape ({B},), got {tuple(torch.as_tensor(spk_id).shape)}")
        if "noise" not in ins and "seeds" not in ins:
            ins["seeds"] = torch.randint(0, 2 ** 62, (B,), dtype=torch.int64).to(dev)
        a = {k: v.to(torch.int64).contiguous() if k in ("text_tokens", "pitch_tokens", "dur_tokens", "mel2ph", "seeds")
             else _lib.as_f32c(v) for k, v in ins.items()}
        pack = self._model_pack(dev)
        prec = _lib.precision_code(self.precision)
        wav = torch.empty(B, T * pack.hop, dtype=torch.float32, device=dev)
        f0_pred = torch.empty(B, T, 2, dtype=torch.float32, device=dev) if hp["use_pitch_embed"] else None
        z_q = torch.empty(B, H, T, dtype=torch.float32, device=dev)
        ptr = lambda k: a[k].data_ptr() if k in a else None   # noqa: E731
        with torch.cuda.device(dev):
            ws = _lib.workspace(dev, pack.workspace_bytes(B, T_ph, T, prec))
            rc = _lib.lib().vsg_model_forward(
                pack.handle, ptr("text_tokens"), ptr("pitch_tokens"), ptr("dur_tokens"), ptr("mel2ph"),
                spk_host.data_ptr() if spk_host is not None else None, ptr("spk_embed"), ptr("f0"), ptr("uv"), ptr("noise"),
                ptr("seeds"), wav.data_ptr(), f0_pred.data_ptr() if f0_pred is not None else None, z_q.data_ptr(), B, T_ph,
                T, prec, ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev))
        _lib.check(rc, "vsg_model_forward")
        self.last_launches = _lib.last_launch_count()
        ret = {"wav_out": wav, "z_q": z_q}
        if f0_pred is not None:
            ret["f0_pred"] = f0_pred
        return ret

    def prior(self, text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed=None, spk_id=None, f0=None, uv=None,
              ret=None, noise=None, sample=False):
        """models/visinger.py:75-90: everything upstream of z_p (plain PyTorch, any device).
        Returns (mu_p, logs_p, tgt_nonpadding [B, 1, T], spk_emb [B, gin, 1]); fills ret["f0_pred"]."""
        ret = {} if ret is None else ret
        # cuDNN convolutions default to TF32 on the GPU, which alone costs ~1e-4 on mu_p (SURVEY.md 8c): in the parity
        # modes ("fp32", "bf16x3") the prior runs in true fp32 so that the whole forward stays inside the reference's fp32
        # tolerance.  The throughput mode ("bf16") lets the prior's convolutions and matmuls use TF32 tensor cores as
        # well -- far below that mode's own bf16 rounding, and the fp32 prior is otherwise 3x the cost of the whole hot path.
        fast = self.precision == "bf16" and getattr(self, "prior_tf32", True)
        # the transformer stacks (text encoder, pitch predictor, frame prior) are native: vsg_relenc_forward in the
        # path's own arithmetic mode -- fp32 kernels for the parity modes, tcgen05 / warp-mma bf16 for the throughput mode
        for m in self.modules():
            if isinstance(m, RelativeEncoder):
                m.precision = "bf16" if self.precision == "bf16" else "fp32"
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = fast
        try:
            with torch.backends.cudnn.flags(enabled=torch.backends.cudnn.enabled, allow_tf32=fast):
                return self._prior(text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed, spk_id, f0, uv, ret, noise, sample)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev

    def _prior(self, text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed, spk_id, f0, uv, ret, noise=None, sample=False):
        mask = (mel2ph > 0).float().unsqueeze(1)
        if mel2ph.is_cuda and getattr(self, "native_length_regulator", True):
            # length regulator + frame positions in one kernel (vsg_length_regulate; SURVEY.md 8 row f2)
            enc = self.text_encoder.encode_tokens(text_tokens, pitch_tokens, dur_tokens)              # [B, H, T_ph]
            table = None
            if self.use_pos_embed:
                table = self.embed_positions.table(mel2ph.shape[1] + 1, enc.device)
            prior_inp = _lib.length_regulate(enc, mel2ph, table)
        else:
            prior_inp = self.text_encoder(text_tokens, pitch_tokens, dur_tokens, mel2ph) * mask
            if self.use_pos_embed:                                                  # models/visinger.py:79-82
                pos = self.embed_positions(prior_inp.shape[0], prior_inp.shape[2], prior_inp.transpose(1, 2)[..., 0])
                prior_inp = prior_inp + pos.transpose(1, 2)
        spk_emb = self.speaker_embedding(spk_embed, spk_id).transpose(1, 2)         # [B, gin, 1]
        cond_pitch = None
        if self.hparams["use_pitch_embed"]:
            cond_pitch = self.forward_pitch(prior_inp, f0, uv, spk_emb, mask, ret)
        if sample:
            self.frame_prior.precision = "bf16" if self.precision == "bf16" else "fp32"
            z_p, _, _ = self.frame_prior.sample(prior_inp, mask, cond_pitch, noise)
            return z_p, mask, spk_emb
        mu_p, logs_p = self.frame_prior(prior_inp, mask, cond_pitch)
        return mu_p, logs_p, mask, spk_emb

    def infer(self, *args, **kwargs):
        """Alias of forward(..., infer=True) (BASELINE.json calls the path `VISinger.infer`)."""
        kwargs["infer"] = True
        return self.forward(*args, **kwargs)

    def speaker_embedding(self, spk_embed=None, spk_id=None):
        out = 0
        if self.hparams["use_spk_embed"]:
            out = out + self.spk_embed_proj(spk_embed)[:, None, :]
        if self.hparams["use_spk_id"]:
            out = out + self.spk_id_proj(spk_id)[:, None, :]
        return out

    def forward_pitch(self, pitch_inp, f0, uv, spk_emb, mask, ret):
        ret["f0_pred"] = pred = self.pitch_predictor(pitch_inp, mask, spk_emb)          # [B, T, 2]
        if f0 is None:
            f0 = pred[:, :, 0]
            voiced = pred[:, :, 1] <= 0
        else:
            voiced = uv == 0
        return (f0 * voiced).unsqueeze(1) * mask                                        # log-f0 on voiced frames
