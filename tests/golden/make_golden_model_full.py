"""Golden vectors for `VISinger.forward(infer=True)` at the FULL config/models/visinger.yaml sizes on a mixed-length
batch (BASELINE.json configs[3] shape: B = 8 utterances drawn from the config-4 length distribution, right-padded to the
longest), from the unmodified reference model.  Run in the build container only:

    python tests/golden/make_golden_model_full.py

The 60.9 M weights are not stored: they are the seeded state dict of tests/model_inputs.py::full_model_mirror, loaded
into the reference through its own load_state_dict (strict).  The fixture keeps outputs only: the waveform at a stride,
the last 20 frames of every utterance and the PADDED region after it in full (the decoder is unmasked,
models/visinger.py:111, so the reference's waveform is non-zero there and must be matched) and f0_pred.
Oracle patches as in make_golden_model.py (SURVEY.md 8c)."""
import os
import sys
import types
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("VISINGER_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, REF)
warnings.filterwarnings("ignore")
import utils  # noqa: E402  (reference package)
pkg = types.ModuleType("utils.audio")
pkg.__path__ = [os.path.join(REF, "utils", "audio")]
sys.modules["utils.audio"] = pkg
from models.visinger import VISinger  # noqa: E402  (reference)
from modules.visinger import encoder as ref_encoder  # noqa: E402

from model_inputs import full_hparams, full_model_mirror, full_model_batch, FULL_GOLDEN_WAV_STRIDE  # noqa: E402

torch.set_grad_enabled(False)
HOP = 300


def _frame_prior_forward(self, x, x_mask, g=None):   # patch (1)
    prior_out = self.encoder(x, x_mask, g)
    prior_out = self.proj(prior_out) * x_mask
    return torch.split(prior_out, self.hidden_channels, dim=1)


ref_encoder.FramePriorNetwork.forward = _frame_prior_forward


def main():
    sd = full_model_mirror().state_dict()
    model = VISinger(73, 117, 132, full_hparams()).eval()
    model.load_state_dict(sd, strict=True)
    batch, noise, lengths = full_model_batch()
    real = torch.randn_like
    torch.randn_like = lambda t, *a, **k: noise.to(t)    # patch (3)
    try:
        out = model(batch["text_tokens"], batch["note_pitch"], batch["note_dur"], batch["mel2ph"],
                    spk_id=batch["spk_ids"], infer=True)
    finally:
        torch.randn_like = real
    wav = out["wav_out"]
    T = batch["mel2ph"].shape[1]
    tails, pads = [], []
    for b, n in enumerate(lengths.tolist()):
        tails.append(wav[b, (n - 20) * HOP: n * HOP].numpy())
        seg = wav[b, n * HOP: min(T, n + 10) * HOP].numpy()
        pads.append(np.pad(seg, (0, 10 * HOP - len(seg))))
    np.savez_compressed(os.path.join(HERE, "full_model.npz"), lengths=lengths, T=T,
                        wav_strided=wav[:, ::FULL_GOLDEN_WAV_STRIDE].numpy(), wav_tails=np.stack(tails),
                        wav_pads=np.stack(pads), f0_pred=out["f0_pred"].numpy())
    print("lengths", lengths.tolist(), "T", T, "wav", tuple(wav.shape), "|wav|max", float(wav.abs().max()),
          "|pad region|max", float(np.abs(np.stack(pads)).max()))


if __name__ == "__main__":
    main()
