"""Golden vectors for the WHOLE `VISinger.forward(infer=True)` from the unmodified reference model.

Run in the build container only:  python tests/golden/make_golden_model.py

Oracle patches (SURVEY.md 8c), none of which touches the hot-path code:
  (1) `FramePriorNetwork.forward` without the `g.transpose(1, 2)` that crashes the shipped reference (App. B-1);
  (2) `post` layers of the flow re-randomised (they are zero-initialised, App. B-2);
  (3) prior noise injected by patching `torch.randn_like`;
  (4) `utils.audio` stubbed as a namespace package (its __init__ imports librosa etc., absent here) and a reduced
      hparams dict (hidden 32) so that the fixture stays small; synthetic note/lyric tensors (SURVEY.md 8d).
"""
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

from model_inputs import SMALL_HPARAMS, synth_utterances  # noqa: E402
from helpers import save_npz_parts  # noqa: E402

torch.set_grad_enabled(False)


def _frame_prior_forward(self, x, x_mask, g=None):   # patch (1)
    prior_out = self.encoder(x, x_mask, g)
    prior_out = self.proj(prior_out) * x_mask
    return torch.split(prior_out, self.hidden_channels, dim=1)


ref_encoder.FramePriorNetwork.forward = _frame_prior_forward


def main():
    torch.manual_seed(1234)
    hp = dict(SMALL_HPARAMS)
    model = VISinger(73, 117, 132, hp).eval()
    gen = torch.Generator().manual_seed(7)
    for f in range(4):                                   # patch (2)
        post = model.flow.flows[2 * f].post
        post.weight.data.copy_(0.05 * torch.randn(post.weight.shape, generator=gen))
        post.bias.data.copy_(0.05 * torch.randn(post.bias.shape, generator=gen))
    batch = synth_utterances(seed=1234, n=3, min_frames=40, max_frames=90)
    T = batch["mel2ph"].shape[1]
    noise = torch.randn(3, hp["hidden_size"], T, generator=gen)
    real = torch.randn_like
    torch.randn_like = lambda t, *a, **k: noise.to(t)    # patch (3)
    try:
        out = model(batch["text_tokens"], batch["note_pitch"], batch["note_dur"], batch["mel2ph"],
                    spk_id=batch["spk_ids"], infer=True)
    finally:
        torch.randn_like = real
    # intermediate taps through the reference's own submodules
    mask = (batch["mel2ph"] > 0).float().unsqueeze(1)
    prior_inp = model.text_encoder(batch["text_tokens"], batch["note_pitch"], batch["note_dur"], batch["mel2ph"]) * mask
    pos = model.embed_positions(prior_inp.shape[0], prior_inp.shape[2], prior_inp.transpose(1, 2)[..., 0])
    prior_inp = prior_inp + pos.transpose(1, 2)
    spk = model.speaker_embedding(None, batch["spk_ids"]).transpose(1, 2)
    cond = model.forward_pitch(prior_inp, None, None, spk, mask, {})
    mu_p, logs_p = model.frame_prior(prior_inp, mask, cond)
    # training-only modules (posterior encoder, CTC phoneme head) are not needed to reproduce forward(infer=True)
    sd = {k: v.numpy() for k, v in model.state_dict().items()
          if not k.startswith(("posterior_encoder.", "phoneme_predictor."))}
    save_npz_parts("small_model", dict(noise=noise.numpy(), wav_out=out["wav_out"].numpy(), f0_pred=out["f0_pred"].numpy(),
                                       mu_p=mu_p.numpy(), logs_p=logs_p.numpy(),
                                       **{"in/" + k: v.numpy() for k, v in batch.items()},
                                       **{"w/" + k: v for k, v in sd.items()}))
    print("wav_out", tuple(out["wav_out"].shape), "|wav|max", float(out["wav_out"].abs().max()),
          "mu_p", tuple(mu_p.shape), "params", sum(v.size for v in sd.values()))


if __name__ == "__main__":
    main()
