"""Synthetic note/lyric inputs and hparams for the whole-model tests (SURVEY.md 8d "Synthetic utterance")."""
import numpy as np
import torch

# reduced `config/models/visinger.yaml` (same keys the model reads, small sizes so fixtures stay small)
SMALL_HPARAMS = dict(
    hidden_size=32, p_dropout=0.1, enc_layers=2, ffn_kernel_size=9, ffn_filter_channels=64, num_heads=2,
    use_pos_embed=True, dec_blocks="1", dec_kernel_size=[3, 7, 11], dec_dilation_sizes=[[1, 3, 5]] * 3,
    upsample_rates=[5, 3], initial_upsample_channels=64, upsample_kernel_sizes=[11, 7], gin_channels=16,
    frame_prior_layers=2, use_pitch_embed=True, pitch_predictor_layers=2, use_phoneme_pred=True,
    phoneme_predictor_layers=1, predictor_grad=0.1, segment_size=32, num_mel_bins=16, num_linear_bins=33,
    use_spk_id=True, use_spk_embed=False, num_spk=2)


def full_hparams():
    """The values of config/models/visinger.yaml + base_task.yaml + preprocess.yaml that the model constructor reads."""
    return dict(
        hidden_size=192, p_dropout=0.1, enc_layers=6, ffn_kernel_size=9, ffn_filter_channels=768, num_heads=2,
        use_pos_embed=True, dec_blocks="1", dec_kernel_size=[3, 7, 11], dec_dilation_sizes=[[1, 3, 5]] * 3,
        upsample_rates=[5, 5, 3, 2, 2], initial_upsample_channels=512, upsample_kernel_sizes=[11, 11, 7, 4, 4],
        gin_channels=256, frame_prior_layers=4, use_pitch_embed=True, pitch_predictor_layers=6, use_phoneme_pred=True,
        phoneme_predictor_layers=2, predictor_grad=0.1, segment_size=32, num_mel_bins=128, num_linear_bins=1025,
        use_spk_id=True, use_spk_embed=False, num_spk=1)


def synth_utterances(seed, n, min_frames=120, max_frames=1280, n_spk=1, lengths=None):
    """`n` right-padded utterances in the collater's tensors (tasks/dataset_utils.py:170-208 names): text_tokens,
    note_pitch, note_dur int64 [B, T_ph] (0 = pad), mel2ph int64 [B, T] (1-based, 0 = pad), spk_ids [B].

    Structure mirrors ko_sing + get_note2dur: syllables of 1-3 phonemes sharing one pitch / duration id, onset and coda
    get 3 frames and the nucleus the rest, <BOS>/<EOS> at the ends with pitch 0 / dur 0, 10 % rests."""
    rng = np.random.default_rng(seed)
    utts = []
    for u in range(n):
        target = int(lengths[u]) if lengths is not None else int(rng.integers(min_frames, max_frames + 1))
        toks, pitch, dur, frames = [2], [0], [0], [3]            # <BOS>-like token, 3 frames
        total = 3
        while total < target - 3:
            syl = int(min(rng.integers(10, 61), target - 3 - total))
            if syl < 7:
                frames[-1] += syl
                total += syl
                break
            nph = int(rng.choice([1, 2, 3], p=[0.2, 0.5, 0.3]))
            rest = rng.random() < 0.1
            p_id = 0 if rest else int(rng.integers(37, 73))
            d_id = int(rng.integers(4, 131))
            if rest:
                nph = 1
            split = {1: [syl], 2: [3, syl - 3], 3: [3, syl - 6, 3]}[nph]
            for fr in split:
                toks.append(3 if rest else int(rng.integers(4, 72)))
                pitch.append(p_id)
                dur.append(d_id)
                frames.append(fr)
            total += syl
        toks.append(1); pitch.append(0); dur.append(0); frames.append(target - total)     # <EOS>
        mel2ph = np.concatenate([np.full(f, i + 1) for i, f in enumerate(frames) if f > 0])
        utts.append((np.array(toks), np.array(pitch), np.array(dur), mel2ph))
    Tph = max(len(u[0]) for u in utts)
    T = max(len(u[3]) for u in utts)

    def pad(a, L):
        return np.pad(a, (0, L - len(a)))

    return dict(text_tokens=torch.from_numpy(np.stack([pad(u[0], Tph) for u in utts])).long(),
                note_pitch=torch.from_numpy(np.stack([pad(u[1], Tph) for u in utts])).long(),
                note_dur=torch.from_numpy(np.stack([pad(u[2], Tph) for u in utts])).long(),
                mel2ph=torch.from_numpy(np.stack([pad(u[3], T) for u in utts])).long(),
                spk_ids=torch.from_numpy(rng.integers(0, n_spk, n)).long())


def config4_lengths(n, seed=1234):
    """BASELINE.json configs[3] / SURVEY.md 8d "Config 4": T_i = clip(round(80 * LogNormal(ln 5.6, 0.45)), 120, 1280)."""
    rng = np.random.default_rng(seed)
    return np.clip(np.round(80.0 * rng.lognormal(np.log(5.6), 0.45, n)), 120, 1280).astype(np.int64)


def full_model_mirror(seed=4321, precision="fp32"):
    """The full-hparams mirror model with seeded weights: constructor init under `seed`, flow `post` layers
    re-randomised (zero-initialised in the reference, SURVEY.md App. B-2).  tests/golden/make_golden_model_full.py loads
    exactly this state dict into the unmodified reference model, so the fixture holds outputs only."""
    from visinger_b200.models.visinger import VISinger
    torch.manual_seed(seed)
    m = VISinger(73, 117, 132, full_hparams(), precision=precision).eval()
    gen = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for f in range(4):
            post = m.flow.flows[2 * f].post
            post.weight.copy_(0.05 * torch.randn(post.weight.shape, generator=gen))
            post.bias.copy_(0.05 * torch.randn(post.bias.shape, generator=gen))
    return m


FULL_GOLDEN_B = 8
FULL_GOLDEN_WAV_STRIDE = 53


def full_model_batch():
    lengths = config4_lengths(64)[:FULL_GOLDEN_B]
    batch = synth_utterances(seed=1234, n=FULL_GOLDEN_B, lengths=lengths)
    T = batch["mel2ph"].shape[1]
    noise = torch.randn(FULL_GOLDEN_B, 192, T, generator=torch.Generator().manual_seed(11))
    return batch, noise, lengths
