"""Generate tests/golden/vc_*.npz by running the REAL reference's voice conversion (needs a checkout of wetts; see
oracle/ref_harness.py).  Writes only the vc_* files; the other fixtures are made by oracle/gen_golden.py.

    python tools/gen_vc_golden.py [NAME ...]          # from the repo root

For each case: the seeded synthetic checkpoint (wetts_b200/synth.py make_state_dict + posterior_state_dict) is loaded
into the reference's own SynthesizerTrn, built with the case's spec_channels; the features are the reference's
`spectrogram_torch` of seeded audio, applied to each utterance at its own length and zero-padded as the reference's
collate does (or, for the mel posterior encoder, seeded positive features given directly); then
`voice_conversion(y, y_lengths, sid_src, sid_tgt)` runs with the posterior encoder's randn_like draw injected.
Inputs and the reference's spec, spec_lengths, z, m_q, logs_q, z_p, z_hat, o_hat and y_mask are stored.
"""
import contextlib
import io
import os
import sys
import warnings

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_harness  # noqa: E402
from wetts_b200 import synth  # noqa: E402
from wetts_b200.hparams import builtin_config  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
N_VOCAB = 64

# name, config, n_speakers, audio lengths in samples (None: mel features given directly, lengths in frames),
# sid_src, sid_tgt, input seed
VC_CASES = [
    # HiFi-GAN ResBlock1, ragged, lengths not multiples of hop; utterance 1 converts to its own speaker
    ("vc_v1_ragged", "baker_v1", 4, [7000, 5123, 3001], [0, 2, 3], [1, 2, 0], 6001),
    # ResBlock2; utterance 0 has >= 64 frames (tcgen05 conv route), utterance 1 fewer
    ("vc_v3_long", "multilingual_v3", 2, [17000, 9000], [0, 1], [1, 0], 6002),
    # VITS2 + Vocos with the 100-channel mel posterior encoder (features given directly; flow_type 1 forward)
    ("vc_vits2_vocos_mel", "baker_vits2_vocos_v1", 2, None, [1, 0], [0, 0], 6003),
]
MEL_FRAMES = [23, 17]


def spec_channels_of(hps):
    if "use_mel_posterior_encoder" in hps.model.keys() and hps.model.use_mel_posterior_encoder:
        return hps.data.n_mel_channels
    return hps.data.filter_length // 2 + 1


def seeded_audio(lengths, sr, gen):
    """sums of three sinusoids plus a little noise, in [-1, 1], zero beyond each length"""
    B, L = len(lengths), max(lengths)
    t = torch.arange(L, dtype=torch.float64)[None, :] / sr
    f = 80 + 900 * torch.rand(B, 3, generator=gen, dtype=torch.float64)
    a = 0.1 + 0.25 * torch.rand(B, 3, generator=gen, dtype=torch.float64)
    x = (a[:, :, None] * torch.sin(2 * torch.pi * f[:, :, None] * t[:, None, :])).sum(dim=1)
    x = x + 0.02 * torch.randn(B, L, generator=gen, dtype=torch.float64)
    x = x.clamp(-1, 1).float()
    return x * (torch.arange(L)[None, :] < torch.tensor(lengths)[:, None])


def build_reference_vc_model(hps, n_speakers, spec_channels, state_dict):
    SynthesizerTrn = ref_harness.import_reference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        net = SynthesizerTrn(N_VOCAB, spec_channels, hps.train.segment_size // hps.data.hop_length,
                             n_speakers=n_speakers, **hps.model).eval()
    missing, unexpected = net.load_state_dict(state_dict, strict=False)
    assert not unexpected, unexpected
    unused = [k for k in missing if not (k.startswith("dec.istft.") or ".post_transformer." in k)]
    assert not unused, unused
    return net


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(1)
    only = set(sys.argv[1:])
    ref_harness.import_reference()
    from utils.mel_processing import spectrogram_torch   # the reference's own, importable once import_reference ran
    for name, cfg_name, n_spk, lengths, sid_src, sid_tgt, seed in VC_CASES:
        if only and name not in only:
            continue
        hps = builtin_config(cfg_name)
        S = spec_channels_of(hps)
        sd = synth.make_state_dict(hps.model, N_VOCAB, n_spk, seed=hps.train.seed)
        sd_q = synth.posterior_state_dict(hps.model, S, n_spk, seed=hps.train.seed + 1)
        net = build_reference_vc_model(hps, n_spk, S, {**sd, **sd_q})
        gen = torch.Generator().manual_seed(seed)
        out = {}
        if lengths is not None:
            n_fft, hop = hps.data.filter_length, hps.data.hop_length
            audio = seeded_audio(lengths, hps.data.sampling_rate, gen)
            specs = []
            with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
                warnings.simplefilter("ignore")
                for b, Lb in enumerate(lengths):
                    specs.append(spectrogram_torch(audio[b:b + 1, :Lb], n_fft, hps.data.sampling_rate, hop,
                                                   hps.data.win_length, center=False)[0])
            spec_lengths = torch.tensor([s.shape[1] for s in specs])
            Tb = 1 + (max(lengths) + (n_fft - hop) - n_fft) // hop     # frames of the batch length
            y = torch.stack([F.pad(s, (0, Tb - s.shape[1])) for s in specs])
            out.update(audio=audio.numpy(), audio_lengths=np.array(lengths, dtype=np.int64))
        else:
            T = max(MEL_FRAMES)
            spec_lengths = torch.tensor(MEL_FRAMES)
            y = torch.exp(0.5 * torch.randn(len(MEL_FRAMES), S, T, generator=gen)) * 0.5
            y = y * (torch.arange(T)[None, None, :] < spec_lengths[:, None, None])
        B, _, T = y.shape
        noise = torch.randn(B, hps.model.inter_channels, T, generator=gen)
        src, tgt = torch.tensor(sid_src), torch.tensor(sid_tgt)
        with torch.no_grad(), ref_harness.injected_noise(None, noise):
            y_lengths = spec_lengths.clone()
            g_src = net.emb_g(src).unsqueeze(-1)
            z, m_q, logs_q, y_mask = net.enc_q(y, y_lengths, g=g_src)
            o_hat, y_mask2, (z2, z_p, z_hat) = net.voice_conversion(y, y_lengths, src, tgt)
        assert torch.equal(z, z2) and torch.equal(y_mask, y_mask2)
        out.update(
            spec=y.numpy(), spec_lengths=spec_lengths.numpy().astype(np.int64), sid_src=src.numpy(), sid_tgt=tgt.numpy(),
            noise=noise.numpy(), config=np.array(cfg_name), n_vocab=np.array(N_VOCAB), n_speakers=np.array(n_spk),
            spec_channels=np.array(S), ckpt_seed=np.array(hps.train.seed), posterior_seed=np.array(hps.train.seed + 1),
            fingerprint=np.array(synth.fingerprint(sd)), posterior_fingerprint=np.array(synth.fingerprint(sd_q)),
            z=z.numpy(), m_q=m_q.numpy(), logs_q=logs_q.numpy(), z_p=z_p.numpy(), z_hat=z_hat.numpy(),
            o_hat=o_hat.numpy(), y_mask=y_mask.numpy(),
        )
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print(name, "T", T, "spec_lengths", spec_lengths.tolist(), "logs_q range",
              (float(logs_q.min()), float(logs_q.max())), "z rms", float(z.pow(2).mean().sqrt()),
              "o_hat rms", float(o_hat.pow(2).mean().sqrt()), os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
