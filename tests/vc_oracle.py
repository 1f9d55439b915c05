"""CPU oracle of the voice-conversion path: a functional restatement of the reference's
`SynthesizerTrn.voice_conversion` (wetts/vits/model/models.py:369-376), its posterior encoder
(encoders.py:60-99), the forward direction of the flow (flows.py:442-449 with 146-176 / 494-513) and
`spectrogram_torch` (utils/mel_processing.py:42-93).

Test infrastructure, in the style of oracle/vits_oracle.py, whose pieces (weight-norm folding, WN,
the inverse flow, the generators) it reuses.  Pinned against the reference by the tests/golden/vc_*.npz
fixtures (tools/gen_vc_golden.py runs the real reference to make them).
"""
import math

import torch
import torch.nn.functional as F

from oracle import vits_oracle as O

POSTERIOR_LAYERS = 16   # models.py:124-132: PosteriorEncoder(spec_channels, inter, hidden, 5, 1, 16, gin)


def posterior_encoder(w, cfg, y, y_lengths, g, noise):
    """encoders.py:91-99 on a folded state dict: (z, m, logs, y_mask).  noise [B,inter,T] ~ N(0,1)."""
    cfg = O._plain(cfg)
    H, C = cfg["hidden_channels"], cfg["inter_channels"]
    m3 = O.seq_mask(y_lengths, y.shape[2])[:, None, :]
    x = F.conv1d(y, w["enc_q.pre.weight"], w["enc_q.pre.bias"]) * m3
    x = O.wn(w, "enc_q.enc", x, m3, g, H, n_layers=POSTERIOR_LAYERS)
    stats = F.conv1d(x, w["enc_q.proj.weight"], w["enc_q.proj.bias"]) * m3
    m, logs = stats[:, :C], stats[:, C:]
    z = (m + noise * torch.exp(logs)) * m3
    return z, m, logs, m3


def flow_forward(w, cfg, z, y_m3, g):
    """flows.py:442-449 with reverse=False: coupling layers 0, 2, 4, 6, each followed by a Flip;
    x1 = m + x1 * mask (mean_only, flows.py:505)."""
    cfg = O._plain(cfg)
    H = cfg["hidden_channels"]
    half = cfg["inter_channels"] // 2
    tflow = cfg.get("use_transformer_flows", False)
    for f in (0, 2, 4, 6):
        p = f"flow.flows.{f}"
        x0, x1 = z[:, :half], z[:, half:]
        xin = x0
        if tflow:   # flows.py:146-151
            xin = O.plain_encoder(w, p + ".pre_transformer", x0 * y_m3, y_m3[:, 0], 2, 2, 3) + x0
        h = F.conv1d(xin, w[p + ".pre.weight"], w[p + ".pre.bias"]) * y_m3
        h = O.wn(w, p + ".enc", h, y_m3, g, H)
        m = F.conv1d(h, w[p + ".post.weight"], w[p + ".post.bias"]) * y_m3
        x1 = m + x1 * y_m3
        z = torch.flip(torch.cat([x0, x1], dim=1), [1])
    return z


def spectrogram(audio, lengths, n_fft, hop):
    """spectrogram_torch(center=False) of each utterance on its own (reflection padding by (n_fft - hop) / 2 at the
    utterance's own length, periodic Hann window, onesided real DFT, sqrt(re^2 + im^2 + 1e-6)), zero-padded to the
    frame count of the batch length L.  audio [B,L] -> (spec [B, n_fft/2+1, F], spec_lengths [B])."""
    B, L = audio.shape
    pad = (n_fft - hop) // 2
    Fmax = 1 + (L + 2 * pad - n_fft) // hop
    K = n_fft // 2 + 1
    n = torch.arange(n_fft, dtype=torch.float64)
    k = torch.arange(K, dtype=torch.float64)
    ang = 2 * math.pi * ((k[:, None] * n[None, :]) % n_fft) / n_fft
    win = torch.hann_window(n_fft, periodic=True, dtype=torch.float64)
    cosb, sinb = torch.cos(ang) * win, torch.sin(ang) * win                 # [K, N]
    spec = torch.zeros(B, K, Fmax)
    lens = torch.zeros(B, dtype=torch.long)
    for b in range(B):
        Lb = int(lengths[b])
        x = F.pad(audio[b:b + 1, None, :Lb].double(), (pad, pad), mode="reflect")[0, 0]
        frames = x.unfold(0, n_fft, hop)                                    # [F_b, N]
        re, im = frames @ cosb.t(), frames @ sinb.t()
        spec[b, :, : frames.shape[0]] = torch.sqrt(re * re + im * im + 1e-6).t().float()
        lens[b] = frames.shape[0]
    return spec, lens


def voice_conversion(sd, cfg, y, y_lengths, sid_src, sid_tgt, noise, folded=False):
    """models.py:369-376.  Returns dict with o_hat, y_mask, z, m_q, logs_q, z_p, z_hat."""
    w = sd if folded else O.fold_weight_norm(sd)
    g_src = F.embedding(sid_src, w["emb_g.weight"])[:, :, None]
    g_tgt = F.embedding(sid_tgt, w["emb_g.weight"])[:, :, None]
    z, m_q, logs_q, y_m3 = posterior_encoder(w, cfg, y, y_lengths, g_src, noise)
    z_p = flow_forward(w, cfg, z, y_m3, g_src)
    z_hat = O.flow_reverse(w, cfg, z_p, y_m3, g_tgt)
    o_hat = O.generator(w, cfg, z_hat * y_m3, g_tgt)
    return dict(o_hat=o_hat, y_mask=y_m3, z=z, m_q=m_q, logs_q=logs_q, z_p=z_p, z_hat=z_hat)
