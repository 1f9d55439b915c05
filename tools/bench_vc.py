"""Voice-conversion throughput: converted audio-seconds per second of SynthesizerTrn.voice_conversion plus the linear
spectrogram, at a size a user would convert, split per phase with CUDA events.

    python tools/bench_vc.py --config baker_v1 --batch 64 --seconds 8 --steps 5 --warmup 2 [--out FILE]

Synthetic seeded checkpoint (wetts_b200/synth.py, with enc_q) and seeded audio; lengths are ragged in
[0.75, 1] x --seconds.  The whole conversion (spectrogram -> voice_conversion) is timed end to end; the phases
(spectrogram, posterior encoder, forward flow, inverse flow, generator) are timed in separate passes through the block
entry points.  The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import wetts_b200  # noqa: E402
from wetts_b200 import synth  # noqa: E402
from wetts_b200.hparams import builtin_config  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:   # the number is still the card's; say the limit could not be read
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return ts


def run(cfg_name, B, seconds, steps, warmup, n_spk=4, seed=11):
    hps = builtin_config(cfg_name)
    S = hps.data.filter_length // 2 + 1
    sd = {**synth.make_state_dict(hps.model, 64, n_spk, seed=hps.train.seed),
          **synth.posterior_state_dict(hps.model, S, n_spk, seed=hps.train.seed + 1)}
    net = wetts_b200.build_model(hps, 64, n_spk, sd, "cuda")
    dev = net.device
    gen = torch.Generator().manual_seed(seed)
    sr = hps.data.sampling_rate
    L = int(seconds * sr)
    lengths = (L * (0.75 + 0.25 * torch.rand(B, generator=gen))).long().clamp_max(L)
    lengths[0] = L
    t = torch.arange(L, dtype=torch.float32)[None, :] / sr
    f = 100 + 800 * torch.rand(B, 1, generator=gen)
    audio = (0.3 * torch.sin(2 * torch.pi * f * t) + 0.02 * torch.randn(B, L, generator=gen))
    audio = (audio * (torch.arange(L)[None, :] < lengths[:, None])).to(dev)
    lengths = lengths.to(dev)
    src = torch.randint(0, n_spk, (B,), generator=gen).to(dev)
    tgt = torch.randint(0, n_spk, (B,), generator=gen).to(dev)
    spec, spec_lengths = net.spectrogram(audio, lengths)
    T = spec.shape[2]
    noise = torch.randn(B, hps.model.inter_channels, T, generator=gen).to(dev)

    def whole():
        sp, sl = net.spectrogram(audio, lengths)
        return net.voice_conversion(sp, sl, src, tgt, noise=noise)

    total = timed(whole, steps, warmup)
    g_src = net.emb_g(src)[:, :, None]
    g_tgt = net.emb_g(tgt)[:, :, None]
    z, _, _, y_mask = net.enc_q(spec, spec_lengths, g=g_src, noise=noise)
    z_p = net.flow(z, y_mask, g=g_src, reverse=False)
    z_hat = net.flow(z_p, y_mask, g=g_tgt, reverse=True)
    zin = z_hat * y_mask
    phases = {
        "spectrogram": timed(lambda: net.spectrogram(audio, lengths), steps, warmup),
        "posterior_encoder": timed(lambda: net.enc_q(spec, spec_lengths, g=g_src, noise=noise), steps, warmup),
        "flow_forward": timed(lambda: net.flow(z, y_mask, g=g_src, reverse=False), steps, warmup),
        "flow_inverse": timed(lambda: net.flow(z_p, y_mask, g=g_tgt, reverse=True), steps, warmup),
        "generator": timed(lambda: net.dec(zin, g=g_tgt), steps, warmup),
    }
    net.check_faults()
    audio_s = float(lengths.sum()) / sr
    med = sorted(total)[len(total) // 2]
    return {
        "config": cfg_name, "batch": B, "max_seconds": seconds, "frames": T, "audio_seconds": audio_s,
        "steps": steps, "warmup": warmup,
        "call_s_median": med, "call_s_all": total, "audio_seconds_per_second": audio_s / med,
        "phase_s_median": {k: sorted(v)[len(v) // 2] for k, v in phases.items()},
        "note": "spectrogram synchronises the stream (its lengths are checked on the host); the phases are timed "
                "in separate passes, so they need not add up to the call exactly",
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--config", action="append", help="builtin config (repeatable); default baker_v1 and multilingual_v3")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--seconds", type=float, default=8.0)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench_vc: no CUDA device (there is no CPU path to measure)")
    res = {"gpu": gpu_info(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%dT%H:%M:%S"),
           "runs": [run(c, a.batch, a.seconds, a.steps, a.warmup) for c in (a.config or ["baker_v1", "multilingual_v3"])]}
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
