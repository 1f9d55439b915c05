"""Generate tests/golden/*.npz and tests/golden/reference_state_dict_layout.json by running the REAL reference
(needs a checkout of wetts; see oracle/ref_harness.py).

    python -m oracle.gen_golden [NAME ...]            # from the repo root; NAME = a case or the layout file

For each case: build the seeded synthetic checkpoint (wetts_b200/synth.py), load it into
the reference's own SynthesizerTrn (`/root/reference/wetts/vits/model/models.py`), run
`infer` with injected noise, and store inputs + the reference's outputs and intermediates.
The fixtures pin oracle/vits_oracle.py (tests/test_oracle_golden.py) and are the final
arbiter for the CUDA path (tests/test_parity_gpu.py).  Test infrastructure only.
"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import ref_harness  # noqa: E402
from wetts_b200 import synth  # noqa: E402
from wetts_b200.hparams import builtin_config  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name, config, n_vocab, n_speakers, x_lengths, (noise_scale, length_scale, noise_scale_w), input seed
CASES = [
    ("v3_ragged", "multilingual_v3", 256, 2, [12, 9], (0.667, 4.0, 0.8), 5678),
    ("v3_single", "multilingual_v3", 256, 2, [7], (0.667, 4.0, 0.8), 5679),
    ("v1_ragged", "baker_v1", 256, 1, [10, 6], (0.667, 3.0, 0.8), 5680),
    ("v2_short", "baker_v2", 256, 1, [3, 4], (0.667, 3.0, 0.8), 5681),
    # BASELINE.json configs[4] family: AISHELL-3 v1 (44.1 kHz, 218 speakers, SDP, HiFi-GAN V1), longer ragged text
    ("aishell3_long", "aishell3_v1", 256, 218, [128, 80], (0.667, 2.0, 0.8), 5682),
    # BASELINE.json configs[0]: Baker v1, batch 1, the CLI utterance (SURVEY.md 8d config 1), CLI scales
    ("baker_v1_cli", "baker_v1", None, 1, "cli", (0.667, 1.0, 0.8), 5683),
    # the route bench.py measures: multilingual v3 at Tx = 128, ragged (every text-encoder / duration-predictor conv takes
    # the tcgen05 kernel at T >= 64); gating fixture for own-duration equality on that route (VERDICT r1 item 1c)
    ("v3_tx128", "multilingual_v3", 256, 2, [128, 97, 64], (0.667, 2.0, 0.8), 5684),
    # SURVEY.md 8f rank 4: the vits2_vocos_v1 recipe (Vocos iSTFT decoder + VITS2 'pre_conv' transformer flows, SDP)
    ("vits2_vocos_short", "baker_vits2_vocos_v1", 64, 1, [9, 6], (0.667, 2.0, 0.8), 5685),
]

# SURVEY.md 8(d) config 1: phoneme string of the wetts.cli example utterance and the synthetic phones.txt rule
# (`sil 0`, then the sorted remaining symbols; examples/baker/run.sh:38-41)
CLI_TOKENS = "sil j in1 #0 t ian1 #0 t ian1 #0 q i4 #0 z en3 #0 m e5 #0 ^ iang4 #4".split()
CLI_VOCAB = ["sil"] + sorted(set(CLI_TOKENS) - {"sil"})

# state-dict layout (name -> shape) of the reference's SynthesizerTrn, which tests/test_host_cpu.py checks the synthetic
# checkpoint against: config, n_vocab, n_speakers
LAYOUT_CASES = [("multilingual_v3", 40, 2), ("baker_v1", 40, 2)]
LAYOUT_FILE = "reference_state_dict_layout.json"


def write_state_dict_layout():
    out = {}
    for cfg_name, n_vocab, n_spk in LAYOUT_CASES:
        hps = builtin_config(cfg_name)
        net = ref_harness.build_reference_model(hps, n_vocab, n_spk, synth.make_state_dict(hps.model, n_vocab, n_spk, seed=3))
        out[cfg_name] = {"n_vocab": n_vocab, "n_speakers": n_spk,
                         "state_dict": {k: list(v.shape) for k, v in net.state_dict().items()}}
    path = os.path.join(GOLDEN_DIR, LAYOUT_FILE)
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print(LAYOUT_FILE, {k: len(v["state_dict"]) for k, v in out.items()}, os.path.getsize(path) // 1024, "KiB")


def make_inputs(n_vocab, n_speakers, x_lengths, seed, max_frames_per_phone=40):
    gen = torch.Generator().manual_seed(seed)
    B, Tx = len(x_lengths), max(x_lengths)
    x = torch.randint(0, n_vocab, (B, Tx), generator=gen)
    lens = torch.tensor(x_lengths, dtype=torch.long)
    x = x * (torch.arange(Tx)[None, :] < lens[:, None])  # zero-pad ids like gpu_triton model.py:117-130
    sid = torch.randint(0, n_speakers, (B,), generator=gen)
    noise_w = torch.randn(B, 2, Tx, generator=gen)
    noise_z = torch.randn(B, 192, Tx * max_frames_per_phone, generator=gen)
    return x, lens, sid, noise_w, noise_z


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(1)
    only = set(sys.argv[1:])
    if not only or LAYOUT_FILE in only:
        write_state_dict_layout()
    for name, cfg_name, n_vocab, n_spk, x_lengths, scales, seed in CASES:
        if only and name not in only:
            continue
        hps = builtin_config(cfg_name)
        cli_ids = None
        if x_lengths == "cli":
            n_vocab = len(CLI_VOCAB)
            cli_ids = [CLI_VOCAB.index(t) for t in CLI_TOKENS]
            x_lengths = [len(cli_ids)]
        sd = synth.make_state_dict(hps.model, n_vocab, n_spk, seed=hps.train.seed)
        net = ref_harness.build_reference_model(hps, n_vocab, n_spk, sd)
        x, lens, sid, noise_w, noise_z = make_inputs(n_vocab, n_spk, x_lengths, seed)
        if cli_ids is not None:
            x = torch.tensor([cli_ids], dtype=torch.long)
        ns, ls, nsw = scales
        r = ref_harness.reference_infer(net, x, lens, sid, ns, ls, nsw, noise_w, noise_z)
        Ty = r["z"].shape[2]
        y_lengths = r["y_mask"].sum(dim=[1, 2]).long()
        out = dict(
            x=x.numpy(), x_lengths=lens.numpy(), sid=sid.numpy(), noise_w=noise_w.numpy(),
            noise_z=noise_z[:, :, :Ty].numpy(), scales=np.array(scales, dtype=np.float64),
            fingerprint=np.array(synth.fingerprint(sd)), n_vocab=np.array(n_vocab), n_speakers=np.array(n_spk),
            config=np.array(cfg_name), ckpt_seed=np.array(hps.train.seed),
            h=r["h"].numpy(), m_p_tx=r["m_p_tx"].numpy(), logs_p_tx=r["logs_p_tx"].numpy(),
            logw=r["logw"].numpy(), w_ceil=r["w_ceil"].numpy(), y_lengths=y_lengths.numpy(),
            z_p=r["z_p"].numpy(), z=r["z"].numpy(), o=r["o"].numpy(),
            attn_argmax=r["attn"][:, 0].argmax(dim=-1).numpy().astype(np.int32),
            attn_rowsum=r["attn"][:, 0].sum(dim=-1).numpy(),
        )
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print(name, "Ty", Ty, "y_lengths", y_lengths.tolist(), "o rms", float(r["o"].pow(2).mean().sqrt()),
              "z rms", float(r["z"].pow(2).mean().sqrt()), os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
