"""Voice conversion without a GPU: the CPU oracle (tests/vc_oracle.py) against the reference-generated vc_* fixtures,
the synthetic posterior-encoder weights against the reference's state-dict layout, and the new Python entry points
failing cleanly when there is no device."""
import json
import os

import numpy as np
import pytest
import torch

from tests import vc_oracle
from tests.golden_util import GOLDEN_DIR, rel_rms_err
from wetts_b200 import synth
from wetts_b200.hparams import builtin_config

VC_CASES = ["vc_v1_ragged", "vc_v3_long", "vc_vits2_vocos_mel"]
ORACLE_TOL = 1e-5


def load_vc_case(name):
    """fixture arrays, config and the synthetic checkpoint (with enc_q) it was made with"""
    d = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    g = {k: d[k] for k in d.files}
    hps = builtin_config(str(g["config"]))
    n_vocab, n_spk, S = int(g["n_vocab"]), int(g["n_speakers"]), int(g["spec_channels"])
    sd = synth.make_state_dict(hps.model, n_vocab, n_spk, seed=int(g["ckpt_seed"]))
    sd_q = synth.posterior_state_dict(hps.model, S, n_spk, seed=int(g["posterior_seed"]))
    for part, key in ((sd, "fingerprint"), (sd_q, "posterior_fingerprint")):
        fp = synth.fingerprint(part)
        assert abs(fp - float(g[key])) <= 1e-9 * abs(fp), "synthetic checkpoint differs from the fixture's"
    t = {k: torch.from_numpy(v) for k, v in g.items() if v.dtype.kind in "fi" and v.ndim > 0}
    return hps, {**sd, **sd_q}, g, t


@pytest.mark.parametrize("name", VC_CASES)
def test_oracle_matches_reference_voice_conversion(name):
    hps, sd, g, t = load_vc_case(name)
    if "audio" in t:
        spec, lens = vc_oracle.spectrogram(t["audio"], t["audio_lengths"], hps.data.filter_length, hps.data.hop_length)
        assert torch.equal(lens, t["spec_lengths"])
        assert rel_rms_err(spec, t["spec"]) < ORACLE_TOL
    r = vc_oracle.voice_conversion(sd, hps.model, t["spec"], t["spec_lengths"], t["sid_src"], t["sid_tgt"], t["noise"])
    for k in ("z", "m_q", "logs_q", "z_p", "z_hat", "o_hat", "y_mask"):
        assert r[k].shape == t[k].shape, k
        assert rel_rms_err(r[k], t[k]) < ORACLE_TOL, (k, rel_rms_err(r[k], t[k]))


def test_posterior_state_dict_matches_reference_layout():
    with open(os.path.join(GOLDEN_DIR, "reference_state_dict_layout.json")) as f:
        layout = json.load(f)
    for cfg_name, entry in layout.items():
        hps = builtin_config(cfg_name)
        ref = {k: v for k, v in entry["state_dict"].items() if k.startswith("enc_q.")}
        ours = synth.posterior_state_dict(hps.model, hps.data.filter_length // 2 + 1, entry["n_speakers"], seed=1)
        assert {k: list(v.shape) for k, v in ours.items()} == ref


def test_make_state_dict_still_omits_enc_q():
    hps = builtin_config("baker_v1")
    assert not [k for k in synth.make_state_dict(hps.model, 40, 2, seed=3) if k.startswith("enc_q.")]


def _model(cfg_name="baker_v1", n_spk=4):
    from wetts_b200 import SynthesizerTrn
    hps = builtin_config(cfg_name)
    return hps, SynthesizerTrn(40, hps.data.filter_length // 2 + 1, 32, n_speakers=n_spk, **hps.model)


def test_voice_conversion_calls_fail_without_a_device():
    from wetts_b200 import WettsError
    try:
        hps, net = _model()
    except WettsError:
        pytest.skip("libwetts_b200 is not built")
    y, lens, sid = torch.rand(1, 513, 8), torch.tensor([8]), torch.tensor([0])
    with pytest.raises(WettsError):
        net.voice_conversion(y, lens, sid, sid)
    with pytest.raises(WettsError):
        net.spectrogram(torch.zeros(1, 4000), torch.tensor([4000]))
    with pytest.raises(WettsError):
        net.enc_q(y, lens)
    with pytest.raises(WettsError):
        net.flow(torch.zeros(1, 192, 8), torch.ones(1, 1, 8), reverse=False)
    if not torch.cuda.is_available():
        with pytest.raises(WettsError):
            net.to("cuda")


def test_posterior_channel_count_is_checked_at_load():
    from wetts_b200 import WettsError
    try:
        hps, net = _model()
    except WettsError:
        pytest.skip("libwetts_b200 is not built")
    sd_q = synth.posterior_state_dict(hps.model, 100, 4, seed=1)
    with pytest.raises(ValueError, match="spec_channels"):
        net.load_state_dict(sd_q)
