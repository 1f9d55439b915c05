"""CPU-side checks: the C-ABI library loads and exports every declared symbol, host logic
(config mirror, synthetic checkpoints, loud failure without a GPU)."""
import json
import os
import re

import pytest
import torch

import wetts_b200
from wetts_b200 import _lib, synth
from wetts_b200.hparams import HParams, builtin_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from wetts_b200 import build
    build.build()
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "wetts_b200.h")).read()
    declared = set(re.findall(r"\b(wetts_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    for name in declared:
        assert hasattr(lib, name)
    assert b"sm_100a" in lib.wetts_version()


def test_hparams_mapping_protocol():
    hps = builtin_config("multilingual_v3")
    assert hps.data.sampling_rate == 16000 and hps["model"]["use_sdp"] is False
    assert "model" in hps and len(hps) == 3
    kw = dict(**hps.model)
    assert kw["upsample_rates"] == [8, 8, 4]
    h2 = HParams(a={"b": 1})
    assert h2.a.b == 1 and list(h2.keys()) == ["a"]


def test_synthetic_checkpoint_is_deterministic_and_nontrivial():
    hps = builtin_config("baker_v1")
    a = synth.make_state_dict(hps.model, 50, 1, seed=1234)
    b = synth.make_state_dict(hps.model, 50, 1, seed=1234)
    assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)
    assert synth.fingerprint(a) == synth.fingerprint(b)
    # tensors the reference zero-initialises must be non-zero (SURVEY §0 finding 5)
    assert a["flow.flows.0.post.weight"].abs().max() > 0
    assert a["dp.flows.1.proj.weight"].abs().max() > 0
    v, g = a["dec.ups.0.weight_v"], a["dec.ups.0.weight_g"]
    assert g.shape == (v.shape[0], 1, 1)          # ConvTranspose1d: per INPUT channel
    assert not torch.allclose(g.flatten(), v.reshape(v.shape[0], -1).norm(dim=1))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_gpu():
    hps = builtin_config("multilingual_v3")
    net = wetts_b200.SynthesizerTrn(10, 513, 32, n_speakers=1, **hps.model)
    with pytest.raises(wetts_b200.WettsError):
        net.to("cuda")
    with pytest.raises(wetts_b200.WettsError):
        net.infer(torch.zeros(1, 4, dtype=torch.long), torch.tensor([4]), torch.tensor([0]))


def test_unsupported_variants_raise():
    hps = builtin_config("multilingual_v3")
    with pytest.raises(NotImplementedError):
        wetts_b200.SynthesizerTrn(10, 513, 32, n_speakers=1, vocoder_type="bigvgan", **hps.model)
    with pytest.raises(NotImplementedError):    # only the 'pre_conv' transformer flow (vits2_vocos_v1 recipe) is built
        wetts_b200.SynthesizerTrn(10, 513, 32, n_speakers=1, use_transformer_flows=True, transformer_flow_type="fft", **hps.model)


def test_vits2_vocos_recipe_constructs_and_maps_its_config():
    """SURVEY.md 8f rank 4: the reference's vits2_vocos_v1 recipe file is accepted unchanged"""
    hps = builtin_config("baker_vits2_vocos_v1")
    net = wetts_b200.SynthesizerTrn(64, 513, 32, n_speakers=1, **hps.model)
    c = net._engine.cfg
    assert (c.vocoder_type, c.flow_type) == (1, 1)
    assert (c.vocos_channels, c.vocos_h_channels, c.vocos_out_channels, c.vocos_num_layers) == (512, 1536, 1026, 8)
    assert (c.vocos_n_fft, c.vocos_hop_length) == (1024, 256) and net._engine.upsample == 256
    sd = synth.make_state_dict(hps.model, 64, 1, seed=1234)
    assert "dec.layers.7.scale" in sd and "flow.flows.6.pre_transformer.attn_layers.1.conv_q.weight" in sd
    assert "dec.conv_pre.weight" not in sd


def test_reference_loads_synthetic_checkpoint():
    """The synthetic state dict must load into the reference's own module: against the reference's state-dict layout
    (name -> shape, recorded by oracle/gen_golden.py), nothing unexpected, no shape mismatch, and the only missing
    tensors are the ones infer never reads (posterior encoder, iSTFT window, VITS2 post_transformer)."""
    layout = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_state_dict_layout.json")))
    assert set(layout) == {"multilingual_v3", "baker_v1"}

    def unused(k):
        return k.startswith("enc_q.") or k.startswith("dec.istft.") or ".post_transformer." in k
    for cfg, spec in layout.items():
        hps = builtin_config(cfg)
        sd = synth.make_state_dict(hps.model, spec["n_vocab"], spec["n_speakers"], seed=3)
        ref = spec["state_dict"]
        assert [k for k in sd if k not in ref] == [], cfg
        assert [k for k in sd if list(sd[k].shape) != ref[k]] == [], cfg
        assert [k for k in ref if k not in sd and not unused(k)] == [], cfg


def test_mma_issue_paths_stay_in_the_uniform_datapath():
    """DESIGN.md 4.5 as a test: in the built library no tcgen05.mma of a production kernel sits under a per-thread
    predicate, and no vector -> uniform register move (R2UR) sits between the MMAs of an issue loop of the f16 kernels
    (the EPI_MRF instantiation of the per-layer kernel once had 170 of them: found by eye, now found by this test)."""
    import shutil
    import sys
    if not (shutil.which("cuobjdump") and shutil.which("c++filt")):
        pytest.skip("cuobjdump / c++filt not available")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_issue_scan as S
    from wetts_b200 import build
    rows = [r for r in S.scan(build.build()) if not S.is_profiling(r["kernel"])]
    names = " ".join(r["kernel"] for r in rows)
    for must in ("fused_mrf16_kernel<32", "fused_mrf16_kernel<64", "conv1d_tc16_kernel<512, 1, 2>", "conv1d_tc16r_kernel<3, false>",
                 "rel_attention_tc_kernel<true>"):
        assert must in names, f"{must} not found in the library's SASS"
    for r in rows:
        assert r["per_thread_predicated_mmas"] == 0, r
        if re.search(r"fused_mrf16_kernel|conv1d_tc16_kernel|conv1d_tc16r_kernel", r["kernel"]):
            assert r["r2ur_between_mmas"] == 0, r
        else:
            assert r["r2ur_between_mmas"] <= 8, r     # 3xTF32 twins, attention (two issue regions)
