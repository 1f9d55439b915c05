"""Voice conversion on the GPU (models.py:369-376) against the reference-generated vc_* fixtures: the linear spectrogram,
the posterior encoder, the forward flow and the whole conversion on every conv route, plus round trips, batch composition
and the error paths."""
import pytest
import torch

from tests.golden_util import rel_rms_err
from tests.test_vc_cpu import VC_CASES, load_vc_case
from wetts_b200 import synth

pytestmark = pytest.mark.gpu

SPEC_TOL = 1e-4
BLOCK_TOL = 3e-4
E2E_TOL = 1e-3
ROUTES = [(1, 16), (1, 32), (0, 16)]   # (tensor_cores, tensor_format)


def _net(name):
    import wetts_b200
    hps, sd, g, t = load_vc_case(name)
    net = wetts_b200.build_model(hps, int(g["n_vocab"]), int(g["n_speakers"]), sd, "cuda")
    return hps, net, t


@pytest.mark.parametrize("name", VC_CASES)
def test_blocks_against_reference(name):
    hps, net, t = _net(name)
    dev = net.device
    if "audio" in t:
        spec, lens = net.spectrogram(t["audio"], t["audio_lengths"])
        spec = spec.cpu()
        assert torch.equal(lens.cpu(), t["spec_lengths"])
        assert spec.shape == t["spec"].shape
        e = rel_rms_err(spec, t["spec"])
        print(f"{name}: spectrogram {e:.3e}")
        assert e < SPEC_TOL
        for b, n in enumerate(t["spec_lengths"].tolist()):
            assert torch.all(spec[b, :, n:] == 0)
    g_src = net.emb_g(t["sid_src"])[:, :, None]
    z, m, logs, y_mask = net.enc_q(t["spec"], t["spec_lengths"], g=g_src, noise=t["noise"])
    errs = {k: rel_rms_err(v.cpu(), t[r]) for k, v, r in (("m", m, "m_q"), ("logs", logs, "logs_q"), ("z", z, "z"))}
    assert torch.equal(y_mask.cpu(), t["y_mask"])
    z_p = net.flow(t["z"].to(dev), y_mask, g=g_src, reverse=False)
    errs["z_p"] = rel_rms_err(z_p.cpu(), t["z_p"])
    print(name, {k: f"{v:.3e}" for k, v in errs.items()})
    assert all(v < BLOCK_TOL for v in errs.values()), errs


@pytest.mark.parametrize("route", ROUTES, ids=lambda r: f"tc{r[0]}_fmt{r[1]}")
@pytest.mark.parametrize("name", VC_CASES)
def test_voice_conversion_end_to_end(name, route):
    hps, net, t = _net(name)
    net.set_option("tensor_cores", route[0]).set_option("tensor_format", route[1])
    o, y_mask, (z, z_p, z_hat) = net.voice_conversion(t["spec"], t["spec_lengths"], t["sid_src"], t["sid_tgt"], noise=t["noise"])
    net.check_faults()
    assert o.shape == t["o_hat"].shape
    assert torch.equal(y_mask.cpu(), t["y_mask"])
    errs = {k: rel_rms_err(v.cpu(), t[k]) for k, v in (("z", z), ("z_p", z_p), ("z_hat", z_hat))}
    errs["o_hat"] = rel_rms_err(o.cpu(), t["o_hat"])
    print(name, route, {k: f"{v:.3e}" for k, v in errs.items()})
    assert errs["z"] < BLOCK_TOL and errs["z_p"] < BLOCK_TOL and errs["z_hat"] < BLOCK_TOL
    assert errs["o_hat"] < E2E_TOL


@pytest.mark.parametrize("name", VC_CASES)
def test_round_trips(name):
    hps, net, t = _net(name)
    dev = net.device
    y_mask = t["y_mask"].to(dev)
    g_src = net.emb_g(t["sid_src"])[:, :, None]
    z = t["z"].to(dev)
    back = net.flow(net.flow(z, y_mask, g=g_src, reverse=False), y_mask, g=g_src, reverse=True)
    e = rel_rms_err(back.cpu(), t["z"])
    print(f"{name}: inverse(forward(z)) vs z {e:.3e}")
    assert e < BLOCK_TOL
    o, _, (zq, _, z_hat) = net.voice_conversion(t["spec"], t["spec_lengths"], t["sid_src"], t["sid_tgt"], noise=t["noise"])
    for b in range(zq.shape[0]):
        if int(t["sid_src"][b]) == int(t["sid_tgt"][b]):
            eb = rel_rms_err(z_hat[b].cpu(), zq[b].cpu())
            print(f"{name}: utterance {b} converted to its own speaker, z_hat vs z {eb:.3e}")
            assert eb < BLOCK_TOL


@pytest.mark.parametrize("name", ["vc_v1_ragged", "vc_v3_long"])
def test_batch_composition(name):
    """One utterance converted alone equals the same utterance in the ragged batch: z, z_p, z_hat on its valid frames and
    the audio on the samples whose receptive field lies inside the utterance (16 frames short of its end)."""
    hps, net, t = _net(name)
    U = net._engine.upsample
    o, _, zs = net.voice_conversion(t["spec"], t["spec_lengths"], t["sid_src"], t["sid_tgt"], noise=t["noise"])
    for b, n in enumerate(t["spec_lengths"].tolist()):
        sl = slice(b, b + 1)
        ob, _, zb = net.voice_conversion(t["spec"][sl, :, :n], t["spec_lengths"][sl], t["sid_src"][sl], t["sid_tgt"][sl],
                                         noise=t["noise"][sl, :, :n])
        same = all(torch.equal(x[b, :, :n], y[0]) for x, y in zip(zs, zb))
        ez = max(rel_rms_err(y[0].cpu(), x[b, :, :n].cpu()) for x, y in zip(zs, zb))
        keep = max(0, n - 16) * U
        eo, same_o = 0.0, True
        if keep:
            eo = rel_rms_err(ob[0, :, :keep].cpu(), o[b, :, :keep].cpu())
            same_o = torch.equal(ob[0, :, :keep], o[b, :, :keep])
        print(f"{name} utterance {b} ({n} frames): z/z_p/z_hat bit-identical {same} (max {ez:.2e}), "
              f"audio bit-identical {same_o} (err {eo:.2e})")
        assert ez < BLOCK_TOL and eo < E2E_TOL


def test_error_paths():
    import wetts_b200
    from wetts_b200 import WettsError
    hps, sd, g, t = load_vc_case("vc_v1_ragged")
    n_vocab, n_spk = int(g["n_vocab"]), int(g["n_speakers"])
    args = (t["spec"], t["spec_lengths"], t["sid_src"], t["sid_tgt"])
    # a checkpoint without enc_q finalizes and infers; voice conversion names the first missing key
    plain = {k: v for k, v in sd.items() if not k.startswith("enc_q.")}
    net = wetts_b200.build_model(hps, n_vocab, n_spk, plain, "cuda")
    with pytest.raises(WettsError, match="enc_q.pre.weight"):
        net.voice_conversion(*args, noise=t["noise"])
    # an incomplete one also finalizes
    part = {k: v for k, v in sd.items() if k != "enc_q.enc.res_skip_layers.7.weight_v"}
    net = wetts_b200.build_model(hps, n_vocab, n_spk, part, "cuda")
    with pytest.raises(WettsError, match=r"enc_q\.enc\.res_skip_layers\.7\.weight_v"):
        net.voice_conversion(*args, noise=t["noise"])
    with pytest.raises(WettsError, match="enc_q"):
        net.spectrogram(t["audio"], t["audio_lengths"])
    # single-speaker model
    sd0 = {**synth.make_state_dict(hps.model, n_vocab, 0, seed=7), **synth.posterior_state_dict(hps.model, 513, 0, seed=8)}
    net0 = wetts_b200.build_model(hps, n_vocab, 0, sd0, "cuda")
    with pytest.raises(WettsError, match="n_speakers"):
        net0.voice_conversion(*args, noise=t["noise"])
    # too-short audio: the whole buffer, or one utterance of a batch
    net = wetts_b200.build_model(hps, n_vocab, n_spk, sd, "cuda")
    with pytest.raises(ValueError):
        net.spectrogram(torch.zeros(1, 384), torch.tensor([384]))
    with pytest.raises(WettsError, match="utterance 1"):
        net.spectrogram(torch.zeros(2, 4000), torch.tensor([4000, 384]))
    # wrong feature channel count
    with pytest.raises(ValueError, match="feature channels"):
        net.voice_conversion(t["spec"][:, :100], t["spec_lengths"], t["sid_src"], t["sid_tgt"])
    # the mel posterior encoder has no linear spectrogram
    hps_m, net_m, _ = _net("vc_vits2_vocos_mel")
    with pytest.raises(NotImplementedError):
        net_m.spectrogram(t["audio"], t["audio_lengths"])
