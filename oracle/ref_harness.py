"""Import and drive the REAL reference (`wetts/vits` of wenet-e2e/wetts, unmodified).

Test infrastructure (see oracle/vits_oracle.py header).  The tree is taken from `/root/reference`
where it exists (authoring container) and otherwise from `oracle/_ref/wetts_vits/`, the byte-identical
copy oracle/build_ref.py places there (git-ignored, travels to the GPU box).  Used by oracle/gen_golden.py
(fixture generation), by the not-gpu test that cross-checks the oracle against the live reference, and by
bench.py's CPU arm (`--impl reference`, `cpu_baseline`), where it is the thing TIMED as the baseline --
never part of the product path.
Recipe: SURVEY.md App. C (librosa stub before import; namespace-package imports).
"""
import contextlib
import io
import os
import sys
import types

import torch

REFERENCE_ROOT = "/root/reference"
# the byte-identical copy that oracle/build_ref.py places under oracle/_ref/ (git-ignored) when the build ran next to a
# wetts checkout, else that checkout itself
_CANDIDATES = (os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "wetts_vits"),
               os.path.join(REFERENCE_ROOT, "wetts", "vits"))
_VITS_DIR = next((d for d in _CANDIDATES if os.path.isfile(os.path.join(d, "model", "models.py"))), _CANDIDATES[0])


def available():
    return os.path.isfile(os.path.join(_VITS_DIR, "model", "models.py"))


def location():
    return _VITS_DIR


def _install_librosa_stub():
    if "librosa" in sys.modules:
        return
    lib = types.ModuleType("librosa")
    util = types.ModuleType("librosa.util")
    filt = types.ModuleType("librosa.filters")
    for name in ("pad_center", "tiny", "normalize"):
        setattr(util, name, lambda *a, **k: None)
    filt.mel = lambda *a, **k: None
    lib.util, lib.filters = util, filt
    sys.modules.update({"librosa": lib, "librosa.util": util, "librosa.filters": filt})


def import_reference():
    """Returns the reference's SynthesizerTrn class."""
    if not available():
        raise RuntimeError("reference tree not present (expected on the GPU box)")
    _install_librosa_stub()
    if _VITS_DIR not in sys.path:
        sys.path.insert(0, _VITS_DIR)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from model.models import SynthesizerTrn  # noqa: E402
    return SynthesizerTrn


def build_reference_model(hps, n_vocab, n_speakers, state_dict):
    """Construct as wetts/vits/inference.py:65-80 does and load `state_dict`
    (enc_q.* stays at its constructor init: never used by infer)."""
    import warnings
    SynthesizerTrn = import_reference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        net = SynthesizerTrn(n_vocab, hps.data.filter_length // 2 + 1,
                             hps.train.segment_size // hps.data.hop_length,
                             n_speakers=n_speakers, **hps.model).eval()
    missing, unexpected = net.load_state_dict(state_dict, strict=False)
    assert not unexpected, unexpected
    # never on the inference path: the posterior encoder, the iSTFT's window buffer (recomputed: hann), and the VITS2
    # coupling layers' post_transformer (constructed, commented out of forward; flows.py:160-162)
    def _unused(k):
        return k.startswith("enc_q.") or k.startswith("dec.istft.") or ".post_transformer." in k
    assert all(_unused(k) for k in missing), [k for k in missing if not _unused(k)]
    return net


@contextlib.contextmanager
def injected_noise(noise_w, noise_z):
    """Make the reference's implicit draws (duration_predictors.py:257 `torch.randn`,
    models.py:267 `torch.randn_like`) return the given tensors (SURVEY §0 finding 7)."""
    orig_randn, orig_like = torch.randn, torch.randn_like

    def fake_randn(*size, **kw):
        shape = tuple(size[0]) if len(size) == 1 and not isinstance(size[0], int) else tuple(size)
        assert noise_w is not None and shape == tuple(noise_w.shape), (shape, None if noise_w is None else noise_w.shape)
        return noise_w.clone()

    def fake_like(t, **kw):
        assert t.shape[0] == noise_z.shape[0] and t.shape[1] == noise_z.shape[1] and t.shape[2] <= noise_z.shape[2]
        return noise_z[:, :, : t.shape[2]].clone()

    torch.randn, torch.randn_like = fake_randn, fake_like
    try:
        yield
    finally:
        torch.randn, torch.randn_like = orig_randn, orig_like


def reference_infer(net, x, x_lengths, sid, noise_scale, length_scale, noise_scale_w, noise_w, noise_z):
    """Run the reference's infer() with injected noise; also recovers logw / w_ceil the way
    infer() computes them (models.py:243-255) for the staged parity of finding 8."""
    with torch.no_grad(), injected_noise(noise_w, noise_z), contextlib.redirect_stdout(io.StringIO()):
        o, attn, y_mask, (z, z_p, m_p, logs_p) = net.infer(
            x, x_lengths, sid=sid, noise_scale=noise_scale, length_scale=length_scale,
            noise_scale_w=noise_scale_w)
        g = net.emb_g(sid).unsqueeze(-1) if net.n_speakers > 0 else None
        h, m_tx, logs_tx, x_mask = net.enc_p(x, x_lengths, g=g)
        if net.use_sdp:
            logw = net.dp(h, x_mask, g=g, reverse=True, noise_scale=noise_scale_w)
        else:
            logw = net.dp(h, x_mask, g=g)
        w_ceil = torch.ceil(torch.exp(logw) * x_mask * length_scale)
    return dict(o=o, attn=attn, y_mask=y_mask, z=z, z_p=z_p, m_p=m_p, logs_p=logs_p, h=h,
                m_p_tx=m_tx, logs_p_tx=logs_tx, logw=logw, w_ceil=w_ceil)
