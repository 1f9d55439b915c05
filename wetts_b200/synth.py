"""Seeded synthetic checkpoints in the reference's on-disk format.

There is no pretrained checkpoint offline, so parity tests and the benchmark run on
random weights.  The tensors produced here use exactly the key names, shapes and
`weight_g`/`weight_v` weight-norm pairs of a reference `SynthesizerTrn.state_dict()`
(reference: wetts/vits/model/models.py:84-158; key patterns in SURVEY.md App. B) so the
same dict loads into the reference module (`load_state_dict`, used by
oracle/gen_golden.py) and into this package's loader.

Deliberate differences from the reference's default init (SURVEY.md §0 finding 5):
  * tensors the reference zero-fills (flow `post`, ConvFlow `proj`, ElementwiseAffine
    `m/logs`; flows.py:491-492, duration_predictors.py:87-88,130-131) are N(0, 0.02^2)
    — otherwise the flow is a pure permutation and parity would pass vacuously;
  * every `weight_g` is ||v|| * (1 + 0.3 N(0,1)) — the default g = ||v|| hides a wrong
    weight-norm axis (ConvTranspose1d normalises per *input* channel, decoders.py:41-48);
  * LayerNorm gamma/beta are perturbed by N(0, 0.1^2).
Generation is plain CPU torch with one seeded Generator, consumed in a fixed key order,
so it reproduces bit-for-bit on any box with the same torch build.
"""
import math

import torch


def _model_dict(hps_model):
    return hps_model.to_dict() if hasattr(hps_model, "to_dict") else dict(hps_model)


def state_dict_spec(hps_model, n_vocab, n_speakers):
    """Ordered list of (key, shape, kind) for the inference-path tensors.

    kind in {'emb', 'conv_w', 'conv_b', 'wn_v', 'wn_g', 'ln_g', 'ln_b', 'rel',
    'small', 'spk'}; `enc_q.*` (posterior encoder, never called by infer;
    models.py:124-132) is intentionally left out.
    """
    m = _model_dict(hps_model)
    H = m["hidden_channels"]
    inter = m["inter_channels"]
    F = m["filter_channels"]
    nh = m["n_heads"]
    nl = m["n_layers"]
    ks = m["kernel_size"]
    gin = m.get("gin_channels", 0)
    use_sdp = m.get("use_sdp", True)
    spec = []

    def conv(prefix, co, ci, k, bias=True, kind="conv_w"):
        spec.append((prefix + ".weight", (co, ci, k), kind))
        if bias:
            spec.append((prefix + ".bias", (co,), "conv_b"))

    def wn_conv(prefix, dim0, dim1, k, bias_len):
        spec.append((prefix + ".bias", (bias_len,), "conv_b"))
        spec.append((prefix + ".weight_g", (dim0, 1, 1), "wn_g"))
        spec.append((prefix + ".weight_v", (dim0, dim1, k), "wn_v"))

    def ln(prefix, c):
        spec.append((prefix + ".gamma", (c,), "ln_g"))
        spec.append((prefix + ".beta", (c,), "ln_b"))

    # text encoder (encoders.py:24-45, attentions.py:50-68,198-223,400-401)
    spec.append(("enc_p.emb.weight", (n_vocab, H), "emb"))
    dk = H // nh
    for i in range(nl):
        a = f"enc_p.encoder.attn_layers.{i}"
        spec.append((a + ".emb_rel_k", (1, 9, dk), "rel"))
        spec.append((a + ".emb_rel_v", (1, 9, dk), "rel"))
        for n in ("conv_q", "conv_k", "conv_v", "conv_o"):
            conv(f"{a}.{n}", H, H, 1)
        ln(f"enc_p.encoder.norm_layers_1.{i}", H)
        conv(f"enc_p.encoder.ffn_layers.{i}.conv_1", F, H, ks)
        conv(f"enc_p.encoder.ffn_layers.{i}.conv_2", H, F, ks)
        ln(f"enc_p.encoder.norm_layers_2.{i}", H)
    conv("enc_p.proj", 2 * inter, H, 1)

    vocos = m.get("vocoder_type", "hifigan") == "vocos"
    if vocos:
        # Vocos generator (decoders.py:250-282): in_conv, cond, norm_pre, ConvNeXt layers (:221-247), norm_post, out_conv
        vc, vh, vo = m.get("vocos_channels", 512), m.get("vocos_h_channels", 1536), m.get("vocos_out_channels", 1026)
        conv("dec.in_conv", vc, inter, 1)
        if gin:
            conv("dec.cond", vc, gin, 1)
        ln("dec.norm_pre", vc)
        for i in range(m.get("vocos_num_layers", 8)):
            p = f"dec.layers.{i}"
            conv(p + ".dw_conv", vc, 1, 3)
            ln(p + ".norm", vc)
            conv(p + ".pw_conv1", vh, vc, 1)
            conv(p + ".pw_conv2", vc, vh, 1)
            spec.append((p + ".scale", (1, vc, 1), "scale"))
        ln("dec.norm_post", vc)
        conv("dec.out_conv", vo, vc, 1, kind="out_small")
    # HiFi-GAN generator (decoders.py:28-61)
    c0 = m["upsample_initial_channel"]
    if not vocos:
        conv("dec.conv_pre", c0, inter, 7)
    ch = c0
    for i, (u, k) in enumerate(zip(m["upsample_rates"], m["upsample_kernel_sizes"])):
        if vocos:
            break
        cin, cout = c0 // (2 ** i), c0 // (2 ** (i + 1))
        wn_conv(f"dec.ups.{i}", cin, cout, k, cout)  # ConvTranspose1d: [C_in, C_out, k]
        ch = cout
    rb = 0
    for i in range(0 if vocos else len(m["upsample_rates"])):
        ch = c0 // (2 ** (i + 1))
        for k, dil in zip(m["resblock_kernel_sizes"], m["resblock_dilation_sizes"]):
            p = f"dec.resblocks.{rb}"
            if str(m["resblock"]) == "1":
                for j in range(len(dil)):
                    wn_conv(f"{p}.convs1.{j}", ch, ch, k, ch)
                for j in range(len(dil)):
                    wn_conv(f"{p}.convs2.{j}", ch, ch, k, ch)
            else:
                for j in range(len(dil)):
                    wn_conv(f"{p}.convs.{j}", ch, ch, k, ch)
            rb += 1
    if not vocos:
        conv("dec.conv_post", 1, ch, 7, bias=False)
        if gin:
            conv("dec.cond", c0, gin, 1)

    # flow: 4 residual coupling layers at even indices (flows.py:417-428, modules.py:33-58)
    half = inter // 2
    tflow = m.get("use_transformer_flows", False)
    if tflow and m.get("transformer_flow_type", "mono_layer_post_residual") != "pre_conv":
        raise NotImplementedError("only the 'pre_conv' transformer flow of the vits2_vocos_v1 recipe is supported")
    for f in (0, 2, 4, 6):
        p = f"flow.flows.{f}"
        if tflow:
            # ResidualCouplingTransformersLayer.pre_transformer (flows.py:112-120): Encoder(96, 96, heads 2, layers 2, k 3,
            # window_size=None -> no relative-position tables)
            for i in range(2):
                a = f"{p}.pre_transformer.attn_layers.{i}"
                for n in ("conv_q", "conv_k", "conv_v", "conv_o"):
                    conv(f"{a}.{n}", half, half, 1)
                ln(f"{p}.pre_transformer.norm_layers_1.{i}", half)
                conv(f"{p}.pre_transformer.ffn_layers.{i}.conv_1", half, half, 3)
                conv(f"{p}.pre_transformer.ffn_layers.{i}.conv_2", half, half, 3)
                ln(f"{p}.pre_transformer.norm_layers_2.{i}", half)
        conv(p + ".pre", H, half, 1)
        for i in range(4):
            wn_conv(f"{p}.enc.in_layers.{i}", 2 * H, H, 5, 2 * H)
        for i in range(4):
            rs = 2 * H if i < 3 else H
            wn_conv(f"{p}.enc.res_skip_layers.{i}", rs, H, 1, rs)
        if gin:
            wn_conv(p + ".enc.cond_layer", 2 * H * 4, gin, 1, 2 * H * 4)
        conv(p + ".post", half, H, 1, kind="small")
        spec[-1] = (p + ".post.bias", (half,), "small")

    # duration predictor
    def dds(prefix, c):
        for i in range(3):
            spec.append((f"{prefix}.convs_sep.{i}.weight", (c, 1, 3), "conv_w"))
            spec.append((f"{prefix}.convs_sep.{i}.bias", (c,), "conv_b"))
        for i in range(3):
            conv(f"{prefix}.convs_1x1.{i}", c, c, 1)
        for i in range(3):
            ln(f"{prefix}.norms_1.{i}", c)
        for i in range(3):
            ln(f"{prefix}.norms_2.{i}", c)

    if use_sdp:
        fc = H  # SDP overrides filter_channels = in_channels (duration_predictors.py:166)
        for grp in ("flows", "post_flows"):
            spec.append((f"dp.{grp}.0.m", (2, 1), "small"))
            spec.append((f"dp.{grp}.0.logs", (2, 1), "small"))
            for j in (1, 3, 5, 7):
                p = f"dp.{grp}.{j}"
                conv(p + ".pre", fc, 1, 1)
                dds(p + ".convs", fc)
                spec.append((p + ".proj.weight", (29, fc, 1), "small"))
                spec.append((p + ".proj.bias", (29,), "small"))
        conv("dp.post_pre", fc, 1, 1)
        conv("dp.post_proj", fc, fc, 1)
        dds("dp.post_convs", fc)
        conv("dp.pre", fc, H, 1)
        conv("dp.proj", fc, fc, 1)
        dds("dp.convs", fc)
        if gin:
            conv("dp.cond", fc, gin, 1)
    else:
        conv("dp.conv_1", 256, H, 3)
        ln("dp.norm_1", 256)
        conv("dp.conv_2", 256, 256, 3)
        ln("dp.norm_2", 256)
        conv("dp.proj", 1, 256, 1)
        if gin:
            conv("dp.cond", H, gin, 1)

    if n_speakers > 0:
        spec.append(("emb_g.weight", (n_speakers, gin), "spk"))
    return spec


def posterior_spec(hps_model, spec_channels):
    """Ordered (key, shape, kind) list of the posterior encoder `enc_q.*` (models.py:124-132, encoders.py:60-89):
    pre 1x1 conv from `spec_channels`, a 16-layer WN (kernel 5, dilation 1) with gin conditioning, proj to 2*inter."""
    m = _model_dict(hps_model)
    H, inter, gin = m["hidden_channels"], m["inter_channels"], m.get("gin_channels", 0)
    spec = [("enc_q.pre.weight", (H, spec_channels, 1), "conv_w"), ("enc_q.pre.bias", (H,), "conv_b")]

    def wn_conv(prefix, dim0, dim1, k):
        spec.extend([(prefix + ".bias", (dim0,), "conv_b"), (prefix + ".weight_g", (dim0, 1, 1), "wn_g"),
                     (prefix + ".weight_v", (dim0, dim1, k), "wn_v")])

    for i in range(16):
        wn_conv(f"enc_q.enc.in_layers.{i}", 2 * H, H, 5)
    for i in range(16):
        wn_conv(f"enc_q.enc.res_skip_layers.{i}", 2 * H if i < 15 else H, H, 1)
    if gin:
        wn_conv("enc_q.enc.cond_layer", 2 * H * 16, gin, 1)
    # proj: m and logs; kept small ("out_small") so that exp(logs) stays moderate on random weights
    spec.extend([("enc_q.proj.weight", (2 * inter, H, 1), "out_small"), ("enc_q.proj.bias", (2 * inter,), "conv_b")])
    return spec


def posterior_state_dict(hps_model, spec_channels, n_speakers, seed=4321):
    """Seeded synthetic `enc_q.*` tensors (fp32, CPU) to add to a make_state_dict() checkpoint for voice conversion.
    `n_speakers` only documents the intended checkpoint: the posterior encoder's shapes do not depend on it."""
    del n_speakers
    return _generate(posterior_spec(hps_model, spec_channels), seed)


def make_state_dict(hps_model, n_vocab, n_speakers, seed=1234):
    """Seeded synthetic `{"key": tensor}` dict (fp32, CPU)."""
    return _generate(state_dict_spec(hps_model, n_vocab, n_speakers), seed)


def _generate(spec, seed):
    gen = torch.Generator(device="cpu")
    gen.manual_seed(seed)
    sd = {}
    pending_v = {}

    def randn(shape):
        return torch.randn(shape, generator=gen, dtype=torch.float32)

    def uniform(shape, bound):
        return (torch.rand(shape, generator=gen, dtype=torch.float32) * 2 - 1) * bound

    for key, shape, kind in spec:
        if kind == "emb":
            t = randn(shape) * shape[1] ** -0.5
        elif kind == "rel":
            t = randn(shape) * shape[2] ** -0.5
        elif kind == "conv_w":
            fan_in = shape[1] * shape[2]
            t = uniform(shape, 1.0 / math.sqrt(fan_in))
        elif kind == "conv_b":
            t = uniform(shape, 0.05)
        elif kind == "wn_v":
            fan_in = shape[1] * shape[2]
            t = uniform(shape, 1.0 / math.sqrt(fan_in))
            g_key = key[: -len("weight_v")] + "weight_g"
            scale = pending_v.pop(g_key)
            sd[g_key] = t.reshape(shape[0], -1).norm(dim=1).reshape(shape[0], 1, 1) * scale
        elif kind == "wn_g":
            pending_v[key] = 1.0 + 0.3 * randn(shape)
            sd[key] = None  # keep insertion order: bias, weight_g, weight_v
            continue
        elif kind == "ln_g":
            t = 1.0 + 0.1 * randn(shape)
        elif kind == "ln_b":
            t = 0.1 * randn(shape)
        elif kind == "small":
            t = 0.02 * randn(shape)
        elif kind == "scale":        # ConvNeXt layer scale (decoders.py:235-237: 1 / num_layers), perturbed
            t = (1.0 / 8.0) * (1.0 + 0.3 * randn(shape))
        elif kind == "out_small":    # Vocos out_conv: log-magnitudes and phases; keep exp(mag) moderate
            fan_in = shape[1] * shape[2]
            t = uniform(shape, 0.5 / math.sqrt(fan_in))
        elif kind == "spk":
            t = randn(shape)
        else:
            raise ValueError(kind)
        sd[key] = t
    assert not pending_v
    return sd


def save_checkpoint(state_dict, path, iteration=0, learning_rate=2e-4):
    """Write the dict in the reference's checkpoint container
    (wetts/vits/utils/task.py:59-76): {"model", "iteration", "optimizer", "learning_rate"}."""
    torch.save({"model": state_dict, "iteration": iteration, "optimizer": {},
                "learning_rate": learning_rate}, path)


def fingerprint(state_dict):
    """Cheap order-independent digest used by the golden fixtures to prove the
    regenerated checkpoint is the one the fixtures were made with."""
    acc = 0.0
    for k in sorted(state_dict):
        t = state_dict[k].double()
        acc += float(t.abs().sum()) + 0.5 * float((t * t).sum())
    return acc
