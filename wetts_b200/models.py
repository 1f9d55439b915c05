"""Host-side mirror of the reference's VITS inference interface, running on libwetts_b200.

Same names, argument meaning and return structure as the reference
(wetts/vits/model/models.py:19-51,228-280,333-363 and the sub-module forwards listed in
SURVEY.md §8b), PyTorch tensors in / PyTorch tensors out, but every tensor operation is a
hand-written sm_100a kernel reached through the C ABI in include/wetts_b200.h.  PyTorch
is used only for device memory, streams and the default RNG.  There is no CPU path:
tensors must live on a CUDA device and the shared library must be built.

Additions over the reference signature (all keyword-only, default = reference behaviour):
`noise_w` [B,2,Tx] and `noise_z` [B,192,>=Ty] inject the standard-normal draws the
reference takes implicitly (duration_predictors.py:257, models.py:267), `durations`
[B,1,Tx] teacher-forces ceil(w) for staged parity (SURVEY.md §0 findings 7-8).
Likewise `voice_conversion(..., noise=)` / `enc_q(..., noise=)` take the posterior encoder's
randn_like draw [B,192,T] (encoders.py:98).
"""
import ctypes as C

import torch

from . import _lib
from ._lib import VitsConfig, WettsError, check


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _f32(t, device):
    return t.to(device=device, dtype=torch.float32).contiguous()


def _i64(t, device):
    return t.to(device=device, dtype=torch.int64).contiguous()


def _lengths_from_mask(mask):
    """[B,1,T] prefix mask -> int64[B] (the kernels take lengths, the reference API takes masks)."""
    return mask.reshape(mask.shape[0], -1).sum(dim=1).round().to(torch.int64).contiguous()


class _Engine:
    """Owns the C handle, the uploaded checkpoint and one grow-only device workspace PER STREAM
    (calls on different streams may overlap; each must have its own scratch, include/wetts_b200.h)."""

    def __init__(self, cfg: VitsConfig):
        self.cfg = cfg
        self.lib = _lib.load()
        self.handle = None
        self.device = None
        self.pending = {}
        self.finalized = False
        self._ws = {}

    # -- lifetime -----------------------------------------------------------
    def attach(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise WettsError("wetts_b200 runs on CUDA devices only (no CPU fallback)")
        if not torch.cuda.is_available():
            raise WettsError("no CUDA device visible: wetts_b200 has no CPU fallback")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        device = torch.device("cuda", idx)
        if self.handle is not None:
            if device == self.device:
                return
            self.close()
        h = C.c_void_p()
        check(self.lib.wetts_vits_create(C.byref(self.cfg), idx, C.byref(h)))
        self.handle, self.device, self.finalized = h, device, False
        if self.pending:
            self._upload()

    def close(self):
        if self.handle is not None:
            self.lib.wetts_vits_destroy(self.handle)
            self.handle = None
            self.finalized = False
            self._ws = {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_state(self, sd):
        self.pending = {k: v.detach().to(torch.float32).contiguous() for k, v in sd.items()
                        if torch.is_tensor(v) and v.is_floating_point()}
        if self.handle is not None:
            dev = self.device
            self.close()
            self.attach(dev)

    def _upload(self):
        for k, v in self.pending.items():
            dims = (C.c_int64 * max(v.dim(), 1))(*v.shape)
            check(self.lib.wetts_vits_set_tensor(self.handle, k.encode(), C.c_void_p(v.data_ptr()), dims, v.dim()))
        check(self.lib.wetts_vits_finalize(self.handle))
        self.finalized = True

    def ready(self):
        if self.handle is None:
            raise WettsError("model is not on a CUDA device: call .to('cuda') / .cuda() first")
        if not self.finalized:
            raise WettsError("no checkpoint loaded: call load_state_dict() / load_checkpoint() first")

    def workspace(self, nbytes, keep_prefix=0):
        """Scratch of the current stream, grown when needed; `keep_prefix` bytes of the old buffer are carried
        over (stage-1 results of infer() live in the prefix of the stage-2 workspace)."""
        key = torch.cuda.current_stream(self.device).cuda_stream
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            new = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            if ws is not None and keep_prefix:
                n = min(ws.numel(), int(keep_prefix))
                new[:n].copy_(ws[:n])
            self._ws[key] = ws = new
        return ws

    @property
    def upsample(self):
        if self.cfg.vocoder_type == 1:
            return int(self.cfg.vocos_hop_length)
        u = 1
        for i in range(self.cfg.n_upsamples):
            u *= self.cfg.upsample_rates[i]
        return u

    def launch_count(self):
        return int(self.lib.wetts_vits_launch_count(self.handle)) if self.handle else 0


class _Block:
    def __init__(self, engine):
        self._e = engine

    def __call__(self, *a, **k):
        return self.forward(*a, **k)


class SpeakerEmbedding(_Block):
    """emb_g (models.py:157-158): sid int64[B] -> [B, gin]."""

    def forward(self, sid):
        e = self._e
        e.ready()
        sid = _i64(sid, e.device)
        g = torch.empty(sid.shape[0], e.cfg.gin_channels, device=e.device, dtype=torch.float32)
        check(e.lib.wetts_speaker_embedding(e.handle, _ptr(sid), sid.shape[0], _ptr(g), _stream(e.device)))
        return g


class TextEncoder(_Block):
    """encoders.py:47-57: forward(x, x_lengths, g=None) -> (x, m, logs, x_mask)."""

    def forward(self, x, x_lengths, g=None):
        e = self._e
        e.ready()
        x, x_lengths = _i64(x, e.device), _i64(x_lengths, e.device)
        B, Tx = x.shape
        H, Cc = e.cfg.hidden_channels, e.cfg.inter_channels
        h = torch.empty(B, H, Tx, device=e.device, dtype=torch.float32)
        m = torch.empty(B, Cc, Tx, device=e.device, dtype=torch.float32)
        logs = torch.empty(B, Cc, Tx, device=e.device, dtype=torch.float32)
        nbytes = e.lib.wetts_text_encoder_workspace_bytes(e.handle, B, Tx)
        ws = e.workspace(nbytes)
        check(e.lib.wetts_text_encoder_forward(e.handle, _ptr(x), _ptr(x_lengths), B, Tx, _ptr(h), _ptr(m), _ptr(logs),
                                               _ptr(ws), ws.numel(), _stream(e.device)))
        x_mask = (torch.arange(Tx, device=e.device)[None, :] < x_lengths[:, None]).to(torch.float32)[:, None, :]
        return h, m, logs, x_mask


class DurationPredictorBlock(_Block):
    """DurationPredictor.forward(x, x_mask, g=None) (duration_predictors.py:297) or
    StochasticDurationPredictor.forward(x, x_mask, w=None, g=None, reverse=False, noise_scale=1.0)
    (:206-212) -- inference (reverse=True) only.  `noise`: optional explicit N(0,1) [B,2,Tx]."""

    def forward(self, x, x_mask, w=None, g=None, reverse=None, noise_scale=1.0, noise=None):
        e = self._e
        e.ready()
        if e.cfg.use_sdp and reverse is not True:
            raise NotImplementedError("the stochastic duration predictor's training branch (reverse=False) is out of scope")
        x = _f32(x, e.device)
        B, _, Tx = x.shape
        lengths = _lengths_from_mask(x_mask.to(e.device))
        gv = None if g is None else _f32(g.reshape(B, -1), e.device)
        if e.cfg.use_sdp:
            noise = torch.randn(B, 2, Tx, device=e.device) if noise is None else _f32(noise, e.device)
        else:
            noise = None
        logw = torch.empty(B, 1, Tx, device=e.device, dtype=torch.float32)
        nbytes = e.lib.wetts_duration_workspace_bytes(e.handle, B, Tx)
        ws = e.workspace(nbytes)
        check(e.lib.wetts_duration_forward(e.handle, _ptr(x), _ptr(lengths), _ptr(gv), _ptr(noise), float(noise_scale),
                                           B, Tx, _ptr(logw), _ptr(ws), ws.numel(), _stream(e.device)))
        return logw


class ResidualCouplingTransformersBlock(_Block):
    """flows.py:442-449: forward(x, x_mask, g=None, reverse=False) -> x.  reverse=True is the direction infer() takes,
    reverse=False the one voice_conversion() takes first (z -> z_p)."""

    def forward(self, x, x_mask, g=None, reverse=False):
        e = self._e
        e.ready()
        z = _f32(x, e.device).clone()
        B, _, Ty = z.shape
        lengths = _lengths_from_mask(x_mask.to(e.device))
        gv = None if g is None else _f32(g.reshape(B, -1), e.device)
        nbytes = e.lib.wetts_flow_workspace_bytes(e.handle, B, Ty)
        ws = e.workspace(nbytes)
        fn = e.lib.wetts_flow_reverse if reverse else e.lib.wetts_flow_forward
        check(fn(e.handle, _ptr(z), _ptr(lengths), _ptr(gv), B, Ty, _ptr(ws), ws.numel(), _stream(e.device)))
        return z


class PosteriorEncoder(_Block):
    """encoders.py:91-99: forward(x, x_lengths, g=None) -> (z, m, logs, x_mask).  x [B, spec_channels, T] features;
    `noise`: optional explicit N(0,1) [B,inter_channels,T] (the reference's randn_like)."""

    def forward(self, x, x_lengths, g=None, *, noise=None):
        e = self._e
        e.ready()
        x, x_lengths = _f32(x, e.device), _i64(x_lengths, e.device)
        B, S, T = x.shape
        Cc = e.cfg.inter_channels
        noise = torch.randn(B, Cc, T, device=e.device) if noise is None else _f32(noise, e.device)
        if tuple(noise.shape) != (B, Cc, T):
            raise ValueError(f"noise has shape {tuple(noise.shape)}, need {(B, Cc, T)}")
        gv = None if g is None else _f32(g.reshape(B, -1), e.device)
        z, m, logs = (torch.empty(B, Cc, T, device=e.device, dtype=torch.float32) for _ in range(3))
        nbytes = e.lib.wetts_posterior_workspace_bytes(e.handle, B, T)
        ws = e.workspace(nbytes)
        check(e.lib.wetts_posterior_encoder_forward(e.handle, _ptr(x), _ptr(x_lengths), _ptr(gv), _ptr(noise), B, T, _ptr(z),
                                                    _ptr(m), _ptr(logs), _ptr(ws), ws.numel(), _stream(e.device)))
        x_mask = (torch.arange(T, device=e.device)[None, :] < x_lengths[:, None]).to(torch.float32)[:, None, :]
        return z, m, logs, x_mask


class Generator(_Block):
    """decoders.py:63-82: forward(x, g=None) -> [B,1,T*prod(upsample_rates)]."""

    def forward(self, x, g=None):
        e = self._e
        e.ready()
        z = _f32(x, e.device)
        B, _, T = z.shape
        gv = None if g is None else _f32(g.reshape(B, -1), e.device)
        out = torch.empty(B, 1, T * e.upsample, device=e.device, dtype=torch.float32)
        nbytes = e.lib.wetts_generator_workspace_bytes(e.handle, B, T)
        ws = e.workspace(nbytes)
        check(e.lib.wetts_generator_forward(e.handle, _ptr(z), None, _ptr(gv), B, T, _ptr(out), _ptr(ws), ws.numel(),
                                            _stream(e.device)))
        return out


class SynthesizerTrn:
    """Drop-in for the inference side of the reference's `SynthesizerTrn`
    (wetts/vits/model/models.py:14-51); constructor arguments are identical so
    `SynthesizerTrn(len(phone_dict), posterior_channels, segment, n_speakers=N, **hps.model)`
    (inference.py:72-76) works unchanged; unknown keys are swallowed by **kwargs as there."""

    def __init__(self, n_vocab, spec_channels, segment_size, inter_channels, hidden_channels, filter_channels,
                 n_heads, n_layers, kernel_size, p_dropout, resblock, resblock_kernel_sizes, resblock_dilation_sizes,
                 upsample_rates, upsample_initial_channel, upsample_kernel_sizes, n_speakers=0, gin_channels=0,
                 use_sdp=True, vocoder_type="hifigan", vocos_channels=512, vocos_h_channels=1536, vocos_out_channels=1026,
                 vocos_num_layers=8, vocos_istft_config=None, **kwargs):
        if vocoder_type not in ("hifigan", "vocos"):
            raise NotImplementedError(f"vocoder_type {vocoder_type!r}: only 'hifigan' and 'vocos' exist in the reference")
        self.use_transformer_flows = bool(kwargs.get("use_transformer_flows", False))
        self.transformer_flow_type = kwargs.get("transformer_flow_type", "mono_layer_post_residual")
        if self.use_transformer_flows and self.transformer_flow_type != "pre_conv":
            raise NotImplementedError("of the VITS2 transformer flows only 'pre_conv' (the vits2_vocos_v1 recipe) is built "
                                      "(SURVEY.md §8f rank 4)")
        if kwargs.get("use_spk_conditioned_encoder", False):
            raise NotImplementedError("speaker-conditioned text encoder is not used by the v1/v2/v3 recipes")
        self.n_vocab, self.spec_channels, self.segment_size = n_vocab, spec_channels, segment_size
        self.inter_channels, self.hidden_channels, self.filter_channels = inter_channels, hidden_channels, filter_channels
        self.n_heads, self.n_layers, self.kernel_size, self.p_dropout = n_heads, n_layers, kernel_size, p_dropout
        self.resblock = str(resblock)
        self.resblock_kernel_sizes = list(resblock_kernel_sizes)
        self.resblock_dilation_sizes = [list(d) for d in resblock_dilation_sizes]
        self.upsample_rates, self.upsample_kernel_sizes = list(upsample_rates), list(upsample_kernel_sizes)
        self.upsample_initial_channel = upsample_initial_channel
        self.n_speakers, self.gin_channels, self.use_sdp = n_speakers, gin_channels, bool(use_sdp)
        self.use_mel_posterior_encoder = bool(kwargs.get("use_mel_posterior_encoder", False))

        c = VitsConfig()
        c.n_vocab, c.n_speakers = n_vocab, n_speakers
        c.inter_channels, c.hidden_channels, c.filter_channels = inter_channels, hidden_channels, filter_channels
        c.n_heads, c.n_layers, c.kernel_size = n_heads, n_layers, kernel_size
        c.gin_channels, c.use_sdp = gin_channels, int(bool(use_sdp))
        c.resblock_type = 1 if self.resblock == "1" else 2
        c.n_resblock_kernels = len(self.resblock_kernel_sizes)
        for j, (k, ds) in enumerate(zip(self.resblock_kernel_sizes, self.resblock_dilation_sizes)):
            c.resblock_kernel_sizes[j] = k
            c.resblock_n_dilations[j] = len(ds)
            for n, d in enumerate(ds):
                c.resblock_dilations[j][n] = d
        c.n_upsamples = len(self.upsample_rates)
        for i, (u, k) in enumerate(zip(self.upsample_rates, self.upsample_kernel_sizes)):
            c.upsample_rates[i], c.upsample_kernel_sizes[i] = u, k
        c.upsample_initial_channel = upsample_initial_channel
        self.vocoder_type = vocoder_type
        if vocoder_type == "vocos":
            ic = dict(vocos_istft_config or {"n_fft": 1024, "hop_length": 256, "win_length": 1024, "center": True})
            if hasattr(vocos_istft_config, "to_dict"):
                ic = vocos_istft_config.to_dict()
            if ic.get("win_length", ic["n_fft"]) != ic["n_fft"] or not ic.get("center", True):
                raise NotImplementedError("Vocos iSTFT: only win_length == n_fft with center=True (the reference recipe)")
            c.vocoder_type = 1
            c.vocos_channels, c.vocos_h_channels, c.vocos_out_channels = vocos_channels, vocos_h_channels, vocos_out_channels
            c.vocos_num_layers, c.vocos_n_fft, c.vocos_hop_length = vocos_num_layers, ic["n_fft"], ic["hop_length"]
        c.flow_type = 1 if self.use_transformer_flows else 0
        self._engine = _Engine(c)
        self.enc_p = TextEncoder(self._engine)
        self.dp = DurationPredictorBlock(self._engine)
        self.flow = ResidualCouplingTransformersBlock(self._engine)
        self.dec = Generator(self._engine)
        self.enc_q = PosteriorEncoder(self._engine)
        if n_speakers > 0:
            self.emb_g = SpeakerEmbedding(self._engine)
        self.training = False

    # -- nn.Module-like plumbing ---------------------------------------------
    def eval(self):
        self.training = False
        return self

    def to(self, device):
        self._engine.attach(device)
        return self

    def cuda(self, device=None):
        return self.to(torch.device("cuda", torch.cuda.current_device() if device is None else device))

    @property
    def device(self):
        return self._engine.device

    def load_state_dict(self, state_dict, strict=False):
        """Accepts the reference's state dict as saved by task.py:59-76 (weight_g/weight_v pairs)
        or with weight-norm already removed (export_onnx.py:79-81).  The posterior encoder (enc_q.*) is loaded
        when present; its input channels must equal spec_channels."""
        for k in ("enc_q.pre.weight", "enc_q.pre.weight_v"):
            w = state_dict.get(k)
            if torch.is_tensor(w) and w.dim() == 3 and w.shape[1] != self.spec_channels:
                raise ValueError(f"{k} takes {w.shape[1]} feature channels, the model was built with "
                                 f"spec_channels={self.spec_channels}")
        self._engine.set_state(state_dict)
        return self

    def launch_count(self):
        return self._engine.launch_count()

    def check_faults(self, synchronize=True):
        """Raises WettsError if a device-side pipeline wait timed out (soft watchdog, include/wetts_b200.h)."""
        e = self._engine
        e.ready()
        check(e.lib.wetts_vits_check_fault(e.handle, _stream(e.device), int(bool(synchronize))))
        return self

    def set_option(self, name, value):
        """Per-model engine option ("tensor_cores", "fused_resblock", "length_aware"); see include/wetts_b200.h."""
        e = self._engine
        e.ready()
        check(e.lib.wetts_vits_set_option(e.handle, name.encode(), int(value)))
        return self

    # -- inference ------------------------------------------------------------
    @torch.no_grad()
    def infer(self, x, x_lengths, sid=None, noise_scale=1, length_scale=1, noise_scale_w=1.0, max_len=None, *,
              noise_w=None, noise_z=None, durations=None, return_attn=True):
        """models.py:228-280.  Returns (o, attn, y_mask, (z, z_p, m_p, logs_p))."""
        e = self._engine
        e.ready()
        dev = e.device
        x, x_lengths = _i64(x, dev), _i64(x_lengths, dev)
        B, Tx = x.shape
        if self.n_speakers > 0:
            if sid is None:
                raise ValueError("sid is required when n_speakers > 0")
            sid = _i64(sid, dev)
        else:
            sid = None
        scales = (C.c_float * 3)(float(noise_scale), float(length_scale), float(noise_scale_w))
        if self.use_sdp:
            noise_w = torch.randn(B, 2, Tx, device=dev) if noise_w is None else _f32(noise_w, dev)
        else:
            noise_w = None
        dur = None if durations is None else _f32(durations.reshape(B, Tx), dev)
        y_lengths = torch.empty(B, dtype=torch.int64, device=dev)
        # stage 1 -- sized without knowing Ty
        nbytes1 = e.lib.wetts_vits_infer_workspace_bytes(e.handle, B, Tx, 1)
        ws = e.workspace(nbytes1)
        max_frames = C.c_int(0)
        st = _stream(dev)
        check(e.lib.wetts_vits_infer_durations(e.handle, _ptr(x), _ptr(x_lengths), _ptr(sid), scales, _ptr(noise_w),
                                               _ptr(dur), B, Tx, _ptr(y_lengths), None, None, C.byref(max_frames),
                                               _ptr(ws), ws.numel(), st))
        Ty = int(max_frames.value)
        # stage 2
        nbytes2 = e.lib.wetts_vits_infer_workspace_bytes(e.handle, B, Tx, Ty)
        if nbytes2 > ws.numel():
            ws = e.workspace(nbytes2, keep_prefix=nbytes1)   # grow, preserving the stage-1 results in the prefix
        Cc = self.inter_channels
        if noise_z is None:
            noise_z = torch.randn(B, Cc, Ty, device=dev)
        else:
            noise_z = _f32(noise_z, dev)
            if noise_z.shape[2] < Ty:
                raise ValueError(f"noise_z has {noise_z.shape[2]} frames, need {Ty}")
        U = e.upsample
        # models.py:270-271: the vocoder runs on (z * y_mask)[:, :, :max_len]; everything before it on all Ty frames
        Tg = Ty if max_len is None else max(1, min(Ty, int(max_len)))
        o = torch.empty(B, 1, Tg * U, device=dev, dtype=torch.float32)
        attn = torch.empty(B, 1, Ty, Tx, device=dev, dtype=torch.float32) if return_attn else None
        y_mask = torch.empty(B, 1, Ty, device=dev, dtype=torch.float32)
        z = torch.empty(B, Cc, Ty, device=dev, dtype=torch.float32)
        z_p, m_p, logs_p = torch.empty_like(z), torch.empty_like(z), torch.empty_like(z)
        check(e.lib.wetts_vits_infer_synthesize(e.handle, _ptr(x_lengths), _ptr(y_lengths), scales, _ptr(noise_z),
                                                noise_z.stride(0), noise_z.stride(1), B, Tx, Ty, Tg, _ptr(o), _ptr(attn),
                                                _ptr(y_mask), _ptr(z), _ptr(z_p), _ptr(m_p), _ptr(logs_p), _ptr(ws),
                                                ws.numel(), st))
        self.last_y_lengths = y_lengths
        return o, attn, y_mask, (z, z_p, m_p, logs_p)

    # -- voice conversion (models.py:369-376) ---------------------------------
    @torch.no_grad()
    def spectrogram(self, audio, audio_lengths):
        """spectrogram_torch (mel_processing.py:42-93, center=False) of each utterance on its own: audio [B,L] (or
        [B,1,L]) in [-1,1], audio_lengths int64[B] -> (spec [B,spec_channels,F], spec_lengths int64[B]) with
        F = 1 + (L + 2p - n_fft) // hop, n_fft = 2 (spec_channels - 1), hop = the upsample factor, p = (n_fft - hop) / 2.
        Frames beyond an utterance's own count are 0.  Synchronises the current stream."""
        if self.use_mel_posterior_encoder:
            raise NotImplementedError("the mel posterior encoder takes mel features: pass them to voice_conversion()")
        e = self._engine
        e.ready()
        audio = _f32(audio, e.device)
        audio = audio.reshape(audio.shape[0], -1)
        lengths = _i64(audio_lengths, e.device)
        B, L = audio.shape
        n_fft, hop = 2 * (self.spec_channels - 1), e.upsample
        pad = (n_fft - hop) // 2
        if L <= pad:
            raise ValueError(f"audio of {L} samples is shorter than the {pad} + 1 the reflection padding needs")
        F = 1 + (L + 2 * pad - n_fft) // hop
        spec = torch.empty(B, self.spec_channels, F, device=e.device, dtype=torch.float32)
        spec_lengths = torch.empty(B, device=e.device, dtype=torch.int64)
        nbytes = e.lib.wetts_spectrogram_workspace_bytes(e.handle, B, L)
        ws = e.workspace(max(int(nbytes), 1))
        check(e.lib.wetts_spectrogram(e.handle, _ptr(audio), _ptr(lengths), B, L, _ptr(spec), _ptr(spec_lengths), _ptr(ws),
                                      ws.numel(), _stream(e.device)))
        return spec, spec_lengths

    @torch.no_grad()
    def voice_conversion(self, y, y_lengths, sid_src, sid_tgt, *, noise=None):
        """models.py:369-376: y [B, spec_channels, T] features (linear spectrogram, see spectrogram(), or mel features for
        the mel posterior encoder), y_lengths int64[B] -> (o_hat [B,1,T*U], y_mask [B,1,T], (z, z_p, z_hat)).
        `noise`: optional explicit N(0,1) [B,inter_channels,T], the posterior encoder's randn_like draw."""
        e = self._engine
        e.ready()
        dev = e.device
        y, y_lengths = _f32(y, dev), _i64(y_lengths, dev)
        B, S, T = y.shape
        if S != self.spec_channels:
            raise ValueError(f"y has {S} feature channels, the posterior encoder takes {self.spec_channels}")
        if self.n_speakers <= 0:
            raise WettsError("voice conversion needs a multi-speaker model (n_speakers == 0)")
        sid_src, sid_tgt = _i64(sid_src, dev), _i64(sid_tgt, dev)
        Cc = self.inter_channels
        noise = torch.randn(B, Cc, T, device=dev) if noise is None else _f32(noise, dev)
        if tuple(noise.shape) != (B, Cc, T):
            raise ValueError(f"noise has shape {tuple(noise.shape)}, need {(B, Cc, T)}")
        o = torch.empty(B, 1, T * e.upsample, device=dev, dtype=torch.float32)
        y_mask = torch.empty(B, 1, T, device=dev, dtype=torch.float32)
        z, z_p, z_hat = (torch.empty(B, Cc, T, device=dev, dtype=torch.float32) for _ in range(3))
        nbytes = e.lib.wetts_vits_voice_conversion_workspace_bytes(e.handle, B, T)
        ws = e.workspace(nbytes)
        check(e.lib.wetts_vits_voice_conversion(e.handle, _ptr(y), _ptr(y_lengths), _ptr(sid_src), _ptr(sid_tgt), _ptr(noise),
                                                B, T, _ptr(o), _ptr(y_mask), _ptr(z), _ptr(z_p), _ptr(z_hat), _ptr(ws),
                                                ws.numel(), _stream(dev)))
        return o, y_mask, (z, z_p, z_hat)

    # -- ONNX-export-shaped entry points (models.py:333-363) ------------------
    def export_forward(self, x, x_lengths, scales, sid):
        s = scales[0]
        return self.infer(x, x_lengths, sid, noise_scale=float(s[0]), length_scale=float(s[1]),
                          noise_scale_w=float(s[2]), return_attn=False)[0]

    def export_encoder_forward(self, x, x_lengths, scales, sid):
        s = scales[0]
        _, _, y_mask, (z, _, _, _) = self.infer(x, x_lengths, sid, noise_scale=float(s[0]), length_scale=float(s[1]),
                                                noise_scale_w=float(s[2]), return_attn=False)
        return (z * y_mask).transpose(1, 2).contiguous()

    @torch.no_grad()
    def export_decoder_forward(self, z, sid):
        """z f32[B,L,192] (time-major, export_onnx.py:127-148) -> audio [B,1,L*U]."""
        e = self._engine
        e.ready()
        z = _f32(z, e.device)
        B, L, _ = z.shape
        sid = _i64(sid, e.device) if self.n_speakers > 0 else None
        out = torch.empty(B, 1, L * e.upsample, device=e.device, dtype=torch.float32)
        nbytes = e.lib.wetts_vits_decoder_workspace_bytes(e.handle, B, L)
        ws = e.workspace(nbytes)
        check(e.lib.wetts_vits_forward_decoder(e.handle, _ptr(z), _ptr(sid), B, L, _ptr(out), _ptr(ws), ws.numel(),
                                               _stream(e.device)))
        return out
