#!/usr/bin/env python
"""Benchmark of the VITS inference hot path (BASELINE.json metric: audio-seconds/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One JSON line on rank 0's stdout (contract in the task statement; DESIGN.md "Measurement").

A step = one pass of the hot path over one batch of synthetic utterances.  Workloads = BASELINE.json configs:
    multilingual_v3_b256x128   configs[2], the configuration the metric is quoted on (default): full infer, 256 x 128 phonemes
    baker_v1_cli_b1            configs[0]: Baker v1, batch 1, the CLI utterance (latency; L2 flushed between steps)
    baker_v1_gen_b64x640       configs[1]: HiFi-GAN V1 Generator only, z f32[64,192,640]   (baker_v3_gen_b64x640: the v3 generator)
    multilingual_v3_b1024x128  configs[3]: 1024 utterances held by rank 0, dealt to the ranks over NCCL (strong scaling)
    aishell3_v1_b32x512        configs[4]: per-GPU share (32 of 128 utterances) of the 512-phoneme AISHELL-3 v1 workload
Multi-GPU (N > 1): one process per GPU.  `--dist sharded` (default): rank 0 holds the request batch (N x the per-GPU batch for
the weak-scaling workloads, the fixed total for the strong-scaling one), ids are scattered and waveforms gathered back to
rank 0 over NCCL INSIDE the timed region (the "trivial batch scatter/gather" of the north_star; wetts_b200/dist.py).
`--dist replicas`: independent per-rank batches, no data-path collective (round-1 behaviour).

`--impl reference` times the reference's own CPU implementation of the path on the host cores: the unmodified
`SynthesizerTrn.infer` from oracle/_ref (placed by oracle/build_ref.py; kind "reference") when present, else the oracle
port (kind "port"), on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step returned (waveforms, and the valid frame counts where the step
returns them) to DIR/<name>.npy, at most 64 MB in all, so that two builds can be compared output for output: the inputs
are seeded, so the same arguments give the same inputs on every run.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on fd 1 even with
# NCCL_DEBUG_FILE set -- seen on the 2-GPU box), so fd 1 is pointed at stderr for the whole run and the JSON line goes to
# a private duplicate of the original stdout.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
sys.stdout.flush()
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

CLI_TOKENS = "sil j in1 #0 t ian1 #0 t ian1 #0 q i4 #0 z en3 #0 m e5 #0 ^ iang4 #4".split()   # SURVEY.md 8(d) config 1
CLI_VOCAB = ["sil"] + sorted(set(CLI_TOKENS) - {"sil"})

# kind: "infer" = full SynthesizerTrn.infer; "generator" = Generator.forward only (decoders.py:63)
# cpu_utts = bounded sample of the CPU arm (utterances per step)
WORKLOADS = {
    "multilingual_v3_b256x128": dict(config="multilingual_v3", n_vocab=256, n_spk=2, batch=256, phonemes=128,
                                     length_scale=2.8, kind="infer", cpu_utts=48, baseline_config=2),
    "baker_v1_cli_b1": dict(config="baker_v1", n_vocab=len(CLI_VOCAB), n_spk=1, batch=1, phonemes=len(CLI_TOKENS),
                            length_scale=1.0, kind="infer", cpu_utts=1, baseline_config=0, cli=True, flush_l2=True),
    "baker_v1_gen_b64x640": dict(config="baker_v1", n_vocab=256, n_spk=1, batch=64, frames=640, kind="generator",
                                 cpu_utts=2, baseline_config=1),
    "baker_v3_gen_b64x640": dict(config="baker_v3", n_vocab=256, n_spk=1, batch=64, frames=640, kind="generator",
                                 cpu_utts=16, baseline_config=1),
    "multilingual_v3_b1024x128": dict(config="multilingual_v3", n_vocab=256, n_spk=2, batch=256, total=1024, phonemes=128,
                                      length_scale=2.8, kind="infer", cpu_utts=48, baseline_config=3, strong=True),
    "aishell3_v1_b32x512": dict(config="aishell3_v1", n_vocab=256, n_spk=218, batch=32, phonemes=512,
                                length_scale=3.0, kind="infer", cpu_utts=1, baseline_config=4),
    "baker_v1_b64x128": dict(config="baker_v1", n_vocab=256, n_spk=1, batch=64, phonemes=128, length_scale=3.4,
                             kind="infer", cpu_utts=4, baseline_config=1),
    "multilingual_v3_b8x32": dict(config="multilingual_v3", n_vocab=256, n_spk=2, batch=8, phonemes=32,
                                  length_scale=2.8, kind="infer", cpu_utts=8, baseline_config=2, flush_l2=True),
}
DEFAULT_WORKLOAD = "multilingual_v3_b256x128"
NOISE_SCALE, NOISE_SCALE_W = 0.667, 0.8   # every reference caller (inference.py:98, cli/model.py:45)

# per-frame work of the HiFi-GAN generator (SURVEY.md §8d / BASELINE.md §4); v1 = HiFi-GAN V1, v3 = the v3 recipe
GEN_FLOP_PER_FRAME = {"v1": 614.9e6, "v3": 45.36e6}
GEN_LAYER_BYTES_PER_FRAME = {"v1": 4.05e6, "v3": 0.749e6}
GEN_COMPULSORY_BYTES_PER_FRAME = 192 * 4 + 256 * 4


def gen_family(cfg_name):
    return "v1" if cfg_name.endswith("_v1") else "v3"


def make_batch(wl, B, seed):
    gen = torch.Generator().manual_seed(seed)
    if wl.get("cli"):
        x = torch.tensor([[CLI_VOCAB.index(t) for t in CLI_TOKENS]] * B, dtype=torch.long)
    else:
        x = torch.randint(0, wl["n_vocab"], (B, wl["phonemes"]), generator=gen)
    lens = torch.full((B,), x.shape[1], dtype=torch.long)
    sid = torch.randint(0, wl["n_spk"], (B,), generator=gen)
    return x, lens, sid


DUMP_BYTES = 64_000_000


def dump_outputs(arrays, out_dir):
    """Writes `arrays` (name -> tensor) as out_dir/<name>.npy: floating point as float32 (float64 stays float64),
    integers as float64 (exact).  Arrays up to 1 MiB are written whole; when the larger ones exceed the rest of
    DUMP_BYTES together, each keeps a share of rows (first dimension, one utterance each) proportional to its size: a
    sorted sample drawn with a fixed seed, so it depends on the shapes only, and the indices of the kept rows go to
    out_dir/<name>_rows.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.detach().cpu() for k, v in arrays.items()}
    host = {k: v.double() if not v.is_floating_point() or v.dtype == torch.float64 else v.float() for k, v in host.items()}
    size = {k: v.numel() * v.element_size() for k, v in host.items()}
    large = {k for k, n in size.items() if n > 1 << 20}
    total = sum(size[k] for k in large)
    budget = DUMP_BYTES - sum(n for k, n in size.items() if k not in large) - 4096 * 2 * len(host)   # .npy headers
    for name, v in host.items():
        nbytes = size[name]
        if name in large and total > budget and v.shape[0] > 1:
            row_bytes = nbytes // v.shape[0] + 8                # + its index in <name>_rows.npy
            keep = max(1, min(v.shape[0], int(budget * nbytes / total) // row_bytes))
            if keep < v.shape[0]:
                rows = torch.randperm(v.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
                np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.double().numpy())
                v = v[rows]
        np.save(os.path.join(out_dir, f"{name}.npy"), v.contiguous().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons, cap = [], None, [], set(), 0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                pw.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
                    cap += n == "sw_power_cap"
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "sw_power_cap_samples": cap, "power_w_max": max(pw) if pw else None}


def peaks():
    """(hbm GB/s, bf16/f16 dense TFLOP/s sustained, burst, source)"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return (d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1500.0)),
                d.get("bf16_tflops", 1700.0), "measured (MEASURED_PEAKS.json)")
    return 6650.0, 1500.0, 1700.0, "fallback (B200_PROFILING.md)"


def measured_traffic(workload):
    """DRAM bytes per generator call from the committed ncu capture (profiles/generator_traffic.json), or None."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "generator_traffic.json")))
        e = d.get(workload) or (d if d.get("workload") == workload else None)
        if e:
            return float(e["generator_dram_bytes_per_step"]), e.get("source")
    except Exception:
        pass
    return None, None


# ------------------------------------------------------------------------------------------------ CPU arm
def _cpu_threads():
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    return n


class CpuArm:
    """The reference's CPU implementation of the path: the unmodified module from oracle/_ref when present
    (kind "reference"), else the oracle port (kind "port").  Test/benchmark infrastructure only."""

    def __init__(self, workload):
        from wetts_b200 import synth
        from wetts_b200.hparams import builtin_config
        self.wl = WORKLOADS[workload]
        self.hps = builtin_config(self.wl["config"])
        self.sd = synth.make_state_dict(self.hps.model, self.wl["n_vocab"], self.wl["n_spk"], seed=self.hps.train.seed)
        self.kind, self.net, self.w = "port", None, None
        try:
            from oracle import ref_harness
            if ref_harness.available():
                with contextlib.redirect_stdout(io.StringIO()):
                    self.net = ref_harness.build_reference_model(self.hps, self.wl["n_vocab"], self.wl["n_spk"], self.sd)
                self.kind = "reference"
        except Exception as e:   # missing optional dependency of the reference tree -> the port
            print(f"[bench] reference module unavailable ({e!r}); CPU arm falls back to the oracle port", file=sys.stderr)
            self.net = None
        if self.net is None:
            from oracle import vits_oracle as O
            self.O = O
            self.w = O.fold_weight_norm(self.sd)

    def inputs(self, n_utts, device="cpu"):
        wl = self.wl
        if wl["kind"] == "generator":
            gen = torch.Generator().manual_seed(5678)
            z = torch.randn(wl["batch"], self.hps.model.inter_channels, wl["frames"], generator=gen)[:n_utts]
            sid = torch.zeros(n_utts, dtype=torch.long)
            return z.to(device), sid.to(device)
        x, lens, sid = make_batch(wl, max(n_utts, 1) if wl.get("cli") else wl["batch"], 5678)
        return x[:n_utts].to(device), lens[:n_utts].to(device), sid[:n_utts].to(device)

    def run(self, n_utts, device="cpu"):
        """One pass over `n_utts` utterances.  Returns (audio seconds, wall seconds, y_lengths or None)."""
        wl, hps = self.wl, self.hps
        hop, sr = hps.data.hop_length, hps.data.sampling_rate
        on_gpu = str(device).startswith("cuda")
        sync = (lambda: torch.cuda.synchronize()) if on_gpu else (lambda: None)
        inputs = self.inputs(n_utts, device)          # seeded on the CPU, then moved
        # the oracle port creates its index tensors with the default device; the reference module follows its inputs
        dev_ctx = torch.device(device) if (on_gpu and self.net is None) else contextlib.nullcontext()
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()), dev_ctx:   # the reference prints per-block timings
            if wl["kind"] == "generator":
                z, sid = inputs
                sync()
                t0 = time.perf_counter()
                if self.net is not None:
                    g = self.net.emb_g(sid).unsqueeze(-1) if wl["n_spk"] > 0 else None
                    self.net.dec(z, g=g)
                else:
                    g = self.w["emb_g.weight"][sid][:, :, None] if wl["n_spk"] > 0 else None
                    self.O.generator(self.w, hps.model, z, g)
                sync()
                dt = time.perf_counter() - t0
                return n_utts * wl["frames"] * hop / sr, dt, None
            x, lens, sid = inputs
            sync()
            t0 = time.perf_counter()
            if self.net is not None:
                o, _, y_mask, _ = self.net.infer(x, lens, sid=sid if wl["n_spk"] > 0 else None, noise_scale=NOISE_SCALE,
                                                 length_scale=wl["length_scale"], noise_scale_w=NOISE_SCALE_W)
                ylen = y_mask.sum(dim=[1, 2]).long()
            else:
                r = self.O.infer(self.w, hps.model, x, lens, sid, NOISE_SCALE, wl["length_scale"], NOISE_SCALE_W, folded=True)
                ylen = r["y_lengths"]
            sync()
            dt = time.perf_counter() - t0
        return float(ylen.sum()) * hop / sr, dt, ylen.cpu()

    def to(self, device):
        if self.net is not None:
            self.net = self.net.to(device)
        else:
            self.w = {k: v.to(device) for k, v in self.w.items()}
        return self

    def pick_threads(self):
        """oneDNN convs on tiny channel counts degrade when oversubscribed: try a few thread counts on one
        utterance and keep the fastest (reported as `cores`).  Remembers the per-utterance time of the winner."""
        n = _cpu_threads()
        best, best_t = None, float("inf")
        for c in sorted({c for c in (8, 16, 32, 64, n) if c <= n}):
            torch.set_num_threads(c)
            _, dt, _ = self.run(1)
            if dt < best_t:
                best, best_t = c, dt
        torch.set_num_threads(best)
        self.seconds_per_utterance = best_t
        return best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    arm = CpuArm(args.workload)
    threads = arm.pick_threads()
    # bounded sample: the whole --steps K run should end within a few minutes (target ~150 s of CPU work)
    n_utts = max(1, min(wl["cpu_utts"], int(150.0 / (max(args.steps, 1) * max(arm.seconds_per_utterance, 1e-3)))))
    for _ in range(1 if args.warmup else 0):
        arm.run(min(2, n_utts))
    tot_audio, tot_t = 0.0, 0.0
    for _ in range(args.steps):
        a, t, _ = arm.run(n_utts)
        tot_audio += a
        tot_t += t
    v = tot_audio / tot_t
    what = "Generator.forward" if wl["kind"] == "generator" else "SynthesizerTrn.infer"
    src = "unmodified reference module (oracle/_ref)" if arm.kind == "reference" else "oracle port"
    sample = f"{n_utts} of the workload's {wl.get('total', wl['batch'])} utterances per step, {what}, {src}"
    line = {
        "impl": "reference", "metric": "audio-seconds/sec (VITS infer)", "value": v, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps,
        "higher_is_better": True, "scaling": "strong" if wl.get("strong") else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": args.workload, "config": wl["config"], "phonemes": wl.get("phonemes"),
                   "frames": wl.get("frames"), "sample": sample, "same_config": False,
                   "note": "metric is normalised per audio-second, so the bounded sample is comparable"},
        "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": threads, "kind": arm.kind, "sample": sample},
        "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import wetts_b200
    from wetts_b200 import _lib, synth
    from wetts_b200 import dist as wdist
    from wetts_b200.hparams import builtin_config

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (wetts_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    wl = dict(WORKLOADS[args.workload])
    if args.batch:
        wl["batch"] = args.batch
    cfg_name, kind = wl["config"], wl["kind"]
    strong = bool(wl.get("strong"))
    sharded = world > 1 and args.dist == "sharded" and kind == "infer"
    lib = _lib.load()
    _lib.check(lib.wetts_set_option(b"tensor_cores", int(args.tensor_cores)))
    _lib.check(lib.wetts_set_option(b"fused_resblock", int(args.fused_resblock)))
    if args.tensor_format:
        _lib.check(lib.wetts_set_option(b"tensor_format", int(args.tensor_format)))
    if args.attention_tc >= 0:
        _lib.check(lib.wetts_set_option(b"attention_tensor_cores", int(args.attention_tc)))
    hps = builtin_config(cfg_name)
    sd = synth.make_state_dict(hps.model, wl["n_vocab"], wl["n_spk"], seed=hps.train.seed)
    net = wetts_b200.build_model(hps, wl["n_vocab"], wl["n_spk"], sd, dev)
    if args.length_aware:
        net.set_option("length_aware", 1)
    hop, sr = hps.data.hop_length, hps.data.sampling_rate
    Cc = hps.model.inter_channels
    ls = wl.get("length_scale", 1.0)
    fam = gen_family(cfg_name)

    # ---- the batch of this rank (replicas / N = 1) or of the job (sharded: held by rank 0)
    if strong:
        B_job = wl["total"]
        B = B_job // world if sharded or world == 1 else wl["batch"]
    else:
        B = wl["batch"]
        B_job = B * world
    # one GPU takes the strong-scaling job in chunks of the per-GPU batch (activations of 1024 utterances do not fit)
    chunk = wl["batch"] if strong and world == 1 else None

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    gen = torch.Generator(device=dev).manual_seed(4321 + rank)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if wl.get("flush_l2") else None

    # ---- end-to-end leg, device -> host: the waveform of step i is copied to pinned host memory on a side stream while
    # step i + 1 computes (what a serving loop does); at most one copy in flight, two host buffers, and the LAST copy is
    # waited for inside the timed region (timed(..., drain=)), so every step's D2H is inside it.  The latency workload
    # (L2 flushed between steps, per-step events) keeps the serial form: copy, then synchronize.
    pipelined = flush_buf is None
    copy_stream = torch.cuda.Stream(device=dev) if pipelined else None
    d2h_state = {"bufs": [None, None], "i": 0, "pending": None}

    def d2h_submit(outs):
        n = sum(o_.numel() for o_ in outs)
        k = d2h_state["i"] & 1
        d2h_state["i"] += 1
        if n and (d2h_state["bufs"][k] is None or d2h_state["bufs"][k].numel() < n):
            d2h_state["bufs"][k] = torch.empty(int(n * 1.25) + 4096, dtype=torch.float32).pin_memory()   # flat: contiguous D2H
        buf = d2h_state["bufs"][k]
        if not pipelined:
            off = 0
            for o_ in outs:
                buf[off:off + o_.numel()].copy_(o_.reshape(-1), non_blocking=True)
                off += o_.numel()
            torch.cuda.current_stream().synchronize()
            return n * 4
        computed = torch.cuda.Event()
        computed.record()
        if d2h_state["pending"] is not None:
            d2h_state["pending"].synchronize()          # the previous step's copy (finished long ago: bounds host buffers to two)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(computed)
            off = 0
            for o_ in outs:
                buf[off:off + o_.numel()].copy_(o_.reshape(-1), non_blocking=True)
                o_.record_stream(copy_stream)
                off += o_.numel()
            done = torch.cuda.Event()
            done.record(copy_stream)
        d2h_state["pending"] = done
        return n * 4

    def d2h_drain():
        if d2h_state["pending"] is not None:
            torch.cuda.current_stream().wait_event(d2h_state["pending"])   # the end-of-region event is recorded after this
            d2h_state["pending"].synchronize()
            d2h_state["pending"] = None

    if kind == "generator":
        T = wl["frames"]
        zc = torch.randn(B, Cc, T, generator=torch.Generator().manual_seed(5678 + rank))
        z_host = zc.pin_memory()
        z_dev = zc.to(dev)
        sid_dev = torch.zeros(B, dtype=torch.long, device=dev)
        g_dev = net.emb_g(sid_dev)[:, :, None] if wl["n_spk"] > 0 else None
        frames_rank, Ty = B * T, T
        U = 1
        for u in hps.model.upsample_rates:
            U *= u
        h2d, d2h = z_host.numel() * 4, B * T * U * 4

        def step_resident():
            return net.dec(z_dev, g=g_dev)

        def step_e2e():
            zz = z_host.to(dev, non_blocking=True)
            o_ = net.dec(zz, g=g_dev)
            d2h_submit([o_])
    else:
        seed_rank = 5678 if sharded or strong else 5678 + rank
        n_make = B_job if (sharded or strong) else B
        x, lens, sid = make_batch(wl, n_make, seed_rank)
        have_batch = (not sharded) or rank == 0
        xh, lh, sh = (x.pin_memory(), lens.pin_memory(), sid.pin_memory()) if have_batch else (None, None, None)
        xd, ld, sdv = (x.to(dev), lens.to(dev), sid.to(dev)) if have_batch else (None, None, None)
        h2d = int(x.numel() + lens.numel() + sid.numel()) * 8 if have_batch else 0
        state = {"frames": 0, "Ty": 0, "d2h": 0}

        def infer_local(a, b_, c, **kw):
            """our public API on this rank's resident tensors; the strong-scaling job on one GPU runs in chunks"""
            if chunk is None or a.shape[0] <= chunk:
                o_, _, ym, _ = net.infer(a, b_, c, NOISE_SCALE, ls, NOISE_SCALE_W, return_attn=False, **kw)
                state["frames"], state["Ty"] = int(net.last_y_lengths.sum()), ym.shape[2]
                return [o_]
            outs, fr = [], 0
            for i in range(0, a.shape[0], chunk):
                o_, _, ym, _ = net.infer(a[i:i + chunk], b_[i:i + chunk], c[i:i + chunk], NOISE_SCALE, ls, NOISE_SCALE_W,
                                         return_attn=False)
                fr += int(net.last_y_lengths.sum())
                state["Ty"] = max(state["Ty"], ym.shape[2])
                outs.append(o_)
            state["frames"] = fr
            return outs

        noise_w = noise_z = None
        if not sharded and chunk is None:
            # probe once to size the injected noise (resident step = deterministic: same Ty every step)
            noise_w = torch.randn(B, 2, x.shape[1], device=dev, generator=gen) if net.use_sdp else None
            infer_local(xd, ld, sdv, noise_w=noise_w)
            noise_z = torch.randn(B, Cc, state["Ty"], device=dev, generator=gen)

        def step_resident():
            if sharded:
                r = wdist.sharded_infer(net, xd, ld, sdv, dev, hop_upsample=256, as_list=False, noise_scale=NOISE_SCALE,
                                        length_scale=ls, noise_scale_w=NOISE_SCALE_W, return_attn=False)
                yl = net.last_y_lengths
                state["frames_local"], state["Ty"] = int(yl.sum()), int(yl.max())
                return r
            if chunk is None:
                return infer_local(xd, ld, sdv, noise_w=noise_w, noise_z=noise_z)
            return infer_local(xd, ld, sdv)

        def step_e2e():
            if sharded:
                a = xh.to(dev, non_blocking=True) if rank == 0 else None
                b_ = lh.to(dev, non_blocking=True) if rank == 0 else None
                c = sh.to(dev, non_blocking=True) if rank == 0 else None
                r = wdist.sharded_infer(net, a, b_, c, dev, hop_upsample=256, as_list=False, noise_scale=NOISE_SCALE,
                                        length_scale=ls, noise_scale_w=NOISE_SCALE_W, return_attn=False)
                outs = [r[0]] if rank == 0 else []
            else:
                a, b_, c = xh.to(dev, non_blocking=True), lh.to(dev, non_blocking=True), sh.to(dev, non_blocking=True)
                outs = infer_local(a, b_, c)                   # noise drawn on the device, as the reference does
            state["d2h"] = d2h_submit(outs)

    def timed(fn, steps, drain=None):
        """EXACTLY `steps` steps between barrier + synchronize; device time from CUDA events on the launch stream
        (per step, so an L2 flush between steps stays outside); `drain` (pipelined copies) runs before the closing event,
        which is recorded after the launch stream has waited for the last copy; returns (max over ranks, this rank's) ms
        and what the last step returned."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        ev_end = torch.cuda.Event(enable_timing=True)
        barrier()
        for i in range(steps):
            if flush_buf is not None:
                flush_buf.fill_(i & 0xFF)
            ev[i][0].record()
            out = fn()
            ev[i][1].record()
            if i + 1 < steps:
                out = None      # released before the next step, as if never held: its memory is reused there
        if drain is not None:
            drain()
        ev_end.record()
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in ev) if flush_buf is not None else ev[0][0].elapsed_time(ev_end)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), ms, out

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local)
    launches0 = net.launch_count()
    sampler.start()
    if args.profile_range:
        torch.cuda.profiler.start()
    total_ms, my_ms, last = timed(step_resident, args.steps)
    if args.profile_range:
        torch.cuda.profiler.stop()
    clocks = sampler.stop()
    launches = net.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        if kind == "generator":
            outs = {"audio": last}
        elif sharded:
            outs = {"audio": last[0], "audio_index_and_samples": last[1]}
        else:
            outs = {"audio" if len(last) == 1 else f"audio_{i}": o_ for i, o_ in enumerate(last)}
            if chunk is None:
                outs["y_lengths"] = net.last_y_lengths
        dump_outputs(outs, args.dump_outputs)
    last = None

    if kind != "generator":
        frames_rank = state.get("frames_local", state["frames"]) if sharded else state["frames"]
        Ty = state["Ty"]
    y_gpu = net.last_y_lengths.cpu() if kind != "generator" and not sharded and chunk is None else None

    for _ in range(2):
        step_e2e()
    d2h_drain()
    e2e_ms, _, _ = timed(step_e2e, args.steps, drain=d2h_drain)
    if kind != "generator":
        d2h = state["d2h"] + 8

    # ---- dominant block: the HiFi-GAN generator, timed alone with CUDA events on the launch stream
    Bg = min(B, wl["batch"])
    Tg = Ty if Ty else wl.get("frames", 640)
    if kind == "generator":
        gen_fn = step_resident
    else:
        z_in = torch.randn(Bg, Cc, Tg, device=dev, generator=gen)
        sid_g = torch.zeros(Bg, dtype=torch.long, device=dev)
        g_in = net.emb_g(sid_g)[:, :, None] if wl["n_spk"] > 0 else None

        def gen_fn():
            return net.dec(z_in, g=g_in)
    for _ in range(2):
        gen_fn()
    gsteps = max(2, min(args.steps, 5))
    gen_ms = timed(gen_fn, gsteps)[0] / gsteps

    # ---- job totals and per-rank attribution
    per_rank = torch.tensor([float(frames_rank), my_ms / args.steps, float(Ty), clocks.get("sm_mhz") or 0.0,
                             float(clocks.get("sw_power_cap_samples", 0))], device=dev, dtype=torch.float64)
    if dist:
        allr = [torch.zeros_like(per_rank) for _ in range(world)]
        dist.all_gather(allr, per_rank)
    else:
        allr = [per_rank]
    allr = [t.tolist() for t in allr]
    frames_job = sum(r[0] for r in allr)
    audio_job = frames_job * hop / sr
    ms_per_step = total_ms / args.steps
    value = audio_job / (ms_per_step / 1e3)
    e2e_value = audio_job / (e2e_ms / args.steps / 1e3)

    cpu = gpu_eager = dur_check = None
    if rank == 0 and world == 1 and not args.no_cpu:
        arm = CpuArm(args.workload)
        threads = arm.pick_threads()
        n_cpu = wl["cpu_utts"]
        a_s, dt, y_cpu = arm.run(n_cpu)
        what = "Generator.forward" if kind == "generator" else "SynthesizerTrn.infer"
        src = "unmodified reference module (oracle/_ref)" if arm.kind == "reference" else "oracle port"
        cpu = {"value": a_s / dt, "unit": "audio-s/s", "cores": threads, "kind": arm.kind,
               "sample": f"{n_cpu} of the workload's utterances, {what}, {src}, {dt:.1f} s", "same_config": False}
        if y_cpu is not None and y_gpu is not None and not net.use_sdp:
            # the duration predictor is deterministic (v3): the GPU's own frame counts of the sampled utterances must
            # equal the reference's (the numerator of the metric comes from them)
            n = min(len(y_cpu), len(y_gpu))
            dur_check = {"utterances": n, "y_length_mismatches": int((y_cpu[:n] != y_gpu[:n]).sum()),
                         "frames_gpu": int(y_gpu[:n].sum()), "frames_reference": int(y_cpu[:n].sum())}
        if not args.no_gpu_eager:
            try:   # the same reference code in eager mode on this GPU (SURVEY.md §8d "reference-on-B200")
                arm.to(dev)
                n_e = min(wl["batch"], max(n_cpu, 16))
                arm.run(n_e, dev)     # warm-up at the timed shape (cuDNN picks its algorithms per shape on first use)
                a_e, dt_e, _ = arm.run(n_e, dev)
                gpu_eager = {"value": a_e / dt_e, "unit": "audio-s/s", "kind": arm.kind + " (PyTorch eager, cuDNN/cuBLAS, fp32)",
                             "sample": f"{n_e} utterances, {dt_e * 1e3:.0f} ms"}
            except Exception as e:
                gpu_eager = {"unavailable": repr(e)[:200]}

    if rank == 0:
        hbm_peak, tens_sus, tens_burst, which = peaks()
        tformat = "tf32"
        try:
            v = (__import__("ctypes").c_int)(0)
            if lib.wetts_get_option(b"tensor_format", __import__("ctypes").byref(v)) == 0 and v.value == 16:
                tformat = "f16"
        except Exception:
            pass
        # dense peak of the operand format in use: kind::f16 = the measured bf16 figure, kind::tf32 = half of it
        tens_peak = (tens_sus if tformat == "f16" else tens_sus / 2.0)
        gen_frames = Bg * Tg if kind != "generator" else frames_rank          # the generator runs the padded tail too
        gen_flop = GEN_FLOP_PER_FRAME[fam] * gen_frames
        gen_bytes = GEN_LAYER_BYTES_PER_FRAME[fam] * gen_frames
        issued = 3.0 * gen_flop if args.tensor_cores else gen_flop          # three operand-split products per fp32 product
        traffic, traffic_src = measured_traffic(args.workload) if (args.fused_resblock and args.tensor_cores and not args.batch) else (None, None)
        line = {
            "metric": "audio-seconds/sec (VITS infer)", "value": value, "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32 (3x%s operand split on tcgen05, fp32 accumulate)" % tformat if args.tensor_cores else "f32",
            "data": "synthetic",
            "config": {"workload": args.workload, "baseline_config_index": wl["baseline_config"], "config": cfg_name,
                       "kind": kind, "tensor_cores": bool(args.tensor_cores), "fused_resblock": bool(args.fused_resblock),
                       "length_aware": bool(args.length_aware),
                       "batch_per_gpu": B, "batch_job": B_job, "phonemes": wl.get("phonemes"), "frames_max": Ty,
                       "valid_frames_job": int(frames_job), "length_scale": ls, "sampling_rate": sr,
                       "scales": [NOISE_SCALE, ls, NOISE_SCALE_W],
                       "parallelism": (f"batch-sharded x{world}: NCCL scatter of ids + gather of waveforms inside the timed region"
                                       if sharded else (f"independent replicas x{world}" if world > 1 else "single GPU")),
                       "l2": ("explicit 256 MiB flush between timed steps" if flush_buf is not None
                              else "working set >> L2 (multi-GB activations per step); no explicit flush")},
            "rtf": 1.0 / value,
            "latency_ms_per_utterance": ms_per_step if B_job == 1 else None,
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms / args.steps,
                    "d2h": "pipelined: step i's copy overlaps step i+1, last copy waited for inside the timed region" if pipelined
                    else "serial: copy, then synchronize, every step"},
            "gpu_launches": int(launches), "gpu_launches_per_step": int(launches) // max(args.steps, 1),
            "clocks": clocks,
            "per_rank": [{"rank": i, "valid_frames": int(r[0]), "ms_per_step": r[1], "frames_max": int(r[2]),
                          "sm_mhz": r[3], "sw_power_cap_samples": int(r[4])} for i, r in enumerate(allr)],
            "roofline": {"bound": "tensor", "kernel": "HiFi-GAN generator conv stack (wetts_generator_forward), timed alone",
                         "achieved": issued / (gen_ms / 1e3) / 1e12, "peak": tens_peak, "unit": "TFLOP/s",
                         "frac": issued / (gen_ms / 1e3) / 1e12 / tens_peak,
                         "flops": f"issued tensor-pipe flops = 3 x algorithmic fp32 flops ({GEN_FLOP_PER_FRAME[fam] / 1e6:.2f} MFLOP/frame x {gen_frames} padded frames)",
                         "fp32_equivalent_tflops": gen_flop / (gen_ms / 1e3) / 1e12,
                         "peak_source": f"{which}: dense {'bf16/f16' if tformat == 'f16' else 'tf32 = bf16 / 2'} sustained; burst {tens_burst if tformat == 'f16' else tens_burst / 2:.0f}",
                         "ms": gen_ms, "traffic": traffic, "traffic_source": traffic_src,
                         "hbm_layer_boundary": {"achieved": gen_bytes / (gen_ms / 1e3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                                "frac": gen_bytes / (gen_ms / 1e3) / 1e9 / hbm_peak,
                                                "algorithmic_bytes": gen_bytes,
                                                "compulsory_bytes": GEN_COMPULSORY_BYTES_PER_FRAME * gen_frames,
                                                "note": "north_star's HBM figure on layer-boundary bytes (BASELINE.md §4); not the binding roof"}},
            "generator_share_of_step": (gen_ms * (B / Bg)) / ms_per_step if kind != "generator" else 1.0,
            "duration_check": dur_check,
            "cpu_baseline": cpu,
            "gpu_eager_baseline": gpu_eager,
        }
        emit(line)
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--dist", default="sharded", choices=["sharded", "replicas"],
                    help="N > 1: rank 0 deals the job over NCCL (default) or independent per-rank batches")
    ap.add_argument("--batch", type=int, default=0, help="override utterances per GPU")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / gpu_eager legs")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the reference-in-eager-mode-on-this-GPU leg")
    ap.add_argument("--profile-range", action="store_true",
                    help="wrap the timed region in cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--tensor-cores", type=int, default=1, help="0: force the fp32 SIMT kernels")
    ap.add_argument("--fused-resblock", type=int, default=1, help="0: one launch per generator conv (no fused MRF stage kernel)")
    ap.add_argument("--tensor-format", type=int, default=0, choices=[0, 16, 32],
                    help="operand format of the fused stage kernels: 16 = f16 split, 32 = 3xTF32, 0 = library default")
    ap.add_argument("--attention-tc", type=int, default=-1, help="1/0: text-encoder attention on the tensor pipe (-1: library default)")
    ap.add_argument("--length-aware", type=int, default=0, help="1: skip generator tiles beyond each utterance's own length")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (rank 0; at most 64 MB, rows sampled "
                         "with a fixed seed beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
