#!/usr/bin/env python
"""bench.py -- AF3-7B audio->text hot path on B200 (driver contract; see DESIGN.md "Measurement").

Workload (BASELINE.json configs[1]): AF3-7B, batch 32 x 30 s clips per GPU, greedy 128-token decode.
One "step" = one pass of the whole path over one batch of synthetic audio:
    log-mel -> AF-Whisper encoder -> projector -> prompt embedding scatter -> Qwen2 prefill -> 127 cached decode steps
`value`  = generated tokens/s for the whole job with the waveform batch already resident in HBM.
`e2e`    = the same through the public API from HOST buffers: pinned-host waveforms + prompt ids are copied to the
           device and the generated ids are read back inside the timed region.
Also reported (BASELINE's metric pair): audio_s_per_s (mel+encoder+projector) and decode_tok_s (cached steps only),
a roofline object for the dominant kernel, and the reference's CPU path timed on this box's host cores.

`--impl reference` times the reference's own implementation of the path (unmodified Hugging Face transformers classes,
see oracle/af3_oracle.py) on the host cores, on bounded samples of the same workload.

Multi-GPU (torchrun, one rank per GPU): weights replicated, every rank runs its own 32-clip batch (weak scaling),
the only collective is the final all-gather of the generated ids (NCCL).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOAD = "AF3-7B batch-32 x 30s clips, greedy 128-token decode"
METRIC = "generated tokens/s, audio->text end to end (log-mel + AF-Whisper encode + prefill + greedy decode), AF3-7B"
B_PER_GPU, CLIP_S, NEW_TOKENS = 32, 30.0, 128
N_PRE, N_POST = 5, 25


# ----------------------------------------------------------------------------------------------------- helpers
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def cpu_throttle_snapshot():
    """cgroup CPU-quota throttling counters of this container (v2 or v1 path); None when not exposed."""
    for path in ("/sys/fs/cgroup/cpu.stat", "/sys/fs/cgroup/cpu/cpu.stat", "/sys/fs/cgroup/cpu,cpuacct/cpu.stat"):
        try:
            kv = dict(ln.split() for ln in open(path).read().strip().splitlines())
            return {"nr_throttled": int(kv.get("nr_throttled", 0)),
                    "throttled_ms": int(kv.get("throttled_usec", int(kv.get("throttled_time", 0)) // 1000)) / 1e3}
        except Exception:
            continue
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])), mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "MEASURED_PEAKS.json (of measured)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "B200_PROFILING.md fallback (of fallback)"}


def af3_config():
    from transformers import AudioFlamingo3Config

    text = dict(vocab_size=152064, hidden_size=3584, intermediate_size=18944, num_hidden_layers=28, num_attention_heads=28,
                num_key_value_heads=4, max_position_embeddings=32768, rms_norm_eps=1e-6, tie_word_embeddings=False,
                rope_parameters={"rope_type": "default", "rope_theta": 1000000.0})
    return AudioFlamingo3Config(audio_config=dict(), text_config=text, audio_token_id=151669)


def synth_batch(B: int, seed: int):
    """Seeded synthetic batch (SURVEY.md 8-d): 30 s noise clips and [5 text] + 750 x <sound> + [25 text] prompts."""
    rs = np.random.RandomState(seed)
    wave = (rs.randn(B, int(CLIP_S * 16000)) * 0.1).astype(np.float32)
    tok = 750
    ids = np.empty((B, N_PRE + tok + N_POST), dtype=np.int64)
    ids[:, :N_PRE] = rs.randint(1, 151643, size=(B, N_PRE))
    ids[:, N_PRE:N_PRE + tok] = 151669
    ids[:, N_PRE + tok:] = rs.randint(1, 151643, size=(B, N_POST))
    return wave, ids


def dump_outputs(out_dir, generated_ids):
    """Writes what the timed path returned in its last step -- the generated ids [global batch, prompt + new tokens], prompt
    included, as generate() returns them -- to out_dir/generated_ids.npy.  Inputs and weights are seeded, so two builds run with
    the same arguments can be compared output for output.  The ids are stored as float64, a floating-point format in which they
    are exact."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "generated_ids.npy", generated_ids.cpu().numpy().astype(np.float64))


def init_synthetic_weights_(model, seed: int):
    """Random-init weights of the AF3-7B architecture directly on the GPU (no checkpoint exists offline):
    N(0, 0.02) matrices / embeddings, zero biases, unit norm gains -- the reference's default init family."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("bias"):
                p.zero_()
            elif "norm" in name and name.endswith("weight"):
                p.fill_(1.0)
            else:
                p.normal_(0.0, 0.02, generator=g)


# ----------------------------------------------------------------------------------------------------- HF on the same GPU
def _cuda_ms(fn, warm=1, iters=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def gpu_reference(model, cfg, dev, feats, fmask, ids, our_stage_ms, our_ms_step):
    """The number the kernels have to beat (SURVEY 8-d, BASELINE.md 3): the reference's own implementation of the path -- unmodified HF
    transformers classes, eager bf16, attn_implementation sdpa -- on the SAME B200, SAME weights (parameters are shared with our model
    through load_state_dict(assign=True): no second copy), same batch: per stage and for the whole generate() call."""
    import transformers
    from transformers import AudioFlamingo3ForConditionalGeneration as HFModel

    with torch.device("meta"):
        ref = HFModel(cfg)
    ref.load_state_dict(model.state_dict(), assign=True)
    for mod in ref.modules():  # non-persistent rotary buffer: fp32, computed on the CPU like the reference does, then moved
        if hasattr(mod, "inv_freq") and hasattr(mod, "compute_default_rope_parameters"):
            inv, _ = mod.compute_default_rope_parameters(mod.config)
            mod.inv_freq = inv.to(dev)
            mod.original_inv_freq = inv.clone().to(dev)
    ref.eval()
    ref.generation_config.pad_token_id = 0
    ref.generation_config.eos_token_id = None
    B, S = ids.shape
    f16 = feats.to(torch.bfloat16)
    am = torch.ones_like(ids)
    out = {"impl": f"HF transformers {transformers.__version__} eager bf16 (sdpa) on the same GPU, same weights, same batch", "stage_ms": {}}
    with torch.no_grad():
        out["stage_ms"]["encode_project"] = _cuda_ms(lambda: ref.get_audio_features(f16, fmask))
        lm = ref.language_model
        x = (torch.randn((B, S, cfg.text_config.hidden_size), device=dev, dtype=torch.float32) * 0.02).to(torch.bfloat16)
        holder = {}

        def prefill():
            holder["o"] = lm(inputs_embeds=x, attention_mask=am, use_cache=True, logits_to_keep=1)

        out["stage_ms"]["prefill"] = _cuda_ms(prefill)
        cache = holder["o"].past_key_values
        tok = torch.randint(1, 1000, (B, 1), device=dev)
        n_dec, state = 8, {"mask": am}

        def decode_steps():
            for _ in range(n_dec):
                state["mask"] = torch.cat([state["mask"], torch.ones((B, 1), dtype=am.dtype, device=dev)], 1)
                lm(input_ids=tok, attention_mask=state["mask"], past_key_values=cache, use_cache=True, logits_to_keep=1)

        out["stage_ms"]["decode_step"] = _cuda_ms(decode_steps, warm=1, iters=1) / n_dec
        del cache, holder
        kw = dict(input_ids=ids, attention_mask=am, input_features=f16, input_features_mask=fmask, do_sample=False)
        ref.generate(**kw, max_new_tokens=4)
        out["generate_ms"] = _cuda_ms(lambda: ref.generate(**kw, max_new_tokens=NEW_TOKENS), warm=0, iters=1)
    out["tokens_per_s"] = B * NEW_TOKENS / (out["generate_ms"] / 1e3)
    out["note"] = ("log-mel is outside the reference's GPU timings (WhisperFeatureExtractor runs on the host); generate_ms = encoder + projector + "
                   "prefill + 127 cached steps, one call after a 4-token warm-up")
    ours = {"encode_project": our_stage_ms.get("encode_project"), "prefill": our_stage_ms.get("prefill"),
            "decode_step": (our_stage_ms.get("decode") or 0) / (NEW_TOKENS - 1) or None}
    out["ours_stage_ms"] = ours
    out["vs_hf_gpu"] = {k: (out["stage_ms"][k] / v if v else None) for k, v in ours.items()}
    out["vs_hf_gpu"]["generate_e2e"] = out["generate_ms"] / our_ms_step
    out["losses"] = [k for k, v in out["vs_hf_gpu"].items() if v is not None and v < 1.0]
    del ref
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------------- ours
def run_ours(args):
    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        # NCCL prints its version banner straight to file descriptor 1 when the first communicator comes up (NCCL_DEBUG_FILE
        # does not move it); stdout carries the ONE JSON line of the contract, so fd 1 points at stderr while the communicator
        # is created (init + one barrier) and is restored afterwards.
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    from audio_flamingo_b200 import AF3FeatureExtractor, AudioFlamingo3ForConditionalGeneration, ops
    from audio_flamingo_b200.sharding import gather_tokens

    cfg = af3_config()
    model = AudioFlamingo3ForConditionalGeneration(cfg)
    model.to_empty(device=dev)
    model.to(torch.bfloat16)
    init_synthetic_weights_(model, seed=0)
    fe = AF3FeatureExtractor(dev)
    # weak scaling (the driver's contract): 32 clips per GPU.  --scaling strong: the global batch of 32 is split over the ranks
    # (SURVEY 8-e asks for this to be REPORTED: decode tokens/s per GPU drops when the per-GPU batch shrinks, the 14 GB of weights are
    # streamed every step regardless)
    B = B_PER_GPU if args.scaling == "weak" else max(B_PER_GPU // world, 1)
    wave_np, ids_np = synth_batch(B, seed=1000 + rank)
    wave_host = torch.from_numpy(wave_np).pin_memory()
    ids_host = torch.from_numpy(ids_np).pin_memory()
    wave_dev = wave_host.to(dev)
    ids_dev = ids_host.to(dev)
    mask_dev = torch.ones_like(ids_dev)
    n_samples = [wave_np.shape[1]] * B
    tokens_host = torch.empty((B * world, ids_np.shape[1] + NEW_TOKENS), dtype=torch.int64).pin_memory()

    def step(from_host: bool):
        if from_host:
            w = wave_host.to(dev, non_blocking=True)
            ids = ids_host.to(dev, non_blocking=True)
        else:
            w, ids = wave_dev, ids_dev
        feats = fe.from_device_waveform(w, n_samples)
        model._mark("mel_done")
        out = model.generate(input_ids=ids, attention_mask=mask_dev, input_features=feats["input_features"],
                             input_features_mask=feats["input_features_mask"], max_new_tokens=NEW_TOKENS, do_sample=False)
        out = gather_tokens(out, assume_equal_length=True)   # the path's only collective (NCCL all-gather of int64 ids; no EOS here)
        if from_host:
            tokens_host.copy_(out, non_blocking=True)  # D2H read of the step's result
        return out

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    host_t = []  # per timed step: [(stage name, host perf_counter when that stage boundary was ENQUEUED)]

    def timed(n_steps, from_host, collect_stages=False):
        barrier()
        ops.LAUNCHES = 0
        stages = []
        out = None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_steps):
            if collect_stages:
                model.stage_events = []
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                model.stage_events.append(("step_start", ev))
                model.stage_host_t = []
            out = step(from_host)
            if collect_stages:
                stages.append(model.stage_events)
                host_t.append(model.stage_host_t)
                model.stage_events = None
                model.stage_host_t = None
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist

            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, ops.LAUNCHES, stages, out

    # The clock sampler (one long-lived `nvidia-smi -lms` process) is started BEFORE the warm-up steps: its start-up (NVML attach)
    # stalls work submission on the GPU for a while, which must not land inside the timed region.  AF3_BENCH_SAMPLER=late
    # restores the old placement (right before the timed steps), =off disables it (diagnostics only: clocks is then null).
    sampler_mode = os.environ.get("AF3_BENCH_SAMPLER", "early")
    sampler = ClockSampler(local)
    if rank == 0 and sampler_mode == "early":
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step(False)
    if rank == 0 and sampler_mode == "early":
        sampler.lines.clear()  # keep only the samples taken during the timed region
    if rank == 0 and sampler_mode == "late":
        sampler.start()
    thr0 = cpu_throttle_snapshot()
    ms_dev, launches, stages, last_out = timed(args.steps, from_host=False, collect_stages=True)
    thr1 = cpu_throttle_snapshot()
    host_cpu = {"cpus_allowed": len(os.sched_getaffinity(0)), "loadavg": os.getloadavg()[0],
                "throttled_during_timed": None if (thr0 is None or thr1 is None) else
                {"nr": thr1["nr_throttled"] - thr0["nr_throttled"], "ms": round(thr1["throttled_ms"] - thr0["throttled_ms"], 1)}}
    clocks = sampler.stop() if (rank == 0 and sampler_mode != "off") else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_out)
    step(True)  # warm the host path (pinned staging, H2D)
    ms_e2e, _, _, _ = timed(args.steps, from_host=True)

    # one profiled step (per-kernel CUDA events around every launch; PDL off so kernels do not overlap their brackets;
    # the decode steps replayed from the CUDA graph are not bracketed, the first -- eager -- decode step is)
    ops.PROFILE = {}
    pdl_env = os.environ.get("AF3_PDL")
    os.environ["AF3_PDL"] = "0"
    torch.cuda.synchronize()
    step(False)
    torch.cuda.synchronize()
    if pdl_env is None:
        os.environ.pop("AF3_PDL")
    else:
        os.environ["AF3_PDL"] = pdl_env
    prof, ops.PROFILE = ops.PROFILE, None

    # one more step with the library's in-graph timeline open (PDL on, CUDA graph, nothing serialised): per-launch %globaltimer
    # stamps of the LAST replay of the decode graph.  A decode-step kernel's duration for the roofline is its SLOT in the chain --
    # last CTA exit minus the predecessor's last exit, dependency latency included; the slots add up to the step.
    trace_by_key = {}
    trace_step_us = None
    try:
        from audio_flamingo_b200.trace import DecodeTrace

        model.release_decode_state()
        with DecodeTrace(dev) as tr:
            step(False)
        tl = tr.graph_launches()
        model.release_decode_state()  # that graph writes into tr.buf on every replay: drop it with the trace
        del tr
        for r in tl:
            if r.get("slot_us") is not None:
                trace_by_key.setdefault(tuple(r["key"]), []).append(r)
        if tl:
            trace_step_us = max(r["exit_max"] for r in tl if r["exit_max"] is not None) - tl[0]["entry_min"]
    except Exception as e:  # measurement aid only
        trace_by_key = {"error": repr(e)}

    def region_ms(fn, iters=3, warm=1):
        """fn() timed on the device, max over ranks (same rule as the main number)."""
        for _ in range(warm):
            fn()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(iters):
            fn()
        a1.record()
        barrier()
        ms = a0.elapsed_time(a1) / iters
        if world > 1:
            import torch.distributed as dist

            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    extras = {}
    if not args.no_extras:
        peaks_x = measured_peaks()
        # ---- BASELINE config 3: encoder-only throughput, 32 x 30 s windows per GPU (256 on 8 GPUs), mel + tower + projector
        W3 = 32
        wave3 = wave_dev if B == W3 else torch.from_numpy(synth_batch(W3, seed=3000 + rank)[0]).to(dev)

        def enc_only():
            f = fe.from_device_waveform(wave3, [wave3.shape[1]] * W3)
            model.get_audio_features(f["input_features"], f["input_features_mask"])

        ms3 = region_ms(enc_only)
        tf3 = W3 * (2.274e12 + 26.15e9) / (ms3 * 1e-3) / 1e12
        extras["config3_encoder_only"] = {
            "workload": "AF3-7B encoder-only (log-mel + AF-Whisper 32 layers + projector), 32 x 30 s windows per GPU (BASELINE configs[2]: 256 on 8 GPUs)",
            "windows_per_gpu": W3, "n_gpus": world, "ms": ms3, "audio_s_per_s": world * W3 * CLIP_S / (ms3 * 1e-3),
            "tflops_per_gpu": tf3, "frac_of_bf16_sustained_peak": tf3 / peaks_x["bf16_tflops_sustained"],
            "flops_per_window": 2.274e12 + 26.15e9}
        del wave3
        # ---- log-mel alone at config-3 scale (256 windows in one launch): the stage is latency-bound at 32 windows
        W256 = 256
        wave256 = torch.randn((W256, int(CLIP_S * 16000)), device=dev, dtype=torch.float32) * 0.1
        ms_mel = region_ms(lambda: ops.logmel(wave256, fe.tables), iters=5)
        mel_bytes = W256 * (480000 * 4 + 128 * 3000 * 4)
        extras["logmel_256_windows"] = {"ms": ms_mel, "algorithmic_bytes": mel_bytes, "gbs": mel_bytes / (ms_mel * 1e-3) / 1e9,
                                        "frac_of_hbm_peak": mel_bytes / (ms_mel * 1e-3) / 1e9 / peaks_x["hbm_gbs"],
                                        "audio_s_per_s_per_gpu": W256 * CLIP_S / (ms_mel * 1e-3)}
        del wave256
        # ---- BASELINE config 5: 4 audio segments (4 x 750 audio tokens) + 512 text tokens per sequence, 2 sequences per GPU (16 on 8)
        B5, SP5 = 2, 4
        rs5 = np.random.RandomState(5000 + rank)
        wave5 = torch.from_numpy((rs5.randn(B5 * SP5, int(CLIP_S * 16000)) * 0.1).astype(np.float32)).to(dev)
        seg = [102, 102, 102, 102, 104]  # 512 text tokens around / between the four <sound> spans
        rows5 = []
        for _ in range(B5):
            row = []
            for k in range(SP5):
                row += rs5.randint(1, 151643, size=seg[k]).tolist() + [151669] * 750
            rows5.append(row + rs5.randint(1, 151643, size=seg[4]).tolist())
        ids5 = torch.tensor(rows5, dtype=torch.int64, device=dev)
        am5 = torch.ones_like(ids5)
        S5 = ids5.shape[1]

        def cfg5():
            f = fe.from_device_waveform(wave5, [wave5.shape[1]] * (B5 * SP5))
            model(input_ids=ids5, attention_mask=am5, input_features=f["input_features"], input_features_mask=f["input_features_mask"],
                  logits_to_keep=1)

        ms5 = region_ms(cfg5)
        fl5 = B5 * (S5 * 2 * 6525618176.0 + 28 * 4 * 28 * 128 * S5 * S5 / 2.0) + B5 * SP5 * (2.274e12 + 26.15e9)
        extras["config5_chat_prefill"] = {
            "workload": "AF3-Chat layout: 4 x 30 s audio segments + 512 text tokens per sequence (S = 3512), 2 sequences per GPU (BASELINE configs[4]: 16 on 8 GPUs), mel + encoder + projector + prefill",
            "seq_per_gpu": B5, "prompt_len": S5, "n_gpus": world, "ms": ms5, "prompt_tok_s": world * B5 * S5 / (ms5 * 1e-3),
            "tflops_per_gpu": fl5 / (ms5 * 1e-3) / 1e12, "frac_of_bf16_sustained_peak": fl5 / (ms5 * 1e-3) / 1e12 / peaks_x["bf16_tflops_sustained"]}
        del wave5
        model.release_decode_state()
        torch.cuda.empty_cache()

    if rank != 0:
        return
    peaks = measured_peaks()
    n_tok_total = B * world * NEW_TOKENS
    ms_step = ms_dev / args.steps
    # stage breakdown (rank 0, mean over steps)
    names = ["mel", "encode_project", "prefill", "decode"]
    keys = [("step_start", "mel_done"), ("start", "audio_done"), ("audio_done", "prefill_done"), ("prefill_done", "decode_done")]
    stage_ms, stage_ms_per_step = {}, {}
    for nm, (a, b) in zip(names, keys):
        vals = []
        for evs in stages:
            d = dict(evs)
            if a in d and b in d:
                vals.append(d[a].elapsed_time(d[b]))
        stage_ms[nm] = sum(vals) / len(vals) if vals else None
        stage_ms_per_step[nm] = [round(v, 3) for v in vals]  # one entry per timed step: shows whether a slow mean is one step or all
    # host-side time spent ENQUEUEING the decode stage of each step (no sync inside): ~= the GPU time when launch-bound,
    # much smaller when the GPU is the bottleneck
    host_decode_enqueue_ms, host_token_gaps = [], []
    for ht in host_t:
        d = {k: v for k, v in (ht or []) if k != "tok"}
        if "prefill_done" in d and "decode_done" in d:
            host_decode_enqueue_ms.append(round((d["decode_done"] - d["prefill_done"]) * 1e3, 3))
            # host time between consecutive token enqueues (token 1 = eager warm step, token 2 = graph capture, then replays)
            ts = [d["prefill_done"]] + [v for k, v in ht if k == "tok"]
            gaps = [(b - a) * 1e3 for a, b in zip(ts, ts[1:])]
            if gaps:
                imax = max(range(len(gaps)), key=gaps.__getitem__)
                host_token_gaps.append({"first3_ms": [round(g, 1) for g in gaps[:3]], "median_ms": round(statistics.median(gaps), 3),
                                        "max_ms": round(gaps[imax], 1), "max_at_token": imax + 1,
                                        "n_over_20ms": sum(g > 20 for g in gaps[3:])})
    audio_ms = (stage_ms["mel"] or 0) + (stage_ms["encode_project"] or 0)
    audio_s_per_s = B * world * CLIP_S / (audio_ms / 1e3) if audio_ms else None
    decode_tok_s = B * world * (NEW_TOKENS - 1) / (stage_ms["decode"] / 1e3) if stage_ms["decode"] else None

    # per-kernel table from the profiled step.  Kernels of the cached decode step were bracketed once (the eager step; the other
    # NEW_TOKENS - 2 steps are graph replays): their time is weighted by the NEW_TOKENS - 1 steps they stand for, so the
    # "dominant kernel" is dominant over the WHOLE step, replays included (VERDICT r01)
    table = []
    S_prompt = int(ids_np.shape[1])
    for key, evs in prof.items():
        kind, a, b, c, flags, phase = key
        ms_list = [e0.elapsed_time(e1) for e0, e1 in evs]
        tot = sum(ms_list)
        n = len(evs)
        weight = (NEW_TOKENS - 1) if phase == "decode" else 1
        row = {"phase": phase or "prefill/encoder", "launches_bracketed": n, "ms_total_bracketed": tot, "ms_per_launch": tot / n,
               "ms_in_step": tot * weight, "timing": "CUDA events around every launch of one profiled step (PDL off for that step)"}
        tr_recs = trace_by_key.get((kind, a, b, c, flags)) if phase == "decode" and isinstance(trace_by_key, dict) else None
        if tr_recs:
            # in-graph slot (see above): replaces the event bracket, which adds 10-15 us of launch gap to every small kernel
            slot_ms = sum(r["slot_us"] for r in tr_recs) / len(tr_recs) / 1e3
            row.update({"ms_per_launch_events": tot / n, "ms_per_launch": slot_ms, "launches_per_decode_step": len(tr_recs),
                        "ms_in_step": slot_ms * len(tr_recs) * (NEW_TOKENS - 1),
                        "body_us": sum(r.get("body_us", 0) for r in tr_recs) / len(tr_recs),
                        "stream_us": sum(r.get("stream_us", 0) or 0 for r in tr_recs) / len(tr_recs),
                        "tail_us": sum(r.get("tail_us", 0) or 0 for r in tr_recs) / len(tr_recs),
                        "timing": "in-graph %globaltimer trace of the last decode-graph replay (PDL on): slot = last CTA exit - predecessor's last exit"})
            tot, n = slot_ms * len(tr_recs), len(tr_recs)
        if kind == "gemm":
            n_feat_w = b * 2 if (flags & 8) else b
            flops = 2.0 * a * n_feat_w * c
            # few-token GEMM: the weight matrix is the traffic (read once); activations / outputs are < 1 % of it
            bytes_alg = 2.0 * n_feat_w * c if a <= 64 else 2.0 * (a * c + n_feat_w * c + a * b)
            row.update({"kernel": "gemm_tcgen05" + ("(swap)" if a <= 64 else ""), "n_tok": a, "n_feat": b, "K": c, "flags": flags,
                        "tflops": flops * n / (tot * 1e-3) / 1e12, "gbs": bytes_alg * n / (tot * 1e-3) / 1e9,
                        "flops_per_launch": flops, "bytes_per_launch": bytes_alg, "bound": "hbm" if a <= 64 else "tensor"})
        elif kind == "attention":
            D = flags // 2
            causal = flags & 1
            flops = 4.0 * a * b * c * D * (0.5 if causal else 1.0)
            row.update({"kernel": "attention_tcgen05", "bh": a, "Tq": b, "Tk": c, "D": D, "causal": causal,
                        "tflops": flops * n / (tot * 1e-3) / 1e12, "flops_per_launch": flops, "bound": "tensor"})
        elif kind == "decode_attention":
            # a = sequences, b = query heads, c = cache capacity; K and V of the live context (prompt + 1 here) once: 4 KV heads x 128 x 2 B x 2
            bytes_alg = 2.0 * 4 * 128 * 2 * (S_prompt + 1) * a
            row.update({"kernel": "decode_attention", "shape": [a, b, c, flags], "gbs": bytes_alg * n / (tot * 1e-3) / 1e9,
                        "bytes_per_launch": bytes_alg, "bound": "hbm"})
        elif kind == "logmel":
            bytes_alg = a * (b * 4 + 128 * (b // 160) * 4)
            row.update({"kernel": "logmel", "n_win": a, "gbs": bytes_alg * n / (tot * 1e-3) / 1e9, "bytes_per_launch": bytes_alg, "bound": "hbm"})
        elif kind in ("rmsnorm", "layernorm"):
            bytes_alg = 2.0 * a * b * 2  # read + write one bf16 row each (the pooled variant reads two)
            row.update({"kernel": kind, "shape": [a, b, c, flags], "gbs": bytes_alg * n / (tot * 1e-3) / 1e9, "bytes_per_launch": bytes_alg,
                        "bound": "hbm"})
        elif kind == "rope":
            bytes_alg = 2.0 * a * b * c * 2
            row.update({"kernel": kind, "shape": [a, b, c, flags], "gbs": bytes_alg * n / (tot * 1e-3) / 1e9, "bytes_per_launch": bytes_alg,
                        "bound": "hbm"})
        else:
            row.update({"kernel": kind, "shape": [a, b, c, flags]})
        table.append(row)
    table.sort(key=lambda r: -r["ms_in_step"])
    # decode step breakdown (ms per step by kernel kind, from the eager step: PDL off, every launch bracketed)
    dec = {}
    for r in table:
        if r["phase"] != "decode":
            continue
        name = f"gemm {r['n_feat']}x{r['K']}" if r["kernel"].startswith("gemm") else r["kernel"]
        dec[name] = dec.get(name, 0.0) + (r["ms_per_launch"] * r["launches_per_decode_step"] if "launches_per_decode_step" in r else r["ms_total_bracketed"])
    ncu = {}
    ncu_file = ROOT / "profiles" / "ncu_summary.json"
    if ncu_file.exists():
        try:
            ncu = json.loads(ncu_file.read_text())
        except Exception:
            ncu = {}

    def roofline_of(r, traffic_key):
        if r is None:
            return None
        if r["bound"] == "tensor":
            peak, ach, unit = peaks["bf16_tflops_sustained"], r["tflops"], "TFLOP/s"
            src = peaks["source"] + ", sustained figure (kernel timed inside a long step)"
        else:
            peak, ach, unit = peaks["hbm_gbs"], r["gbs"], "GB/s"
            src = peaks["source"]
        desc = {k: r[k] for k in ("n_tok", "n_feat", "K", "flags", "bh", "Tq", "Tk", "D", "shape") if k in r}
        return {"kernel": f"{r['kernel']} {desc}", "phase": r["phase"], "bound": r["bound"], "achieved": ach, "peak": peak, "unit": unit,
                "frac": ach / peak, "peak_source": src, "ms_per_launch": r["ms_per_launch"], "ms_in_step": r["ms_in_step"],
                "share_of_step": r["ms_in_step"] / ms_step, "algorithmic_per_launch": r.get("flops_per_launch") if r["bound"] == "tensor" else r.get("bytes_per_launch"),
                "traffic": ncu.get(traffic_key), "timing": r["timing"]}

    rated = [r for r in table if "bound" in r]
    top = rated[0] if rated else None
    roofline = roofline_of(top, "gemm_decode_traffic_bytes" if (top and top["kernel"].endswith("(swap)")) else "gemm_prefill_traffic_bytes")
    top_prefill = next((r for r in rated if r["kernel"] == "gemm_tcgen05"), None)
    roofline_prefill_gemm = roofline_of(top_prefill, "gemm_prefill_traffic_bytes")
    # decode-step HBM roofline (whole step): weights once + KV of the live context
    dec_bytes = 2.0 * (6525618176 + 544997376) + 57344.0 * (S_prompt + NEW_TOKENS // 2) * B
    decode_roofline = None
    if stage_ms["decode"]:
        step_ms = stage_ms["decode"] / (NEW_TOKENS - 1)
        gbs = dec_bytes / (step_ms * 1e-3) / 1e9
        decode_roofline = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                           "ms_per_decode_step": step_ms, "bytes_per_step": dec_bytes}

    gpu_ref = None
    if world == 1 and not args.no_gpu_reference and args.scaling == "weak":
        try:
            feats0 = fe.from_device_waveform(wave_dev, n_samples)
            gpu_ref = gpu_reference(model, cfg, dev, feats0["input_features"], feats0["input_features_mask"], ids_dev, stage_ms, ms_step)
        except Exception as e:  # reported context; never let it kill the GPU line
            gpu_ref = {"error": repr(e)}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_reference(sample="small")
        except Exception as e:  # the baseline is reported context; never let it kill the GPU line
            cpu = {"error": repr(e)}

    line = {
        "metric": METRIC, "value": n_tok_total / (ms_step / 1e3), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic (seeded noise audio, random-init AF3-7B weights, random prompt ids)",
        "config": {"workload": WORKLOAD, "per_gpu_batch": B, "global_batch": B * world, "clip_seconds": CLIP_S, "prompt_len": int(ids_np.shape[1]),
                   "new_tokens": NEW_TOKENS, "parallelism": f"dp{world} (batch sharded, weights replicated)",
                   "l2": "inputs larger than L2 (16.5 GB of weights streamed every step; no flush needed)"},
        "e2e": {"value": n_tok_total / (ms_e2e / args.steps / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": int(wave_host.numel() * 4 + ids_host.numel() * 8),
                "d2h_bytes_per_step": int(tokens_host.numel() * 8), "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "audio_s_per_s": audio_s_per_s, "decode_tok_s": decode_tok_s, "stage_ms": stage_ms, "stage_ms_per_step": stage_ms_per_step, "host_decode_enqueue_ms": host_decode_enqueue_ms, "host_token_gaps": host_token_gaps, "host_cpu": host_cpu,
        "roofline": roofline, "roofline_prefill_gemm": roofline_prefill_gemm, "roofline_decode_step": decode_roofline,
        "kernels": table[:32], "decode_step_kernel_ms": dec, "decode_step_us_in_graph_trace": trace_step_us,
        "gpu_reference": gpu_ref, "extras": extras,
        "cpu_baseline": cpu, "clocks": clocks,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------- reference (CPU)
class CpuReference:
    """The reference's own PyTorch path (unmodified HF classes) on this box's host cores, bf16, all threads.
    Bounded samples of the SAME workload, composed linearly where the path is linear:
      * audio: WhisperFeatureExtractor + full 32-layer AF-Whisper encoder + projector on n_win windows of 30 s
      * prefill: Qwen2 decoder on one 780-token prompt with `layers` of the 28 identical layers (x 28/layers) + LM head
      * decode: cached q_len=1 steps at the workload's batch 32 / context 780 on the same sampled layers
    """

    def __init__(self, layers: int = 4, n_win: int = 1, n_dec: int = 1):
        from oracle import af3_oracle as O  # the checker; allowed here (cpu_baseline / --impl reference legs only)
        from transformers import AudioFlamingo3Config, AudioFlamingo3ForConditionalGeneration

        self.O = O
        self.cores = self._best_threads()
        torch.set_num_threads(self.cores)
        self.dtype, self.dtype_probe = self._best_dtype()
        self.host = self._host_info()
        self.layers, self.n_win, self.n_dec, self.S = layers, n_win, n_dec, 780
        text = dict(O.AF3_7B["text"])
        theta = text.pop("rope_theta")
        text["num_hidden_layers"] = layers
        self.cfg = AudioFlamingo3Config(audio_config=dict(O.AF3_7B["audio"]),
                                        text_config=dict(text, rope_parameters={"rope_type": "default", "rope_theta": theta}),
                                        audio_token_id=151669)
        with torch.device("meta"):
            model = AudioFlamingo3ForConditionalGeneration(self.cfg)
        model = model.to_empty(device="cpu").to(self.dtype).eval()
        torch.manual_seed(0)
        base = (torch.randn(1 << 22) * 0.02).to(torch.bfloat16)  # N(0, 0.02) block tiled into every tensor (fast init)
        with torch.no_grad():
            for name, p in model.named_parameters():
                flat = p.view(-1)
                if name.endswith("bias"):
                    flat.zero_()
                elif "norm" in name:
                    flat.fill_(1.0)
                else:
                    for o in range(0, flat.numel(), base.numel()):
                        n = min(base.numel(), flat.numel() - o)
                        flat[o:o + n] = base[:n].to(flat.dtype)
        for m in model.modules():  # rotary inv_freq is a non-persistent buffer: recompute after to_empty
            if hasattr(m, "inv_freq") and hasattr(m, "compute_default_rope_parameters"):
                inv, _ = m.compute_default_rope_parameters(m.config)
                m.inv_freq = inv
                m.original_inv_freq = inv.clone()
        self.model = model

    @staticmethod
    def _host_flags():
        try:
            for ln in open("/proc/cpuinfo"):
                if ln.startswith("flags"):
                    return set(ln.split(":", 1)[1].split())
        except OSError:
            pass
        return set()

    @staticmethod
    def _best_threads() -> int:
        """FIXED rule (VERDICT r01: the probed choice flipped between runs and moved the CPU figure 10x): one thread per physical core
        this process may use -- logical CPUs in the affinity mask / 2 (SMT) -- capped at 64, beyond which torch's CPU GEMMs stop scaling
        on these dual-socket hosts (DESIGN.md, round-1 measurements)."""
        try:
            n = len(os.sched_getaffinity(0))
        except AttributeError:
            n = os.cpu_count() or 1
        return max(1, min(n // 2 if n >= 4 else n, 64))

    @classmethod
    def _best_dtype(cls):
        """FIXED rule: bf16 (the dtype the reference's model card runs in) when the host has a native bf16 GEMM path (AMX-BF16 or
        AVX512-BF16), else fp32 -- emulated bf16 GEMMs are several times slower than fp32 and the CPU arm should not lose to an emulated
        dtype.  Decided from the ISA flags, not from a timing probe."""
        flags = cls._host_flags()
        native = bool({"amx_bf16", "avx512_bf16"} & flags)
        return (torch.bfloat16 if native else torch.float32), {"rule": "ISA flags", "native_bf16": native}

    @staticmethod
    def _host_info():
        """CPU model / relevant ISA flags / load: the CPU arm has been measured 100x apart on different boxes (DESIGN.md);
        this is what lets a reader tell a slow host from a slow implementation."""
        model, flags = None, set()
        try:
            for ln in open("/proc/cpuinfo"):
                if model is None and ln.startswith("model name"):
                    model = ln.split(":", 1)[1].strip()
                elif ln.startswith("flags") and not flags:
                    flags = set(ln.split(":", 1)[1].split())
        except OSError:
            pass
        return {"cpu_model": model, "logical_cpus": os.cpu_count(),
                "isa": sorted(f for f in ("amx_bf16", "amx_tile", "avx512_bf16", "avx512f", "avx2") if f in flags),
                "loadavg_1min": round(os.getloadavg()[0], 1)}

    @torch.no_grad()
    def sample(self):
        from transformers.cache_utils import DynamicCache

        O, cfg, model, S, layers, n_win, n_dec = self.O, self.cfg, self.model, self.S, self.layers, self.n_win, self.n_dec
        t_all0 = time.time()
        waves = O.synth_waveforms(n_win, CLIP_S, seed=1)
        t0 = time.time()
        feats, fmask = O.hf_features(waves)
        t_mel = time.time() - t0
        t0 = time.time()
        model.get_audio_features(feats.to(self.dtype), fmask)
        t_enc = time.time() - t0
        lm = model.language_model
        body = lm.model   # Qwen2Model: embedding + the sampled layers + final norm, WITHOUT the LM head (timed on its own below, so no
        #                   difference of two near-equal noisy times is ever taken -- VERDICT r01)
        emb = torch.randn(1, S, cfg.text_config.hidden_size).to(self.dtype) * 0.02
        t0 = time.time()
        body(inputs_embeds=emb, use_cache=True)
        t_pre_layers = time.time() - t0
        # decode at the workload's batch/context with a synthetic cache (prefilling 32 x 780 on the CPU would take minutes)
        Bd = B_PER_GPU
        cache = DynamicCache(config=cfg.text_config)
        Hkv, D = cfg.text_config.num_key_value_heads, cfg.text_config.hidden_size // cfg.text_config.num_attention_heads
        for li in range(layers):
            cache.update(torch.randn(Bd, Hkv, S, D).to(self.dtype), torch.randn(Bd, Hkv, S, D).to(self.dtype), li)
        ids = torch.randint(0, 1000, (Bd, 1))
        t0 = time.time()
        for i in range(n_dec):
            body(input_ids=ids, attention_mask=torch.ones(Bd, S + 1 + i, dtype=torch.long), past_key_values=cache, use_cache=True)
        t_dec_layers = (time.time() - t0) / n_dec
        x1 = torch.randn(Bd, cfg.text_config.hidden_size).to(self.dtype)
        lm.lm_head(x1)
        t0 = time.time()
        lm.lm_head(x1)
        t_head = time.time() - t0
        scale = 28.0 / layers
        B = B_PER_GPU
        t_audio = (t_mel + t_enc) / n_win * B
        t_prefill = t_pre_layers * scale * B + t_head            # head on the 32 last positions, once
        t_decode_step = t_dec_layers * scale + t_head
        total = t_audio + t_prefill + (NEW_TOKENS - 1) * t_decode_step
        import transformers

        dname = "bf16" if self.dtype == torch.bfloat16 else "fp32"
        return {
            "dtype": dname, "dtype_rule": self.dtype_probe, "host": self.host,
            "value": B * NEW_TOKENS / total, "unit": "tokens/s", "cores": self.cores, "kind": "reference",
            "sample": (f"HF transformers {transformers.__version__} {dname} on CPU, {self.cores} threads: mel+32-layer encoder+projector on {n_win} x 30 s "
                       f"window(s) (x{B}/{n_win}); prefill of one 780-token prompt on {layers}/28 decoder layers (x28/{layers} x{B}); "
                       f"{n_dec} cached decode step(s) at batch 32 / context 780 on {layers}/28 layers (x28/{layers}) x127; LM head timed once"),
            "audio_s_per_s": B * CLIP_S / t_audio, "decode_tok_s": B / t_decode_step,
            "seconds": {"mel_per_window": t_mel / n_win, "encode_per_window": t_enc / n_win, "prefill_sampled_layers_1seq": t_pre_layers,
                        "decode_step_sampled_layers_b32": t_dec_layers, "lm_head_b32": t_head, "sample_wall": time.time() - t_all0},
            "estimated_workload_seconds": total,
        }


def cpu_reference(sample: str = "small"):
    ref = CpuReference(layers=4, n_win=1, n_dec=1)
    ref.sample()  # untimed: the first pass through the HF modules / oneDNN primitives is several times slower than the second
    return ref.sample()


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    ref = CpuReference(layers=4, n_win=1, n_dec=2)
    for _ in range(args.warmup):
        ref.sample()
    vals = [ref.sample() for _ in range(args.steps)]
    total = sum(r["estimated_workload_seconds"] for r in vals) / len(vals)
    v = B_PER_GPU * NEW_TOKENS / total
    res = dict(vals[-1], value=v)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "tokens/s", "n_gpus": world, "steps": len(vals), "warmup": args.warmup,
        "ms_per_step": total * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": res.get("dtype", "bf16"),
        "data": "synthetic (seeded noise audio, random-init AF3-7B weights)",
        "config": {"workload": WORKLOAD, "per_gpu_batch": B_PER_GPU, "global_batch": B_PER_GPU, "clip_seconds": CLIP_S, "prompt_len": 780,
                   "new_tokens": NEW_TOKENS, "parallelism": "host CPU, all threads"},
        "cpu_baseline": res,
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip timing HF transformers (eager bf16) on the same GPU")
    ap.add_argument("--no-extras", action="store_true", help="skip the BASELINE config 3 / config 5 / 256-window log-mel measurements")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (driver contract): 32 clips per GPU; strong: a global batch of 32 split over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the generated ids of the last timed step to DIR/generated_ids.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours (the reference arm times CPU samples, it returns no ids)")
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the AF3 hot path has no CPU fallback"}))
        sys.exit(1)
    run_ours(args)


if __name__ == "__main__":
    main()
