"""Host-side logic of the path (no GPU): sharding arithmetic, the token gather over world_size-2 gloo, prompt
helpers, module surface / state_dict key parity with the reference."""
import os
import socket

import numpy as np
import pytest
import torch
from hypothesis import given, settings, strategies as st

from audio_flamingo_b200.processing import expand_audio_spans, expand_audio_tokens, left_pad, split_windows
from audio_flamingo_b200.sharding import gather_tokens, shard_rows


@given(st.integers(0, 300), st.integers(1, 8))
@settings(max_examples=200, deadline=None)
def test_shard_rows_partitions(n, world):
    spans = [shard_rows(n, world, r) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == n
    assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
    sizes = [b - a for a, b in spans]
    assert max(sizes) - min(sizes) <= 1


@given(st.lists(st.integers(1, 20), min_size=1, max_size=40), st.integers(1, 8))
@settings(max_examples=200, deadline=None)
def test_shard_rows_weighted(weights, world):
    n = len(weights)
    spans = [shard_rows(n, world, r, weights) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == n
    assert all(0 <= a <= b <= n for a, b in spans)
    assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
    loads = [sum(weights[a:b]) for a, b in spans]
    assert max(loads) <= sum(weights) / world + max(weights)  # balanced up to one sequence


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, counts):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    L = 7
    local = torch.arange(counts[rank] * L, dtype=torch.int64).view(counts[rank], L) + 1000 * rank
    out = gather_tokens(local, counts)
    exp = torch.cat([torch.arange(c * L, dtype=torch.int64).view(c, L) + 1000 * r for r, c in enumerate(counts)])
    assert torch.equal(out, exp), (rank, out, exp)
    dist.destroy_process_group()


@pytest.mark.parametrize("counts", [[4, 4], [3, 1]])
def test_gather_tokens_gloo_world2(counts):
    import torch.multiprocessing as mp

    mp.spawn(_gather_worker, args=(2, _free_port(), counts), nprocs=2, join=True)


def _gather_ragged_worker(rank, world, port):
    """Rank 0 stopped early on EOS (5 columns, 2 rows), rank 1 ran to the end (9 columns, 3 rows): the collective must see
    equal shapes (ADVICE r01: mismatched L hangs / corrupts NCCL) and the short shard comes back right-padded."""
    import torch.distributed as dist

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rows, L = [(2, 5), (3, 9)][rank]
    local = torch.arange(rows * L, dtype=torch.int64).view(rows, L) + 1000 * (rank + 1)
    out = gather_tokens(local, [2, 3], pad_token_id=77)
    exp0 = torch.full((2, 9), 77, dtype=torch.int64)
    exp0[:, :5] = torch.arange(10, dtype=torch.int64).view(2, 5) + 1000
    exp1 = torch.arange(27, dtype=torch.int64).view(3, 9) + 2000
    assert torch.equal(out, torch.cat([exp0, exp1])), (rank, out)
    dist.destroy_process_group()


def test_gather_tokens_ragged_lengths_gloo_world2():
    import torch.multiprocessing as mp

    mp.spawn(_gather_ragged_worker, args=(2, _free_port()), nprocs=2, join=True)


def test_gather_identity_without_process_group():
    t = torch.arange(6).view(2, 3)
    assert gather_tokens(t) is t


def test_prompt_helpers():
    ids = expand_audio_tokens([5, 9, 7], 9, 4)
    assert ids == [5, 9, 9, 9, 9, 7]
    a, m = left_pad([[1, 2, 3], [4]], pad_id=0)
    assert a.tolist() == [[1, 2, 3], [0, 0, 4]] and m.tolist() == [[1, 1, 1], [0, 0, 1]]
    assert expand_audio_spans([1, 9, 2, 9, 3], 9, [2, 3]) == [1, 9, 9, 2, 9, 9, 9, 3]
    with pytest.raises(ValueError):
        expand_audio_spans([1, 9, 2], 9, [2, 3])
    chunks, per = split_windows([np.zeros(480000 * 25, np.float32)])
    assert per == [20] and len(chunks) == 20  # 600 s cap (AF3P:82,160)


def test_state_dict_keys_match_reference():
    """Same module tree / parameter names / shapes as the reference model (drop-in load_state_dict)."""
    from oracle import af3_oracle as O

    from audio_flamingo_b200 import AudioFlamingo3ForConditionalGeneration

    ref = O.hf_model("tiny", seed=0)
    ours = AudioFlamingo3ForConditionalGeneration(ref.config)
    a = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    b = {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    assert a == b


def test_model_refuses_cpu():
    from oracle import af3_oracle as O

    from audio_flamingo_b200 import AF3Error, AudioFlamingo3Encoder

    enc = AudioFlamingo3Encoder(O.hf_config("tiny").audio_config)
    with pytest.raises(AF3Error, match="no CPU fallback"):
        enc(torch.zeros(1, 128, 3000), torch.ones(1, 3000, dtype=torch.int32))


def test_kv_cache_reset_restores_fresh_state():
    """generate() reuses one AF3KVCache (and the decode graph captured over its buffers) for successive prompts: reset() must
    give back the state of a fresh cache -- zero rows, zero left-padding, position 0 -- in the SAME storages."""
    import torch

    from audio_flamingo_b200.modeling import AF3KVCache

    c = AF3KVCache(n_layers=2, B=3, Hkv=2, Tmax=8, D=4, device="cpu")
    ptrs = (c.k.data_ptr(), c.v.data_ptr(), c.kv_start.data_ptr(), c.pos_dev.data_ptr(), c.ctx_dev.data_ptr())
    c.k.fill_(1.5), c.v.fill_(float("inf"))      # whatever an earlier prompt left behind, finite or not
    c.kv_start.copy_(torch.tensor([0, 2, 5], dtype=torch.int32))
    c.length = 7
    c.pos_dev.fill_(7), c.ctx_dev.fill_(8)
    c.reset()
    assert (c.k.data_ptr(), c.v.data_ptr(), c.kv_start.data_ptr(), c.pos_dev.data_ptr(), c.ctx_dev.data_ptr()) == ptrs
    assert c.length == 0 and c.get_seq_length() == 0
    assert not c.k.any() and not c.v.any() and not c.kv_start.any()
    assert int(c.pos_dev) == 0 and int(c.ctx_dev) == 1


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the driver's reference arm; CPU only) must print exactly one JSON line carrying the contract
    keys, on the same metric / unit / config.workload as our arm."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    import bench

    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["config"]["workload"] == bench.WORKLOAD and d["value"] > 0 and d["steps"] == 2   # exactly --steps samples, no time cap
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["dtype"] in ("bf16", "fp32")
    assert cb["dtype_rule"]["rule"] == "ISA flags" and "cpu_model" in cb["host"] and "sample" in cb
    assert "4/28 decoder layers" in cb["sample"]            # >= 4 sampled layers, fixed thread count (VERDICT r01)


def test_bench_dump_outputs_keeps_every_token_id(tmp_path):
    """`bench.py --dump-outputs DIR` writes the generated ids as float64 (the dump format) with every id of the 152 064-token
    vocabulary unchanged.  That the array is the last timed step's gathered output is wiring in the GPU arm, not checked here."""
    import torch

    import bench

    ids = torch.arange(152064, dtype=torch.int64).view(16, -1)
    bench.dump_outputs(tmp_path / "out", ids)
    a = np.load(tmp_path / "out" / "generated_ids.npy")
    assert a.dtype == np.float64 and a.shape == (16, 9504)
    assert np.array_equal(a.astype(np.int64), ids.numpy())


def test_own_mel_filterbank_is_bit_identical_to_the_reference_table():
    """a2 of SURVEY 8-a: the product builds the 201 x 128 slaney filterbank itself; it must equal, bit for bit, the table the
    reference builds ([O] WFE:95-103 -> AU:453-544).  Only this test imports the reference generator."""
    from transformers.audio_utils import mel_filter_bank

    from audio_flamingo_b200.processing import slaney_mel_filterbank

    ref = mel_filter_bank(num_frequency_bins=201, num_mel_filters=128, min_frequency=0.0, max_frequency=8000.0, sampling_rate=16000,
                          norm="slaney", mel_scale="slaney")
    ours = slaney_mel_filterbank(128, 201, 8000.0)
    assert ours.dtype == ref.dtype == np.float64 and ours.shape == ref.shape == (201, 128)
    assert np.array_equal(ours, ref)


def test_product_does_not_import_reference_package_for_constants():
    import pathlib

    src = (pathlib.Path(__file__).resolve().parent.parent / "audio_flamingo_b200" / "processing.py").read_text()
    assert "transformers" not in src.replace("transformers.audio_utils.mel_filter_bank(201", "")  # the docstring names it once


def test_music_flamingo_timestamps_match_reference_index_arithmetic():
    """Own, sync-free formulation of the frame start times vs the reference's ([O] modular_musicflamingo.py:250-285), on prompts
    with one run spanning two windows, two runs in one row, and a run touching the row end."""
    from transformers.models.musicflamingo.modeling_musicflamingo import MusicFlamingoForConditionalGeneration as HF

    from audio_flamingo_b200.modeling import MusicFlamingoForConditionalGeneration as Ours

    class Cfg:
        audio_token_id = 7
        audio_frame_step = 0.01

    class Holder:
        config = Cfg()
        _mf_frame_step = 0.01

    cases = [
        (torch.tensor([[1, 1, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 2, 2, 2, 2], [3, 7, 7, 7, 4, 7, 7, 7, 7, 7, 5, 5, 5, 5, 5, 5]]), [6, 4, 3, 5]),
        (torch.tensor([[0, 0, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7], [5, 5, 5, 5, 5, 5, 5, 5, 5, 7, 7, 7, 7, 7]]), [5, 5, 2, 5]),
        (torch.tensor([[7, 7, 7, 1]]), [3]),
    ]
    for ids, post in cases:
        post = torch.tensor(post)
        ref = HF._build_audio_timestamps(Holder(), ids, post, 8).float()
        ours = Ours._build_audio_timestamps(Holder(), ids, post, 8)
        assert ours.dtype == torch.float32 and torch.equal(ours, ref), (ids, ours[:, 0], ref[:, 0])


def test_kv_cache_grows_like_dynamic_cache():
    """forward(use_cache=True) reserves room for a continuation and the cache grows on demand (ADVICE r01: a zero reserve made the
    first cached step write past the allocation): capacity buckets, live rows preserved, rows beyond stay zero."""
    from audio_flamingo_b200.modeling import AF3KVCache

    assert [AF3KVCache.bucket(n) for n in (0, 1, 256, 257, 781, 908)] == [256, 256, 256, 512, 1024, 1024]
    c = AF3KVCache(n_layers=2, B=2, Hkv=1, Tmax=256, D=4, device="cpu")
    c.k[:, :, :, :200] = 1.0
    c.v[:, :, :, :200] = 2.0
    c.length = 200
    c.ensure_capacity(256)
    assert c.Tmax == 256
    c.ensure_capacity(257)
    assert c.Tmax == 512 and c.k.shape == (2, 2, 1, 512, 4) and c.length == 200
    assert bool((c.k[:, :, :, :200] == 1).all()) and bool((c.v[:, :, :, :200] == 2).all())
    assert not c.k[:, :, :, 200:].any() and not c.v[:, :, :, 200:].any()


def test_kv_capacity_planning_long_audio():
    """SURVEY 8-f.2: a 10-minute clip = 20 windows = 15 000 audio tokens; AF3-7B costs 57 344 B of KV per token per sequence."""
    from audio_flamingo_b200.sharding import kv_bytes_per_token, plan_kv_capacity, shard_rows

    assert kv_bytes_per_token(28, 4, 128) == 57344
    geo = dict(n_layers=28, n_kv_heads=4, head_dim=128)
    p = plan_kv_capacity([15030] * 4, 128, hbm_free_bytes=140 << 30, activation_bytes_per_token=115_000, **geo)
    assert p["tmax"] == 15360 and p["kv_bytes"] == 4 * 15360 * 57344            # 0.88 GB per sequence, the survey's 0.86 GB + bucket
    assert p["fits"] and p["max_batch"] == (140 << 30) // (15360 * 57344 + 15030 * 115_000)
    chunked = plan_kv_capacity([15030] * 4, 128, hbm_free_bytes=140 << 30, activation_bytes_per_token=115_000, prefill_chunk_size=2048, **geo)
    assert chunked["max_batch"] > p["max_batch"] and chunked["activation_bytes"] == 4 * 2048 * 115_000
    assert not plan_kv_capacity([15030] * 200, 128, hbm_free_bytes=140 << 30, **geo)["fits"]
    # ragged long-audio batch: balance the shards by WINDOW count, all windows of a sequence on one rank (SURVEY 8-e)
    windows = [20, 1, 1, 2, 20, 3, 1, 12]
    spans = [shard_rows(len(windows), 2, r, windows) for r in range(2)]
    loads = [sum(windows[a:b]) for a, b in spans]
    assert spans[0][1] == spans[1][0] and abs(loads[0] - loads[1]) <= max(windows)


def test_packing_leaves_one_copy_of_the_decoder_projections():
    """pack_weights() re-points q/k/v (+ biases) and gate/up at views of the fused matrices the kernels read (VERDICT r01: the
    decoder projections were kept twice, +8.5 GB at AF3-7B).  CPU-checkable: storages are shared, state_dict values unchanged."""
    from oracle import af3_oracle as O

    from audio_flamingo_b200.modeling import Qwen2ForCausalLM

    cfg = O.hf_config("tiny")
    torch.manual_seed(0)
    lm = Qwen2ForCausalLM(cfg.text_config)
    before = {k: v.clone() for k, v in lm.state_dict().items()}
    lm.pack_weights()
    after = lm.state_dict()
    assert all(torch.equal(before[k], after[k]) for k in before)
    l0, (wqkv, bqkv, wgu) = lm.model.layers[0], lm._packed[0]
    for p in (l0.self_attn.q_proj.weight, l0.self_attn.k_proj.weight, l0.self_attn.v_proj.weight):
        assert p.untyped_storage().data_ptr() == wqkv.untyped_storage().data_ptr()
    assert l0.self_attn.v_proj.bias.untyped_storage().data_ptr() == bqkv.untyped_storage().data_ptr()
    assert lm._swiglu_concat and l0.mlp.up_proj.weight.untyped_storage().data_ptr() == wgu.untyped_storage().data_ptr()
    with torch.no_grad():
        l0.mlp.gate_proj.weight[3, 5] = 7.0          # an in-place parameter update is what the kernels read
    assert float(wgu[3, 5]) == 7.0


class _FakeStep:
    """Stands in for the decode runner's step object: counts calls and raises the device-side "all finished" flag at a chosen token."""

    def __init__(self, all_done_at, cap=64):
        self.done_flags = torch.zeros((cap,), dtype=torch.int32)
        self.all_done_at, self.tokens, self.model_steps, self.finished = all_done_at, 0, 0, 0

    def _bookkeeping(self):
        if self.all_done_at is not None and self.tokens >= self.all_done_at:
            self.done_flags[self.tokens] = 1
        self.tokens += 1

    def __call__(self):
        self._bookkeeping()
        self.model_steps += 1
        return torch.zeros((1, 4))

    def finish(self):
        self._bookkeeping()
        self.finished += 1


@pytest.mark.parametrize("max_new,all_done_at,has_eos,expect_tokens,expect_model_steps", [
    (5, None, False, 5, 4),      # no EOS handling: max_new tokens, max_new - 1 cached steps, the last token only gets its bookkeeping
    (1, None, True, 1, 0),       # a single new token never runs a cached step
    (20, 2, True, 3, 8),         # every row finished at token index 2: 3 tokens returned; the flags are read after 8 tokens
    (20, 7, True, 8, 8),         # finished exactly at a check boundary
    (20, 8, True, 9, 16),        # ... one token later: seen at the next check
    (12, 11, True, 12, 11),      # finished on the very last token
    (12, None, True, 12, 11),    # EOS handling on, nobody finishes
])
def test_token_loop_counts_and_eos_cut(max_new, all_done_at, has_eos, expect_tokens, expect_model_steps):
    """modeling._token_loop on a fake step object: how many tokens are returned, how many cached steps are enqueued, that the last
    token goes through finish() (no model step after it), and that the cached-length bookkeeping follows the enqueued steps."""
    import types

    from audio_flamingo_b200.modeling import AudioFlamingo3ForConditionalGeneration as M

    me = types.SimpleNamespace(EOS_CHECK_EVERY=M.EOS_CHECK_EVERY, stage_host_t=None)
    cache = types.SimpleNamespace(length=100)
    step = _FakeStep(all_done_at)
    kept = []
    n = M._token_loop(me, step, cache, kept, has_eos, max_new)
    assert n == expect_tokens
    assert step.model_steps == expect_model_steps and cache.length == 100 + expect_model_steps
    assert step.finished == (1 if step.tokens == max_new else 0)
    assert len(kept) <= n   # logits kept per returned token at most (the caller seeds the list with the prefill logits)


def test_trace_records_slots_and_per_cta_tails():
    """trace.DecodeTrace.graph_launches on a hand-made stamp buffer: slots add up to the step, stream / tail split at the last
    accumulator, per-CTA "accumulator -> exit" statistics (what separates publishing a split-K partial from reducing)."""
    from audio_flamingo_b200 import trace as T

    tr = T.DecodeTrace(torch.device("cpu"), n_slots=4)
    raw = tr.buf.view(4, -1, 4)
    t0 = 1_000_000
    # launch 0 ("rmsnorm", 2 CTAs): entry, dependency resolved, -, exit
    raw[0, 0] = torch.tensor([t0 + 0, t0 + 1000, 0, t0 + 3000])
    raw[0, 1] = torch.tensor([t0 + 100, t0 + 1000, 0, t0 + 3100])
    # launch 1 (few-token GEMM, 3 CTAs): two publish a partial (1.5 us after their accumulator), one reduces (6 us)
    raw[1, 0] = torch.tensor([t0 + 2000, t0 + 4000, t0 + 9000, t0 + 10500])
    raw[1, 1] = torch.tensor([t0 + 2100, t0 + 4100, t0 + 9500, t0 + 11000])
    raw[1, 2] = torch.tensor([t0 + 2200, t0 + 4000, t0 + 10000, t0 + 16000])
    tr.log = [(("rmsnorm", 32, 3584, 0, 0, "decode"), 0, 1), (("gemm", 32, 3584, 3584, 4, "decode"), 1, 2), ("graph_capture", 0, 2)]
    L = tr.graph_launches()
    assert [r["kind"] for r in L] == ["rmsnorm", "gemm 3584x3584"]
    assert L[0]["slot_us"] == pytest.approx(3.1) and L[1]["slot_us"] == pytest.approx(16.0 - 3.1)
    assert sum(r["slot_us"] for r in L) == pytest.approx(16.0)          # the slots add up to the step
    assert L[1]["gap_us"] == pytest.approx(4.0 - 3.1) and L[1]["lead_us"] == pytest.approx(2.0)
    assert L[1]["stream_us"] == pytest.approx(6.0) and L[1]["tail_us"] == pytest.approx(6.0)
    assert L[1]["cta_tail_us"]["min"] == pytest.approx(1.5) and L[1]["cta_tail_us"]["max"] == pytest.approx(6.0)
    assert L[1]["mid_spread_us"] == pytest.approx(1.0)
    agg = T.DecodeTrace.aggregate(L)
    assert agg["gemm 3584x3584"]["n"] == 1


def test_launch_shares_weights_decode_kernels(tmp_path):
    """profiles/launch_shares.py: the few-token GEMMs, decode attention and row-block RMSNorm of the profiled eager decode steps are
    weighted up to the 127 cached steps of the workload, prefill kernels are not (ncu prints template arguments with or without
    the "(int)" casts depending on the version)."""
    import subprocess
    import sys

    hdr = '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"'
    def row(i, name, ns):
        return f'"{i}","1","python","h","{name}","1","7","(1, 1, 1)","(1, 1, 1)","0","10.0","s","gpu__time_duration.sum","ns","{ns}"'
    names = [("void af3::gemm_kernel<256, 1, 4, 0, 8, 4, 0>(CUtensorMap_st, int)", 4_000_000),
             ("void af3::gemm_kernel<32, 2, 6, 1, 8, 4, 0>(CUtensorMap_st, int)", 50_000),
             ("void af3::gemm_kernel<(int)32, (int)1, (int)10, (bool)1, (int)4, (int)4, (bool)0>(CUtensorMap_st, int)", 30_000),
             ("void af3::decode_attn_kernel<8, 3>(CUtensorMap_st, int)", 18_000),
             ("af3::rope_table_kernel(float *)", 2_000)]
    src = tmp_path / "launches.csv"
    src.write_text("==PROF== noise\n" + hdr + "\n" + "\n".join(row(i, n, v) for i, (n, v) in enumerate(names)) + "\n")
    dst = tmp_path / "shares.md"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, os.path.join(root, "profiles", "launch_shares.py"), str(src), str(dst)], check=True, capture_output=True)
    lines = [l for l in dst.read_text().splitlines() if l.startswith("| ") and "`" in l]
    by = {l.split("`")[1]: l.split("|") for l in lines}
    w = 127.0   # one profiled decode step (one rope_table launch) -> x 127
    assert by["void af3::gemm_kernel<32, 2, 6, 1, 8, 4, 0>"][1].strip() == f"{50_000 * w / 1e6:.2f}" and by["void af3::gemm_kernel<32, 2, 6, 1, 8, 4, 0>"][4].strip() == "yes"
    k = [x for x in by if x.startswith("void af3::gemm_kernel<(int)32")][0]
    assert by[k][4].strip() == "yes"
    assert by["void af3::gemm_kernel<256, 1, 4, 0, 8, 4, 0>"][1].strip() == "4.00" and by["void af3::gemm_kernel<256, 1, 4, 0, 8, 4, 0>"][4].strip() == ""
    assert by["void af3::decode_attn_kernel<8, 3>"][4].strip() == "yes"
