"""CPU: host-side logic of the data plane against the oracle."""
import numpy as np
import torch

from oracle import kernels as K
from swiftllm_b200.model_config import LlamaModelConfig, LLAMA3_8B
from swiftllm_b200.worker.model import build_rope_tables, select_seq_block_size
from swiftllm_b200.worker.weight import tp_slice


def test_seq_block_size_matches_reference_heuristic():
    rng = np.random.default_rng(0)
    cases = [[4096] * 256, [11], [131072], [1], [65, 64, 63], [2048] * 7]
    cases += [rng.integers(1, 9000, size=int(rng.integers(1, 300))).tolist() for _ in range(50)]
    for lens in cases:
        for nkv in (1, 2, 8):
            assert select_seq_block_size(nkv, lens, max(lens)) == K.select_seq_block_size(nkv, lens)[0]


def test_rope_tables_match_oracle():
    for cfg in (dict(LLAMA3_8B), dict(LLAMA3_8B, rope_scaling={"factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
                                                                "original_max_position_embeddings": 1024, "rope_type": "llama3"}),
                dict(LLAMA3_8B, rope_scaling=2.0, max_position_embeddings=512)):
        mc = LlamaModelConfig(cfg)
        for dt in (torch.float16, torch.bfloat16):
            cos, sin = build_rope_tables(mc, dt)
            ocos, osin = K.rope_tables(mc.head_dim, mc.rope_theta, mc.max_position_embeddings, mc.rope_scaling, dt)
            assert torch.equal(cos, ocos) and torch.equal(sin, osin)


def test_tp_slices_partition_the_weights():
    w = torch.arange(8 * 6).reshape(8, 6)
    rows = [tp_slice(w, 0, r, 4) for r in range(4)]
    cols = [tp_slice(w, 1, r, 2) for r in range(2)]
    assert torch.equal(torch.cat(rows, 0), w) and torch.equal(torch.cat(cols, 1), w)
    assert tp_slice(w, None, 1, 2) is w


def test_llama3_8b_config_shapes():
    mc = LlamaModelConfig(LLAMA3_8B)
    assert (mc.num_layers, mc.num_q_heads, mc.num_kv_heads, mc.head_dim, mc.ffn_inter_dim) == (32, 32, 8, 128, 14336)
    assert mc.get_kvslot_size(torch.bfloat16) == 128 * 1024        # 128 KiB of KV per token


def test_row_stride_of_contiguous_and_fused_qkv_views():
    from swiftllm_b200 import _lib
    import pytest
    nq, nkv, D, T = 8, 2, 128, 5
    qkv = torch.zeros(T, (nq + 2 * nkv) * D)
    q = qkv[:, : nq * D].unflatten(1, (nq, D)); k = qkv[:, nq * D:(nq + nkv) * D].unflatten(1, (nkv, D))
    assert _lib.row_stride(q) == (nq + 2 * nkv) * D and _lib.row_stride(k) == (nq + 2 * nkv) * D
    assert _lib.row_stride(q[2:]) == (nq + 2 * nkv) * D
    assert _lib.row_stride(torch.zeros(T, nq, D)) == nq * D
    assert _lib.row_stride(torch.zeros(1, nq, D)) >= nq * D
    with pytest.raises(AssertionError):
        _lib.row_stride(torch.zeros(T, D, nq).transpose(1, 2))          # heads not contiguous within a token


def test_fused_qkv_weight_views_share_storage():
    """q_proj / k_proj / v_proj stay available as row views of the fused GEMM operand (weight.py:131-133 semantics)."""
    from swiftllm_b200.worker.weight import LlamaTransformerLayerWeight, synthetic_getter
    cfg = dict(LLAMA3_8B, num_hidden_layers=1, hidden_size=256, num_attention_heads=4, num_key_value_heads=2,
               intermediate_size=512, vocab_size=64)
    mc = LlamaModelConfig(cfg)
    w = LlamaTransformerLayerWeight(0, mc, torch.float32)
    w.load_weights(synthetic_getter(seed=1, device="cpu"), 0, 1, "cpu")
    D = mc.head_dim
    assert w.qkv_proj.shape == ((4 + 2 * 2) * D, 256)
    assert w.q_proj.data_ptr() == w.qkv_proj.data_ptr() and w.q_proj.shape == (4 * D, 256)
    assert torch.equal(torch.cat([w.q_proj, w.k_proj, w.v_proj]), w.qkv_proj)
    assert w.up_gate_proj.shape == (2 * 512, 256)                        # [up ; gate]
    # TP slices of the fused operand are the per-rank q | k | v rows
    w1 = LlamaTransformerLayerWeight(0, mc, torch.float32); w1.load_weights(synthetic_getter(seed=1, device="cpu"), 1, 2, "cpu")
    assert torch.equal(w1.q_proj, w.q_proj[2 * D:]) and torch.equal(w1.k_proj, w.k_proj[D:]) and torch.equal(w1.v_proj, w.v_proj[D:])
    assert torch.equal(w1.o_proj, w.o_proj[:, 2 * D:]) and torch.equal(w1.down_proj, w.down_proj[:, 256:])
    assert torch.equal(w1.up_gate_proj, torch.cat([w.up_gate_proj[256:512], w.up_gate_proj[512 + 256:]]))


def test_bench_line_contract_helpers(tmp_path):
    """bench.py helpers that run without a GPU: the workload description, the thread cap of the CPU arm and the files of
    --dump-outputs (the same column sample every run, within 64 MB at the flagship shape)."""
    import importlib.util, os, types
    spec = importlib.util.spec_from_file_location("bench", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    args = types.SimpleNamespace(model="llama3-8b", batch=256, seqlen=4096)
    cfg = bench.workload_config(args, bench.model_dict("llama3-8b"), 2)
    assert cfg["global_batch"] == 256 and cfg["seq_len"] == 4096 and cfg["parallelism"] == "tp2" and "workload" in cfg
    assert 1 <= bench.cpu_threads() <= 32
    assert bench.METRIC == "decode_tokens_per_s" and bench.UNIT == "tokens/s"
    B, V = 256, 128256
    logits = torch.arange(V, dtype=torch.float32).expand(B, V)             # each logit holds its column index
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), torch.arange(B), logits)
    tok, a, b = (np.load(tmp_path / p) for p in ("a/tokens.npy", "a/logits_sample.npy", "b/logits_sample.npy"))
    assert tok.dtype == np.float64 and np.array_equal(tok, np.arange(B))
    assert a.dtype == np.float32 and a.shape == (B, bench.DUMP_LOGIT_COLUMNS) and np.array_equal(a, b)
    assert (np.diff(a[0]) > 0).all() and (a == a[0]).all()                  # distinct columns, the same for every sequence
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    bench.dump_outputs(str(tmp_path / "c"), torch.arange(B), None)          # sharded lm_head: tokens only
    assert os.listdir(tmp_path / "c") == ["tokens.npy"]


def test_model_config_matches_the_reference_parser(golden):
    """The unmodified reference's LlamaModelConfig (recorded in tests/golden/model_config.npz by oracle/gen_golden.py) and ours
    expose the same values for every attribute the reference defines, over GQA / MHA / scaled-RoPE / legacy-key configs."""
    import json
    cases = json.loads(str(golden("model_config")["cases"]))
    assert len(cases) == 5
    for case in cases:
        ours = LlamaModelConfig(case["config"])
        for name, value in case["attrs"].items():
            assert getattr(ours, name) == value, name
        for key, dt in (("float16", torch.float16), ("bfloat16", torch.bfloat16)):
            assert ours.get_kvslot_size(dt) == case["kvslot_size"][key]
