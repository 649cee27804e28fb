"""
Golden-vector generator.  TEST INFRASTRUCTURE ONLY.

Executes the UNMODIFIED reference (swiftLLM at /root/reference) on CPU -- Triton kernels under
TRITON_INTERPRET=1, `LlamaModel` under the cuda->cpu shim of `oracle/ref_shim.py` -- on seeded
inputs and stores inputs + outputs under `tests/golden/*.npz`.  Run in the build container:

    python oracle/gen_golden.py [name ...] # re-executes itself with `python -O`; names: GENERATORS below

(`-O` strips the reference's `assert weight.device.type == "cuda"`, weight.py:49, which cannot
hold on a CPU-only box; nothing else changes.)  Versions are recorded in each file.
"""
from __future__ import annotations

import json
import os
import sys
import tempfile

if __debug__ and __name__ == "__main__":
    os.execv(sys.executable, [sys.executable, "-O"] + sys.argv)

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def _versions():
    import triton
    return json.dumps({"torch": torch.__version__, "triton": triton.__version__, "numpy": np.__version__,
                       "mode": "TRITON_INTERPRET=1 on CPU", "reference": "interestingLSY/swiftLLM @ /root/reference"})


def _np(t):
    if isinstance(t, torch.Tensor):
        return t.detach().cpu().numpy()
    return np.asarray(t)


def save(name, **arrays):
    arrays = {k: _np(v) for k, v in arrays.items()}
    arrays["_versions"] = np.asarray(_versions())
    path = os.path.join(GOLDEN, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"wrote {path}  ({os.path.getsize(path)/1024:.1f} KiB)")


class _NS:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def gen_elementwise(swiftllm):
    from swiftllm.worker.kernels.rmsnorm import rmsnorm_inplace, fused_add_rmsnorm_inplace
    from swiftllm.worker.kernels.silu_and_mul import silu_and_mul_inplace
    from swiftllm.worker.kernels.rotary_emb import rotary_embedding_inplace

    g = torch.Generator().manual_seed(1234)
    out = {}
    # rmsnorm / fused_add_rmsnorm  (rmsnorm.py:26-37, 67-89)
    T, H = 5, 256
    x = (torch.randn(T, H, generator=g) * 1.5).half()
    r = (torch.randn(T, H, generator=g) * 0.7).half()
    w = (1 + 0.1 * torch.randn(H, generator=g)).half()
    eps = 1e-5
    x1 = x.clone(); rmsnorm_inplace(x1, w, eps)
    x2 = x.clone(); r2 = r.clone(); fused_add_rmsnorm_inplace(x2, r2, w, eps)
    out.update(rms_x=x, rms_r=r, rms_w=w, rms_eps=eps, rms_out=x1, farms_x_out=x2, farms_r_out=r2)
    # silu_and_mul  (silu_and_mul.py:25-34)
    T, F = 3, 512
    xs = (torch.randn(T, 2 * F, generator=g) * 2).half()
    xs_out = xs.clone(); silu_and_mul_inplace(xs_out)
    out.update(silu_x=xs, silu_out=xs_out)
    # rotary  (rotary_emb.py:44-58)
    for tag, (T, nq, nkv, D) in {"a": (6, 8, 2, 64), "b": (3, 8, 2, 128)}.items():
        q = torch.randn(T, nq, D, generator=g).half()
        k = torch.randn(T, nkv, D, generator=g).half()
        ang = torch.rand(T, D // 2, generator=g) * 6.28
        cos, sin = torch.cos(ang).half(), torch.sin(ang).half()
        qo, ko = q.clone(), k.clone()
        rotary_embedding_inplace(qo, ko, _NS(position_cos=cos, position_sin=sin))
        out.update({f"rot{tag}_q": q, f"rot{tag}_k": k, f"rot{tag}_cos": cos, f"rot{tag}_sin": sin,
                    f"rot{tag}_q_out": qo, f"rot{tag}_k_out": ko})
    save("elementwise", **out)


def gen_kvcache_and_paged(swiftllm):
    from swiftllm.worker.kernels.kvcache_mgmt import store_kvcache
    from swiftllm.worker.kernels.paged_attn import paged_attention

    g = torch.Generator().manual_seed(4321)
    # ---- store_kvcache: 2 prefill seqs (20, 5 tokens) + 1 decoding seq (len 18)  (kvcache_mgmt.py:81-122)
    L, nkv, bs, D, nblk = 2, 2, 16, 64, 8
    mc = _NS(num_layers=L, num_kv_heads=nkv, head_dim=D, num_q_heads=4)
    ec = _NS(block_size=bs, max_blocks_per_seq=4)
    block_table = torch.full((5, 4), -1, dtype=torch.int32)
    block_table[3, :2] = torch.tensor([5, 1]); block_table[0, :1] = torch.tensor([7]); block_table[2, :2] = torch.tensor([2, 6])
    seq_ids = torch.tensor([3, 0, 2], dtype=torch.int32)
    st = _NS(seq_ids=seq_ids, num_prefill_seqs=2, num_prefill_tokens=25, num_decoding_seqs=1,
             prefill_seq_start_locs=torch.tensor([0, 20], dtype=torch.int32),
             prefill_seq_lens=torch.tensor([20, 5], dtype=torch.int32), max_prefill_len=20,
             decoding_seq_lens=torch.tensor([18], dtype=torch.int32))
    k = torch.randn(26, nkv, D, generator=g).half()
    v = torch.randn(26, nkv, D, generator=g).half()
    kc = torch.zeros(nblk, L, nkv, bs, D, dtype=torch.float16); vc = torch.zeros_like(kc)
    store_kvcache(k, v, kc, vc, block_table, mc, ec, st, 1)
    save("store_kvcache", k=k, v=v, block_table=block_table, seq_ids=seq_ids, prefill_seq_start_locs=st.prefill_seq_start_locs,
         prefill_seq_lens=st.prefill_seq_lens, decoding_seq_lens=st.decoding_seq_lens, cur_layer=1, block_size=bs,
         k_cache_out=kc, v_cache_out=vc)

    # ---- paged attention, BASELINE config 1: 1 request x 1 KV block  (paged_attn.py:152-222)
    out = {}
    L, nq, nkv, bs, D, nblk = 2, 4, 2, 16, 64, 4
    mc = _NS(num_layers=L, num_kv_heads=nkv, head_dim=D, num_q_heads=nq)
    ec = _NS(block_size=bs, max_blocks_per_seq=4)
    kc = torch.randn(nblk, L, nkv, bs, D, generator=g).half(); vc = torch.randn(nblk, L, nkv, bs, D, generator=g).half()
    bt = torch.full((3, 4), -1, dtype=torch.int32); bt[1, 0] = 2
    q = torch.randn(1, nq, D, generator=g).half()
    st = _NS(num_decoding_seqs=1, num_prefill_seqs=0, seq_ids=torch.tensor([1], dtype=torch.int32),
             decoding_seq_lens=torch.tensor([11], dtype=torch.int32), softmax_scale=D ** -0.5,
             seq_block_size=64, num_seq_blocks=1)
    o = torch.zeros(1, nq * D, dtype=torch.float16)
    paged_attention(q, kc, vc, bt, mc, ec, st, 1, o)
    out.update(c1_q=q, c1_k_cache=kc, c1_v_cache=vc, c1_block_table=bt, c1_seq_ids=st.seq_ids, c1_seq_lens=st.decoding_seq_lens,
               c1_cur_layer=1, c1_block_size=bs, c1_seq_block_size=64, c1_num_seq_blocks=1, c1_scale=st.softmax_scale, c1_o=o)

    # ---- paged attention, multi-block / multi-split / ragged, GQA 4, D=128, shuffled blocks
    L, nq, nkv, bs, D, nblk = 2, 8, 2, 16, 128, 32
    mc = _NS(num_layers=L, num_kv_heads=nkv, head_dim=D, num_q_heads=nq)
    ec = _NS(block_size=bs, max_blocks_per_seq=24)
    kc = torch.randn(nblk, L, nkv, bs, D, generator=g).half(); vc = torch.randn(nblk, L, nkv, bs, D, generator=g).half()
    lens = [300, 17, 64, 1]
    perm = torch.randperm(nblk, generator=g).tolist()
    bt = torch.full((6, 24), -1, dtype=torch.int32)
    sids = [4, 0, 5, 2]
    pos = 0
    for sid, ln in zip(sids, lens):
        n = (ln + bs - 1) // bs
        bt[sid, :n] = torch.tensor(perm[pos:pos + n], dtype=torch.int32); pos += n
    q = torch.randn(len(lens), nq, D, generator=g).half()
    S = 64
    st = _NS(num_decoding_seqs=len(lens), num_prefill_seqs=0, seq_ids=torch.tensor(sids, dtype=torch.int32),
             decoding_seq_lens=torch.tensor(lens, dtype=torch.int32), softmax_scale=D ** -0.5,
             seq_block_size=S, num_seq_blocks=(max(lens) + S - 1) // S)
    o = torch.zeros(len(lens), nq * D, dtype=torch.float16)
    paged_attention(q, kc, vc, bt, mc, ec, st, 0, o)
    out.update(c2_q=q, c2_k_cache=kc, c2_v_cache=vc, c2_block_table=bt, c2_seq_ids=st.seq_ids, c2_seq_lens=st.decoding_seq_lens,
               c2_cur_layer=0, c2_block_size=bs, c2_seq_block_size=S, c2_num_seq_blocks=st.num_seq_blocks,
               c2_scale=st.softmax_scale, c2_o=o)
    save("paged_attention", **out)


def gen_prefill(swiftllm):
    """The reference's own Triton prefill kernel (prefill_attn.py:102-139; unused at its call site but part
    of kernels/)."""
    from swiftllm.worker.kernels.prefill_attn import prefill_attention
    g = torch.Generator().manual_seed(99)
    nq, nkv, D = 4, 2, 64
    lens = [37, 150, 1]
    T = sum(lens)
    q = torch.randn(T, nq, D, generator=g).half(); k = torch.randn(T, nkv, D, generator=g).half(); v = torch.randn(T, nkv, D, generator=g).half()
    starts = [0, 37, 187]
    mc = _NS(num_q_heads=nq, num_kv_heads=nkv, head_dim=D)
    st = _NS(num_prefill_seqs=3, prefill_seq_start_locs=torch.tensor(starts, dtype=torch.int32),
             prefill_seq_lens=torch.tensor(lens, dtype=torch.int32), max_prefill_len=max(lens), softmax_scale=D ** -0.5)
    o = torch.zeros(T, nq, D, dtype=torch.float16)
    with ref_shim.cuda_as_cpu():
        prefill_attention(q, k, v, o, mc, None, st)
    save("prefill_attention", q=q, k=k, v=v, start_locs=st.prefill_seq_start_locs, seq_lens=st.prefill_seq_lens,
         scale=st.softmax_scale, o=o)


def gen_block_mgmt(swiftllm):
    from swiftllm.worker.block_manager import BlockManager
    with ref_shim.cuda_as_cpu():
        bm = BlockManager("GPU", 24, 8, 6, 16)
        bm.block_table.fill_(-1)      # reference leaves it torch.empty; pin the unused entries
        trace = []

        def snap(tag, ret=None):
            trace.append((tag, bm.block_table.clone(), bm.num_seq_allocated_blocks.clone(), bm.is_block_free.clone(),
                          bm.num_free_blocks, None if ret is None else ret.clone()))
        t = lambda x: torch.tensor(x, dtype=torch.int32)
        ops = [
            ("alloc", [3, 1, 6], [20, 1, 40]),
            ("alloc", [3, 1, 6], [33, 16, 41]),      # grow: 3 -> 3 blocks, 1 stays, 6 stays
            ("free", [1]),
            ("alloc", [0, 1], [50, 17]),
            ("gather", [6, 3]),
            ("alloc", [7, 6], [16, 96]),
            ("free", [0, 7, 6, 1]),
        ]
        for op in ops:
            if op[0] == "alloc":
                r = bm.allocate_blocks_for_seqs(t(op[1]), t(op[2])); snap("alloc", r)
            elif op[0] == "free":
                bm.free_blocks_for_seqs(t(op[1])); snap("free")
            else:
                r = bm.gather_allocated_blocks_and_free(t(op[1])); snap("gather", r)
    arrays = {"ops": np.asarray(json.dumps(ops))}
    for i, (tag, bt, nsab, free, nfree, ret) in enumerate(trace):
        arrays[f"s{i}_block_table"] = bt; arrays[f"s{i}_num_seq_allocated_blocks"] = nsab
        arrays[f"s{i}_is_block_free"] = free; arrays[f"s{i}_num_free_blocks"] = nfree
        if ret is not None:
            arrays[f"s{i}_ret"] = ret
    save("block_mgmt", **arrays)


TINY = dict(model_type="llama", num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2, hidden_size=256,
            vocab_size=512, max_position_embeddings=256, intermediate_size=512, rope_theta=10000.0, rms_norm_eps=1e-5,
            hidden_act="silu")


def gen_model(swiftllm):
    """End-to-end: the unmodified `LlamaModel` (model.py) on a tiny random Llama: prefill -> 3 decode steps ->
    mixed batch -> swap out/in -> decode -> free.  Records greedy tokens, logits (input of torch.argmax),
    block-manager state after every call."""
    tmp = tempfile.mkdtemp()
    with open(os.path.join(tmp, "config.json"), "w") as f:
        json.dump(TINY, f)
    ec = swiftllm.EngineConfig(model_path=tmp, use_dummy=True, block_size=16, gpu_mem_utilization=0.9, num_cpu_blocks=8,
                               max_seqs_in_block_table=8, max_blocks_per_seq=8, max_batch_size=4, max_tokens_in_batch=64)
    arrays = {"config": np.asarray(json.dumps(TINY)),
              "engine": np.asarray(json.dumps(dict(block_size=16, num_cpu_blocks=8, max_seqs_in_block_table=8,
                                                   max_blocks_per_seq=8, num_blocks=12)))}
    logits_log = []
    real_argmax = torch.argmax

    def spy_argmax(x, *a, **k):
        logits_log.append(x.detach().clone())
        return real_argmax(x, *a, **k)

    with ref_shim.cuda_as_cpu(), torch.inference_mode():
        torch.manual_seed(7)
        model = swiftllm.LlamaModel(ec)
        model.load_weights()
        # overwrite the +-1e-3 dummy weights (weight.py:215-218) with realistic-scale seeded values
        g = torch.Generator().manual_seed(2024)
        w = model.weight

        def fill(t, std, mean=0.0):
            t.copy_((torch.randn(t.shape, generator=g) * std + mean).to(t.dtype))
        fill(w.wte, 0.5); fill(w.lm_head, 0.05); fill(w.final_norm, 0.05, 1.0)
        arrays.update(wte=w.wte, lm_head=w.lm_head, final_norm=w.final_norm)
        for i, lw in enumerate(w.layers):
            fill(lw.attn_norm, 0.05, 1.0); fill(lw.ffn_norm, 0.05, 1.0)
            for n in ("q_proj", "k_proj", "v_proj", "o_proj", "up_gate_proj", "down_proj"):
                fill(getattr(lw, n), 0.06)
            for n in ("attn_norm", "ffn_norm", "q_proj", "k_proj", "v_proj", "o_proj", "up_gate_proj", "down_proj"):
                arrays[f"l{i}_{n}"] = getattr(lw, n)
        model.init_kvcache_and_swap(12)
        model.gpu_block_manager.block_table.fill_(-1); model.cpu_block_manager.block_table.fill_(-1)

        torch.argmax = spy_argmax
        steps = []

        def snap(tag, toks=None):
            i = len(steps)
            steps.append(tag)
            for name, bm in (("gpu", model.gpu_block_manager), ("cpu", model.cpu_block_manager)):
                arrays[f"t{i}_{name}_block_table"] = bm.block_table.clone()
                arrays[f"t{i}_{name}_nsab"] = bm.num_seq_allocated_blocks.clone()
                arrays[f"t{i}_{name}_free"] = bm.is_block_free.clone()
                arrays[f"t{i}_{name}_nfree"] = bm.num_free_blocks
            if toks is not None:
                arrays[f"t{i}_tokens"] = np.asarray(toks, dtype=np.int64)
                arrays[f"t{i}_logits"] = logits_log[-1]

        rng = np.random.default_rng(5)
        prompts = [rng.integers(0, 512, size=n).tolist() for n in (19, 5)]
        calls = []
        # 1. prefill two sequences (seq ids 2 and 5)
        toks = model.forward(prompts, [2, 5], []); calls.append(dict(op="forward", input_ids=prompts, seq_ids=[2, 5], dec_lens=[])); snap("prefill", toks)
        lens = [len(p) for p in prompts]
        last = toks
        # 2. three decode steps
        for _ in range(3):
            lens = [l + 1 for l in lens]
            ids = [[t] for t in last]
            last = model.forward(ids, [2, 5], lens); calls.append(dict(op="forward", input_ids=ids, seq_ids=[2, 5], dec_lens=lens)); snap("decode", last)
        # 3. mixed batch: one new prefill (seq id 0, 21 tokens) + the two decoding seqs
        newp = rng.integers(0, 512, size=21).tolist()
        lens = [l + 1 for l in lens]
        ids = [newp] + [[t] for t in last]
        toks = model.forward(ids, [0, 2, 5], lens); calls.append(dict(op="forward", input_ids=ids, seq_ids=[0, 2, 5], dec_lens=lens)); snap("mixed", toks)
        last3 = toks
        # 4. swap seq 2 out, then back in, then decode all three
        model.swap_out_seqs([2]); calls.append(dict(op="swap_out", seq_ids=[2])); snap("swap_out")
        model.swap_in_seqs([2]); calls.append(dict(op="swap_in", seq_ids=[2])); snap("swap_in")
        lens3 = [22] + [l + 1 for l in lens]
        ids = [[t] for t in last3]
        toks = model.forward(ids, [0, 2, 5], lens3); calls.append(dict(op="forward", input_ids=ids, seq_ids=[0, 2, 5], dec_lens=lens3)); snap("decode_after_swap", toks)
        # 5. free
        model.free_seqs_resources([0, 5]); calls.append(dict(op="free", seq_ids=[0, 5])); snap("free")
        torch.argmax = real_argmax
        arrays["k_cache_final"] = model.k_cache.clone(); arrays["v_cache_final"] = model.v_cache.clone()
    arrays["calls"] = np.asarray(json.dumps(calls)); arrays["steps"] = np.asarray(json.dumps(steps))
    save("model_tiny", **arrays)


def gen_model_config(swiftllm):
    """The reference's LlamaModelConfig over GQA / MHA / scaled-RoPE / legacy-key configs: every attribute it defines and
    its KV-slot size per dtype, one JSON record per config."""
    from swiftllm.model_config import LlamaModelConfig
    from swiftllm_b200.model_config import LLAMA3_8B
    base = dict(LLAMA3_8B)
    cfgs = [base, dict(base, rope_scaling={"factor": 8.0, "low_freq_factor": 1.0}),
            {k: v for k, v in base.items() if k not in ("num_key_value_heads", "rope_theta", "rope_scaling")},
            dict({k: v for k, v in base.items() if k != "rope_theta"}, rotary_base=12345), dict(base, rope_scaling=2.0)]
    cases = []
    for c in cfgs:
        ref = LlamaModelConfig(c)
        cases.append({"config": c, "attrs": vars(ref),
                      "kvslot_size": {"float16": ref.get_kvslot_size(torch.float16),
                                      "bfloat16": ref.get_kvslot_size(torch.bfloat16)}})
    save("model_config", cases=np.asarray(json.dumps(cases)))


GENERATORS = {"elementwise": gen_elementwise, "kvcache_and_paged": gen_kvcache_and_paged, "prefill": gen_prefill,
              "block_mgmt": gen_block_mgmt, "model": gen_model, "model_config": gen_model_config}


def main(names):
    """`names`: generators to run (all when empty), e.g. `python oracle/gen_golden.py model_config`."""
    os.makedirs(GOLDEN, exist_ok=True)
    swiftllm = ref_shim.import_reference()
    for name in names or GENERATORS:
        GENERATORS[name](swiftllm)


if __name__ == "__main__":
    main(sys.argv[1:])
