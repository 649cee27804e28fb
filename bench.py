#!/usr/bin/env python
"""bench.py - decode tokens/s of the paged-attention data plane (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this implementation
  python bench.py --impl reference ...                            # CPU arm: torch-eager oracle port on host cores
  torchrun --nproc-per-node N bench.py --gpus N ...               # N > 1: tensor parallel (heads / FFN columns)
  python bench.py ... --dump-outputs DIR                          # also write the last timed step's outputs as .npy

Workload (BASELINE.json configs[1]): Llama-3-8B shapes, bf16, pure decode, batch 256, every sequence at
seq_len 4096, block_size 16, synthetic seeded weights N(0, 0.02) and a KV cache pre-filled with N(0, 1).
A "step" is one LlamaModel.forward over the batch = one new token per sequence.

One JSON line on stdout (rank 0).  Keys beyond the base contract:
  value      device-resident throughput: K CUDA-graph replays of the decode step, token ids fed back on the device
  e2e        the same step through the public API (LlamaModel.forward with host lists): per step one pinned H2D copy
             of the metadata and one D2H read of the sampled tokens inside the timed region
  roofline   paged-decode kernel: algorithmic bytes / mean CUDA-event duration of its launches over K eager steps
  cpu_baseline  the oracle (CPU torch-eager restatement of the reference forward) on a bounded sample
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "decode_tokens_per_s"
UNIT = "tokens/s"
# --dump-outputs: the full logits of the flagship step (256 x 128256) are 131 MB in fp32; a fixed column sample keeps every
# sequence comparable at 8 MB
DUMP_LOGIT_COLUMNS = 8192


_T0 = time.perf_counter()


def stage(msg: str):
    """Progress line on stderr: where the wall time of a run goes (the JSON line on stdout is the only stdout output)."""
    sys.stderr.write(f"[bench +{time.perf_counter() - _T0:6.1f}s] {msg}\n"); sys.stderr.flush()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--seqlen", type=int, default=4096)
    ap.add_argument("--model", type=str, default="llama3-8b", choices=["llama3-8b", "llama3-70b", "tiny"])
    ap.add_argument("--layers", type=int, default=0, help="override the layer count (debug only; marks the run reduced)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--fused-allreduce", dest="fused_allreduce", action="store_true", default=None,
                    help="TP: force the one-shot peer-memory all-reduce fused with add+RMSNorm (default: automatic, tp 2..4)")
    ap.add_argument("--two-shot-allreduce", dest="fused_allreduce", action="store_const", const="two_shot",
                    help="TP: the row-owner (reduce-scatter + all-gather) variant of the fused exchange (meant for tp 8)")
    ap.add_argument("--nvls-allreduce", dest="fused_allreduce", action="store_const", const="two_shot_nvls",
                    help="TP: two-shot fused exchange with in-switch reduction / broadcast (multimem.ld_reduce / multimem.st)")
    ap.add_argument("--ll-allreduce", dest="fused_allreduce", action="store_const", const="ll",
                    help="TP: barrier-free push exchange (LL protocol) for decode-sized steps, two-shot above 1024 rows")
    ap.add_argument("--ll-nvls-allreduce", dest="fused_allreduce", action="store_const", const="ll_nvls",
                    help="TP: the LL exchange with the normalised rows broadcast by the NVSwitch (multimem.st)")
    ap.add_argument("--nccl-allreduce", dest="fused_allreduce", action="store_false",
                    help="TP: force NCCL all-reduce + separate add/norm kernel")
    ap.add_argument("--shard-lm-head", dest="shard_lm_head", action="store_true", default=None,
                    help="TP: vocabulary-sharded lm_head + (max, argmax) all-gather instead of a replicated lm_head (default: tp >= 4)")
    ap.add_argument("--no-shard-lm-head", dest="shard_lm_head", action="store_false")
    ap.add_argument("--fuse-rotary-store", dest="fuse_rotary_store", action="store_true", default=True,
                    help="decode: rotary + KV store in one launch per layer (default)")
    ap.add_argument("--no-fuse-rotary-store", dest="fuse_rotary_store", action="store_false")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-triton", action="store_true",
                    help="skip timing the unmodified reference's Triton path (baseline/_ref/src) on this GPU (N = 1 only)")
    ap.add_argument("--ref-triton-dtypes", type=str, default="fp16,bf16",
                    help="reference Triton arm: fp16 = the tree as shipped, bf16 = its fp16 literals patched in a temp copy")
    ap.add_argument("--ref-triton-timeout", type=int, default=150,
                    help="seconds per dtype for the reference Triton arm (a cache hit takes ~25 s; a cold JIT needs ~8 min and is cut off)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity check at the benchmarked shape")
    ap.add_argument("--parity-seqs", type=int, default=2, help="sequences re-run through the CPU oracle (tokens + logits)")
    ap.add_argument("--no-live-traffic", action="store_true", help="skip the ncu DRAM-byte measurement of the decode kernel")
    ap.add_argument("--no-prefill", action="store_true")
    ap.add_argument("--cpu-sample-seqs", type=int, default=8)
    ap.add_argument("--profile-range", type=int, default=0,
                    help="profiling aid: run this many eager decode steps inside cudaProfilerStart/Stop and exit "
                         "(use with ncu --profile-from-start off); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed: DIR/tokens.npy (the sampled token "
                         "of every sequence, float64) and DIR/logits_sample.npy (the logits of every sequence at "
                         f"{DUMP_LOGIT_COLUMNS} fixed, seeded vocabulary columns, float32; not written with a sharded lm_head)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def model_dict(name, layers=0):
    from swiftllm_b200.model_config import LLAMA3_8B, LLAMA3_70B
    if name == "llama3-8b":
        d = dict(LLAMA3_8B)
    elif name == "llama3-70b":
        d = dict(LLAMA3_70B)
    else:
        d = dict(model_type="llama", num_hidden_layers=2, num_attention_heads=8, num_key_value_heads=2, hidden_size=1024,
                 vocab_size=1024, max_position_embeddings=8192, intermediate_size=2048, rope_theta=500000.0,
                 rms_norm_eps=1e-5, hidden_act="silu", rope_scaling=None)
    if layers > 0:
        d["num_hidden_layers"] = layers
    return d


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.p = None
        self.idx = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill(); out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_threads() -> int:
    """Threads used by the CPU arm: every host core up to 32 (beyond that the 8-sequence sample's GEMMs stop scaling and
    oversubscription makes the number noisy; the count actually used is reported as `cores`)."""
    return max(1, min(os.cpu_count() or 1, 32))


# --------------------------------------------------------------------------- CPU arm (oracle port)
def cpu_decode_sample(cfg_full: dict, batch: int, seqlen: int, sample_seqs: int, steps: int = 1, warmup: int = 0):
    """Torch-eager CPU forward (oracle/model.py) on a bounded sample of the workload: `sample_seqs` of the `batch`
    sequences at the full sequence length, 1 and 2 of the L layers, fp32 on all host cores.  The per-layer and
    pre/post-layer times are extrapolated linearly to L layers and to the full batch (decode attention and GEMV-like
    GEMMs scale linearly in sequences on a CPU).  Returns tokens/s of the whole job + a description."""
    from oracle.model import OracleLlama, OracleWeights
    torch.set_num_threads(cpu_threads())
    L = cfg_full["num_hidden_layers"]
    bs = 16
    nblk = sample_seqs * ((seqlen + bs - 1) // bs)
    NL = 2
    cfg = dict(cfg_full); cfg["num_hidden_layers"] = NL
    w = OracleWeights.random(cfg, dtype=torch.float32, seed=0, std=0.02)
    m = OracleLlama(cfg, w, block_size=bs, num_blocks=nblk, num_cpu_blocks=0, max_seqs_in_block_table=sample_seqs,
                    max_blocks_per_seq=(seqlen + bs - 1) // bs, attn="fast", dtype=torch.float32)
    g = torch.Generator().manual_seed(1)
    m.k_cache.normal_(generator=g); m.v_cache.normal_(generator=g)
    ids = [[int(t)] for t in torch.randint(0, cfg["vocab_size"], (sample_seqs,), generator=g)]
    sids = list(range(sample_seqs))
    lens = [seqlen] * sample_seqs
    for _ in range(max(1, warmup)):
        m.forward(ids, sids, lens)
    tl, tp = [], []
    for _ in range(max(1, steps)):
        m.forward(ids, sids, lens)
        tl.append(m.last_times["layers"] / NL); tp.append(m.last_times["pre_post"])
    # the least-disturbed of the repetitions: the host cores are shared with whatever else runs on the box (the value moved 2x
    # between boxes in round 1 when a median over 1-3 steps was used)
    t_layer, t_prepost = min(tl), min(tp)
    del m, w
    t_full_sample = L * t_layer + t_prepost
    scale = batch / sample_seqs
    tok_s = batch / (t_full_sample * scale)
    sample = (f"{sample_seqs} of {batch} sequences at seq_len {seqlen}, fp32, {NL} of {L} layers timed "
              f"(best of {max(1, steps)} repetitions: t_layer={t_layer:.3f}s, t_pre+post={t_prepost:.3f}s), extrapolated linearly to {L} layers "
              f"and {batch} sequences")
    return tok_s, sample, t_full_sample * scale


def run_reference(args):
    """`--impl reference`: the reference's CPU-executable restatement (oracle port; the reference itself is Python +
    Triton and cannot run without a GPU/interpreter at this size) timed on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = model_dict(args.model, args.layers)
    t0 = time.perf_counter()
    tok_s, sample, t_step = cpu_decode_sample(cfg, args.batch, args.seqlen, args.cpu_sample_seqs,
                                              steps=max(3, min(args.steps, 6)), warmup=max(1, min(args.warmup, 2)))
    cores = cpu_threads()
    line = {"impl": "reference", "metric": METRIC, "value": tok_s, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32 (CPU oracle port of the bf16 path)", "data": "synthetic",
            "config": workload_config(args, cfg, 1),
            "cpu_baseline": {"value": tok_s, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": tok_s, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    emit(line)


def workload_config(args, cfg, n):
    return {"workload": f"{args.model} pure decode, batch {args.batch}, seq_len {args.seqlen}, block_size 16 "
                        f"(BASELINE.json configs[1])",
            "layers": cfg["num_hidden_layers"], "global_batch": args.batch, "seq_len": args.seqlen,
            "parallelism": f"tp{n}", "l2": "inputs larger than L2 (KV working set and weights >> 126 MB)"}



# --------------------------------------------------------------------------- reference Triton arm (north_star: "next to the
# reference's own Triton path on one B200"): the UNMODIFIED reference under baseline/_ref/src, in its own process
def run_reference_triton(args, dtypes):
    """Runs scripts/ref_triton_bench.py once per dtype BEFORE this process allocates its own 143 GB (both need most of the
    GPU).  Same workload, same public call (LlamaModel.forward: host lists in, host ints out), same step count and
    warm-up, CUDA events around the K steps.  Returns {dtype: json-line-or-error}."""
    out = {}
    script = os.path.join(ROOT, "scripts", "ref_triton_bench.py")
    last = {}
    try:
        last = json.load(open(os.path.join(ROOT, "profiles", "ref_triton_last_measured.json")))
    except Exception:  # noqa: BLE001
        pass
    for dt in dtypes:
        stage(f"reference Triton arm ({dt}) ...")
        env = dict(os.environ, REF_DTYPE=dt, REF_BATCH=str(args.batch), REF_SEQLEN=str(args.seqlen),
                   REF_STEPS=str(args.steps), REF_WARMUP=str(max(args.warmup, 3)), CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0"))
        t0 = time.perf_counter()
        try:
            r = subprocess.run([sys.executable, script], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                               timeout=args.ref_triton_timeout)
            lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
            if r.returncode == 0 and lines:
                d = json.loads(lines[-1])
            else:
                d = {"error": f"rc={r.returncode}: " + (r.stderr.strip().splitlines()[-1][:300] if r.stderr.strip() else "no output")}
        except subprocess.TimeoutExpired:
            # Cold Triton cache: the reference's phase-1 kernel unrolls 128 pages (tl.static_range, paged_attn.py:88) and is
            # compiled three times (cur_layer specialisations); ptxas needs ~8 minutes for that.  scripts/ref_triton_bench.py
            # reads a pre-built cache from baseline/_ref/triton_cache when it travelled with the repo.
            d = {"error": f"timed out after {args.ref_triton_timeout} s (cold Triton JIT cache: ~8 min of ptxas for the reference's "
                          f"128-way unrolled kernel)"}
        except Exception as e:  # noqa: BLE001
            d = {"error": str(e)[:300]}
        if "error" in d and dt in last:
            d["last_measured"] = last[dt]            # committed record of an earlier run on a B200 (profiles/), labelled as such
        d["wall_s"] = round(time.perf_counter() - t0, 1)
        out[dt] = d
    return out


# --------------------------------------------------------------------------- live DRAM traffic of the decode kernel (ncu)
def measure_traffic_live(args, mc, n):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the paged-decode kernel at this run's geometry
    (scripts/paged_attn_traffic.py under ncu, second launch).  Returns (bytes, source) or (None, reason)."""
    import shutil
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "--csv",
           "-k", "regex:paged_attn(_tc)?_kernel", "--launch-skip", "1", "--launch-count", "1",
           sys.executable, os.path.join(ROOT, "scripts", "paged_attn_traffic.py"), "--batch", str(args.batch),
           "--seqlen", str(args.seqlen), "--nq", str(mc.num_q_heads // n), "--nkv", str(mc.num_kv_heads // n),
           "--head-dim", str(mc.head_dim)]
    try:
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=150,
                           env=dict(os.environ, SLLM_PAGED_ATTN_GEN=os.environ.get("SLLM_PAGED_ATTN_GEN", "")))
    except Exception as e:  # noqa: BLE001
        return None, f"ncu failed: {str(e)[:120]}"
    import csv, io
    rows = [l for l in r.stdout.splitlines() if l.startswith('"')]
    vals = {}
    kern = None
    for row in csv.DictReader(io.StringIO("\n".join(rows))):
        try:
            vals[row["Metric Name"]] = float(row["Metric Value"].replace(",", ""))
            kern = row.get("Kernel Name", kern)
        except (KeyError, ValueError):
            continue
    if "dram__bytes_read.sum" not in vals or "dram__bytes_write.sum" not in vals:
        tail = (r.stdout.strip().splitlines() or r.stderr.strip().splitlines() or ["no output"])[-1][:160]
        return None, f"ncu produced no dram__bytes (rc={r.returncode}): {tail}"
    return vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"], \
        (f"live: ncu dram__bytes_read.sum ({vals['dram__bytes_read.sum']:.0f}) + dram__bytes_write.sum ({vals['dram__bytes_write.sum']:.0f}) "
         f"of one launch of {kern} at this geometry (scripts/paged_attn_traffic.py, 1-layer cache, scattered pages)")


# --------------------------------------------------------------------------- parity at the benchmarked shape (oracle = checker)
def parity_check(model, mc, ids, sids, lens, n_rows=8, n_seqs=2, tp_rank=0, tp_size=1, full_getter=None):
    """Outside every timed region.  (a) n_rows sampled (sequence, kv head) GQA groups of the paged-decode kernel's output at
    the benchmarked batch x seq_len, in three layers, against oracle.kernels.paged_attention_exact (fp64) on the pages of
    exactly those sequences (TP: rank 0 checks the heads of its own shard); (b) n_seqs whole sequences re-run through the CPU
    oracle (oracle.model.OracleLlama, fp64 attention, the UNSHARDED weights and this cache's pages - TP: the kv-head shards of
    those sequences are gathered from every rank): sampled token and logits.  Collective under TP (every rank calls it);
    rank 0 raises AssertionError on mismatch and returns the report, the other ranks return None."""
    import torch.distributed as dist
    from oracle import kernels as K
    from oracle.model import OracleLlama, OracleWeights
    from swiftllm_b200.worker.layers import transformer_layer as TL
    B, bs, D, L = len(sids), 16, mc.head_dim, mc.num_layers
    nkv, nq = mc.num_kv_heads // tp_size, mc.num_q_heads // tp_size                # this rank's shard
    g = nq // nkv
    rng = torch.Generator().manual_seed(99)
    layers = sorted({0, L // 2, L - 1})
    picks = [(int(torch.randint(0, B, (1,), generator=rng)), int(torch.randint(0, nkv, (1,), generator=rng))) for _ in range(n_rows)]
    seqs = sorted({int(x) for x in torch.randint(0, B, (max(n_seqs, 1) * 4,), generator=rng).tolist()})[:n_seqs]
    cap = {}
    orig = TL.paged_attention

    def hooked(q, k_cache, v_cache, block_table, mcfg, ecfg, st, cur_layer, o):
        orig(q, k_cache, v_cache, block_table, mcfg, ecfg, st, cur_layer, o)
        if cur_layer in layers:
            cap[cur_layer] = (q.detach().clone(), o.detach().clone())
    was_graph = model.engine_config.use_cuda_graph
    model.engine_config.use_cuda_graph = False
    model.post_layer.keep_logits = True
    TL.paged_attention = hooked
    try:
        toks = model.forward(ids, sids, lens)                   # under TP every rank runs this step (exchanges inside)
    finally:
        TL.paged_attention = orig
        model.engine_config.use_cuda_graph = was_graph
    logits = model.post_layer.last_logits.float().cpu()
    model.post_layer.keep_logits = False; model.post_layer.last_logits = None
    bt = model.gpu_block_manager.block_table

    # kv-head shards of the sampled sequences -> rank 0 (pages of the step just run, all layers)
    kv = {}
    for b in seqs:
        nb = (lens[b] + bs - 1) // bs
        blocks = bt[sids[b], :nb].long()
        kl, vl = model.k_cache[blocks].contiguous(), model.v_cache[blocks].contiguous()      # [nb, L, nkv_local, bs, D]
        if tp_size > 1:
            gk = [torch.empty_like(kl) for _ in range(tp_size)] if tp_rank == 0 else None
            gv = [torch.empty_like(vl) for _ in range(tp_size)] if tp_rank == 0 else None
            dist.gather(kl, gk, dst=0); dist.gather(vl, gv, dst=0)
            if tp_rank == 0:
                kv[b] = (torch.cat([t.cpu() for t in gk], dim=2), torch.cat([t.cpu() for t in gv], dim=2))
        else:
            kv[b] = (kl.cpu(), vl.cpu())
    if tp_rank != 0:
        dist.barrier()                                           # rank 0 is running the CPU oracle
        return None

    def _parity_rank0(res):
        worst = 0.0
        for li in layers:
            q, o = cap[li]
            for (b, h) in picks:
                nb = (lens[b] + bs - 1) // bs
                blocks = bt[sids[b], :nb].long()
                kk = model.k_cache[blocks, li, h].cpu().unsqueeze(1).unsqueeze(1)       # [nb, 1, 1, bs, D]
                vv = model.v_cache[blocks, li, h].cpu().unsqueeze(1).unsqueeze(1)
                qq = q[b, h * g:(h + 1) * g].cpu().unsqueeze(0)                          # [1, g, D]
                ref = K.paged_attention_exact(qq, kk, vv, torch.arange(nb, dtype=torch.int32).unsqueeze(0), [0], [lens[b]],
                                              D ** -0.5, bs, 0)                          # fp64 [1, g*D]
                got = o[b, h * g * D:(h + 1) * g * D].double().cpu()
                err = float((got - ref[0]).abs().max() / ref.abs().max())
                worst = max(worst, err)
                res["attention_rows"].append({"layer": li, "seq": b, "kv_head": h + tp_rank * nkv, "rel_err_vs_fp64": err})
        res["attention_worst_rel_err"] = worst
        res["attention_tol"] = 8e-3
        assert worst <= 8e-3, f"paged attention at the benchmarked shape is off the fp64 oracle by {worst:.3e} (> 8e-3 of max|o|)"

        # (b) whole sequences through the CPU oracle with the unsharded weights and this cache's pages
        if n_seqs > 0:
            NQ, NKV, Fd = mc.num_q_heads, mc.num_kv_heads, mc.ffn_inter_dim
            w = OracleWeights(L)
            if tp_size == 1:
                mw = model.weight
                w.wte, w.lm_head, w.final_norm = mw.wte.cpu(), mw.lm_head.cpu(), mw.final_norm.cpu()
                nqd, nkvd = NQ * D, NKV * D
                for lw, ml in zip(w.layers, mw.layers):
                    qkv = ml.qkv_proj.cpu()
                    lw.q_proj, lw.k_proj, lw.v_proj = qkv[:nqd], qkv[nqd:nqd + nkvd], qkv[nqd + nkvd:]
                    lw.attn_norm, lw.ffn_norm = ml.attn_norm.cpu(), ml.ffn_norm.cpu()
                    lw.o_proj, lw.up_gate_proj, lw.down_proj = ml.o_proj.cpu(), ml.up_gate_proj.cpu(), ml.down_proj.cpu()
            else:
                # the shards came from a deterministic getter: regenerate the FULL tensors (same bits every rank sliced from)
                H, V, dt = mc.hidden_size, mc.vocab_size, model.dtype
                get = lambda key, shape: full_getter(key, shape, dt).to(dt).cpu()
                w.wte, w.lm_head, w.final_norm = get("model.embed_tokens.weight", (V, H)), get("lm_head.weight", (V, H)), get("model.norm.weight", (H,))
                for i, lw in enumerate(w.layers):
                    pre = f"model.layers.{i}."
                    lw.attn_norm, lw.ffn_norm = get(pre + "input_layernorm.weight", (H,)), get(pre + "post_attention_layernorm.weight", (H,))
                    lw.q_proj = get(pre + "self_attn.q_proj.weight", (H, H))
                    lw.k_proj, lw.v_proj = get(pre + "self_attn.k_proj.weight", (NKV * D, H)), get(pre + "self_attn.v_proj.weight", (NKV * D, H))
                    lw.o_proj = get(pre + "self_attn.o_proj.weight", (H, H))
                    lw.up_gate_proj = torch.cat((get(pre + "mlp.up_proj.weight", (Fd, H)), get(pre + "mlp.gate_proj.weight", (Fd, H))), dim=0)
                    lw.down_proj = get(pre + "mlp.down_proj.weight", (H, Fd))
            bps = max((lens[b] + bs - 1) // bs for b in seqs)
            cfgd = dict(hidden_size=mc.hidden_size, num_attention_heads=NQ, num_key_value_heads=NKV, intermediate_size=Fd,
                        num_hidden_layers=L, vocab_size=mc.vocab_size, rms_norm_eps=mc.rms_norm_eps, rope_theta=mc.rope_theta,
                        max_position_embeddings=mc.max_position_embeddings, rope_scaling=mc.rope_scaling)
            def run_oracle(weights, dtype, tables=None):
                orc = OracleLlama(cfgd, weights, block_size=bs, num_blocks=len(seqs) * bps, num_cpu_blocks=0, max_seqs_in_block_table=len(seqs),
                                  max_blocks_per_seq=bps, attn="exact", dtype=dtype)
                if tables is not None:
                    orc.cos, orc.sin = tables                                        # the model's tables (rounded to the storage dtype)
                for j, b in enumerate(seqs):
                    nb = (lens[b] + bs - 1) // bs
                    orc.k_cache[j * bps:j * bps + nb] = kv[b][0].to(dtype)
                    orc.v_cache[j * bps:j * bps + nb] = kv[b][1].to(dtype)
                    orc.gpu_block_manager.allocate_blocks_for_seqs([j], [lens[b]])   # lowest ids first -> j*bps .. j*bps+nb-1
                    assert list(np.asarray(orc.gpu_block_manager.block_table[j][:nb])) == list(range(j * bps, j * bps + nb))
                t = orc.forward([ids[b] for b in seqs], list(range(len(seqs))), [lens[b] for b in seqs])
                return t, orc.last_logits.double(), (orc.cos, orc.sin)

            # (i) the oracle in the storage dtype (the reference's rounding points restated, CPU GEMMs), (ii) the SAME inputs (16-bit
            # weights, 16-bit cache pages, the model's rounded rope tables) evaluated in fp32 without any intermediate rounding (fp64
            # attention): the definition both (i) and the product approximate.  The product must be as close to (ii) as (i) is:
            # over 32 layers, 16-bit storage rounding alone puts two correct implementations ~3-4 % of max|logit| apart.
            ref_toks, ref_logits, tables = run_oracle(w, model.dtype)
            for lw in w.layers:
                for n_ in ("attn_norm", "ffn_norm", "q_proj", "k_proj", "v_proj", "o_proj", "up_gate_proj", "down_proj"):
                    setattr(lw, n_, getattr(lw, n_).float())
            w.wte, w.lm_head, w.final_norm = w.wte.float(), w.lm_head.float(), w.final_norm.float()
            true_toks, true_logits, _ = run_oracle(w, torch.float32, (tables[0].float(), tables[1].float()))
            for j, b in enumerate(seqs):
                tl_, rl, gl = true_logits[j], ref_logits[j], logits[b].double()
                scale = float(tl_.abs().max())
                err_prod, err_orc = float((gl - tl_).abs().max()) / scale, float((rl - tl_).abs().max()) / scale
                top2 = torch.topk(tl_, 2).values
                margin = float(top2[0] - top2[1])
                same = int(toks[b]) == int(true_toks[j])
                res["sequences"].append({"seq": b, "token": int(toks[b]), "exact_arithmetic_token": int(true_toks[j]), "storage_dtype_oracle_token": int(ref_toks[j]),
                                         "token_equal": same, "product_logit_err_vs_exact": err_prod, "storage_dtype_oracle_logit_err_vs_exact": err_orc,
                                         "product_vs_storage_dtype_oracle": float((gl - rl).abs().max()) / scale,
                                         "exact_top1_margin_rel": margin / scale})
                assert err_prod <= max(2.0 * err_orc, 2 ** -6), \
                    f"sequence {b}: product logits are {err_prod:.3e} of max|logit| from exact arithmetic, the storage-dtype oracle only {err_orc:.3e}"
                assert same or margin <= 2 * err_prod * scale, \
                    f"sequence {b}: token {toks[b]} != exact-arithmetic token {true_toks[j]} with top-1 margin {margin / scale:.3e} > 2 x logit error {err_prod:.3e}"
            res["logit_criterion"] = "product error vs exact arithmetic <= max(2 x the storage-dtype oracle's own error, 2^-6)"

    res = {"attention_rows": [], "sequences": [], "tp": tp_size}
    try:
        _parity_rank0(res)
        res["ok"] = True
    except AssertionError as e:
        # TP: the other ranks wait at the barrier below and the line must still be printed (marked invalid); TP = 1: fail the run
        res["ok"], res["error"] = False, str(e)[:400]
        if tp_size == 1:
            raise
    finally:
        if tp_size > 1:
            dist.barrier()
    return res


def dump_outputs(out_dir, tokens, logits):
    """--dump-outputs: `tokens` [B] and, unless None, a fixed column sample of `logits` [B, V] as .npy files under out_dir."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "tokens.npy"), tokens.cpu().numpy().astype(np.float64))
    if logits is not None:
        V = logits.shape[1]
        cols = np.sort(np.random.default_rng(0).choice(V, size=min(V, DUMP_LOGIT_COLUMNS), replace=False))
        sample = logits.index_select(1, torch.from_numpy(cols).to(logits.device)).float().cpu().numpy()
        np.save(os.path.join(out_dir, "logits_sample.npy"), sample)


# --------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch.distributed as dist
    import swiftllm_b200
    from swiftllm_b200 import _lib
    from swiftllm_b200.worker.kernels import paged_attn as pa_mod
    from swiftllm_b200.worker.weight import synthetic_getter

    n = args.gpus
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == n, f"--gpus {n} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {n}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if n > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    ref_triton = None
    if n == 1 and not args.no_ref_triton and args.model == "llama3-8b" and not args.layers and not args.profile_range:
        ref_triton = run_reference_triton(args, [d for d in args.ref_triton_dtypes.split(",") if d in ("fp16", "bf16")])

    stage("building the model shard + KV cache")
    cfg = model_dict(args.model, args.layers)
    mc = swiftllm_b200.LlamaModelConfig(cfg)
    B, S, bs = args.batch, args.seqlen, 16
    blocks_per_seq = (S + bs - 1) // bs
    ec = swiftllm_b200.EngineConfig(model_path="", use_dummy=False, block_size=bs, gpu_mem_utilization=0.97, num_cpu_blocks=0,
                                    max_seqs_in_block_table=B, max_blocks_per_seq=blocks_per_seq + 8, max_batch_size=B,
                                    max_tokens_in_batch=max(B, 16384), dtype="bfloat16", tp_size=n, tp_rank=rank,
                                    use_cuda_graph=not args.no_graph, fused_allreduce=args.fused_allreduce,
                                    shard_lm_head=args.shard_lm_head, fuse_rotary_store=args.fuse_rotary_store)
    model = swiftllm_b200.LlamaModel(ec, mc)
    model.load_weights(synthetic_getter(seed=0, std=0.02, device=dev))
    # set before the decode graph is captured, so that replays leave their logits where post_layer.last_logits points;
    # a sharded lm_head would have to gather the full logits in every step for that
    model.post_layer.keep_logits = bool(args.dump_outputs) and not model.post_layer.sharded
    num_blocks = B * blocks_per_seq + 64
    model.init_kvcache_and_swap(num_blocks)
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    chunk = max(1, num_blocks // 64)
    with torch.inference_mode():
        for s in range(0, num_blocks, chunk):                  # N(0,1) KV so softmax sees realistic, finite data
            model.k_cache[s:s + chunk].normal_(generator=g)
            model.v_cache[s:s + chunk].normal_(generator=g)
    torch.cuda.synchronize()

    gen = torch.Generator().manual_seed(7)
    ids0 = [[int(t)] for t in torch.randint(0, mc.vocab_size, (B,), generator=gen)]
    sids = list(range(B))
    lens = [S] * B

    def barrier():
        if n > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if n > 1:
            t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
        return ms

    # ---- e2e: public API, host lists in, host ints out
    state = {"ids": ids0}

    def step_e2e():
        toks = model.forward(state["ids"], sids, lens)            # H2D metadata + D2H tokens inside
        state["ids"] = [[t] for t in toks]

    for _ in range(max(args.warmup, 3)):
        step_e2e()
    if args.profile_range > 0:
        model.engine_config.use_cuda_graph = False
        model.forward(state["ids"], sids, lens)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for _ in range(args.profile_range):
            model.forward(state["ids"], sids, lens)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    stage("timed region: e2e, then device-resident")
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = _lib.LAUNCH_CALLS
    ms_e2e = timed(step_e2e, args.steps)
    e2e_calls = _lib.LAUNCH_CALLS - launches0

    # ---- value: device-resident (CUDA-graph replay with on-device token feedback), or eager forward_async
    graph = None
    if not args.no_graph and model._graphs:
        graph = next(iter(model._graphs.values()))

    def step_resident():
        if graph is not None:
            graph["meta"][:B].copy_(graph["tokens"].to(torch.int32))     # next step's ids = sampled tokens, on device
            graph["graph"].replay()
        else:
            state["tokens"] = model.forward_async(state["ids"], sids, lens)

    for _ in range(max(args.warmup, 3)):
        step_resident()
    ms_val = timed(step_resident, args.steps)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, graph["tokens"] if graph is not None else state["tokens"], model.post_layer.last_logits)

    stage("roofline pass (events around every decode-attention launch)")
    # ---- roofline of the dominant kernel (paged decode attention): eager steps with events around each launch
    model.engine_config.use_cuda_graph = False
    pa_mod.TIMING_EVENTS = []
    l0 = _lib.LAUNCH_CALLS
    model.forward(state["ids"], sids, lens)
    launches_per_step = _lib.LAUNCH_CALLS - l0
    pa_mod.TIMING_EVENTS = []
    for _ in range(args.steps):
        model.forward_async(state["ids"], sids, lens)
    torch.cuda.synchronize()
    durs = [a.elapsed_time(b) for a, b in pa_mod.TIMING_EVENTS]
    pa_mod.TIMING_EVENTS = None
    model.engine_config.use_cuda_graph = not args.no_graph
    nkv_l, nq_l = mc.num_kv_heads // n, mc.num_q_heads // n
    alg_bytes = sum(lens) * nkv_l * mc.head_dim * 2 * 2 + 2 * B * nq_l * mc.head_dim * 2
    pa_ms = statistics.mean(durs)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    achieved = alg_bytes / (pa_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    if rank == 0 and not args.no_live_traffic:
        stage("live DRAM traffic of the decode kernel (ncu subprocess)")
        torch.cuda.synchronize()
        traffic, traffic_src = measure_traffic_live(args, mc, n)
    tpath = os.path.join(ROOT, "profiles", "paged_attn_traffic.json")
    if traffic is None and os.path.exists(tpath) and n == 1 and args.model == "llama3-8b" and B == 256 and S == 4096 and not args.layers:
        tj = json.load(open(tpath))
        traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], f"committed constant, {tj['source']} (live ncu: {traffic_src})"

    # rank 0 may have spent ~10 s in the ncu subprocess: meet at a HOST-level barrier (NCCL, no watchdog) before the next
    # collective step, so that no rank sits inside a fused exchange kernel (which traps after ~1-2 minutes of spinning) meanwhile
    barrier()

    # ---- parity at the benchmarked shape (outside the timed regions): sampled attention rows + whole sequences vs the oracle
    parity = None
    if not args.no_parity and args.model != "llama3-70b":
        stage("oracle parity at the benchmarked shape")
        parity = parity_check(model, mc, state["ids"], sids, lens, n_rows=8, n_seqs=args.parity_seqs, tp_rank=rank, tp_size=n,
                              full_getter=synthetic_getter(seed=0, std=0.02, device=dev))
    pa_gen = os.environ.get("SLLM_PAGED_ATTN_GEN", "")
    kname = "paged_attn_kernel (gen 1: cp.async + mma.sync)" if pa_gen == "1" else \
        "paged_attn_tc_kernel (gen 2: tcgen05 + TMA, persistent)"

    # ---- optional: prefill tokens/s (secondary metric of BASELINE.json)
    prefill = None
    if not args.no_prefill:
        stage("prefill tokens/s")
        try:
            model.free_seqs_resources(sids)
            Bp, Lp = 4, 4096
            pids = [torch.randint(0, mc.vocab_size, (Lp,), generator=gen).tolist() for _ in range(Bp)]
            psids = list(range(Bp))

            def step_prefill():
                model.forward(pids, psids, [])
                model.free_seqs_resources(psids)
            for _ in range(2):
                step_prefill()
            ms_p = timed(step_prefill, 3)
            prefill = {"value": Bp * Lp / (ms_p / 3 * 1e-3), "unit": UNIT, "batch": Bp, "prompt_len": Lp}
        except Exception as e:  # noqa: BLE001
            prefill = {"error": str(e)[:200]}

    if rank != 0:
        _finish_distributed(model, n)
        return

    cpu = None
    if n == 1 and not args.no_cpu_baseline:
        stage("CPU baseline (oracle port, bounded sample)")
        tok_s, sample, _ = cpu_decode_sample(cfg, B, S, args.cpu_sample_seqs, steps=4, warmup=1)
        cpu = {"value": tok_s, "unit": UNIT, "cores": cpu_threads(), "kind": "port", "sample": sample}

    ms_step = ms_val / args.steps
    line = {
        "metric": METRIC, "value": B / (ms_step * 1e-3), "unit": UNIT, "n_gpus": n, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": workload_config(args, cfg, n),
        "e2e": {"value": B / (ms_e2e / args.steps * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": 3 * B * 4, "d2h_bytes_per_step": B * 8},
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_note": f"{launches_per_step} native (libswiftllm_b200.so) launch calls per decode step "
                             f"({'replayed from a CUDA graph' if graph is not None else 'eager'}); GEMMs/embedding/argmax are library calls on top",
        "roofline": {"kernel": kname, "bound": "hbm", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes, "mean_launch_ms": pa_ms, "launches_timed": len(durs),
                     "how": "CUDA events around every paged_attention launch over K eager decode steps on the launching stream"},
        "tp_exchange": None if n == 1 else (
            ("fused barrier-free push exchange (LL tags in the data): reduce-scatter + add + rmsnorm + all-gather in one kernel"
             + (", all-gather by multimem.st" if model.comm.nvls else "") if getattr(model.comm, "ll", False)
             else "fused NVLS reduce-scatter + add + rmsnorm + all-gather (one kernel, two-shot, multimem)" if getattr(model.comm, "nvls", False)
             else "fused peer-memory reduce-scatter + add + rmsnorm + all-gather (one kernel, two-shot)" if model.comm.two_shot
             else "fused peer-memory all-reduce + add + rmsnorm (one kernel)") if model.comm is not None
            else "ncclAllReduce + fused_add_rmsnorm"),
        "lm_head": "vocabulary-sharded (all-gather of per-rank argmax)" if getattr(model.weight, "lm_head_sharded", False) else "replicated",
        "fuse_rotary_store": bool(args.fuse_rotary_store),
        "clocks": clk,
        "cpu_baseline": cpu,
        "prefill": prefill,
        "parity_at_bench_shape": parity,
    }
    if ref_triton is not None:
        e2e_v = line["e2e"]["value"]
        blk = {"what": "the UNMODIFIED reference (baseline/_ref/src: its Triton kernels + cuBLAS + its own host path) on this GPU, "
                       "same workload, LlamaModel.forward with host lists in / host ints out (comparable to `e2e`), own process, "
                       "run before this arm; dummy weights of the reference (values do not affect timing)",
               "runs": ref_triton}
        for dt, d in ref_triton.items():
            if "value" in d:
                blk[f"e2e_over_reference_{dt}"] = e2e_v / d["value"]
        line["reference_triton"] = blk
    if args.layers:
        line["reduced"] = "layer count overridden: NOT a valid BASELINE measurement"
    if parity is not None and not parity.get("ok", False):
        line["invalid"] = "the oracle parity check at the benchmarked shape FAILED: " + str(parity.get("error"))
    stage("done")
    emit(line)
    _finish_distributed(model, n)


def _finish_distributed(model, n):
    """Leave a multi-rank run without hanging: NCCL kernels captured in live CUDA graphs make
    destroy_process_group() block, so drop the graphs, synchronise, rendezvous once and hard-exit."""
    if n <= 1:
        return
    import torch.distributed as dist
    model._graphs.clear()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush(); sys.stderr.flush()
    os._exit(0)


_REAL_STDOUT = None


def _protect_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, torchrun notices) write to fd 1
    from C code, so point fd 1 at stderr for the whole run and keep a private duplicate for the result line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    _protect_stdout()
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        with torch.inference_mode():
            run_ours(args)


if __name__ == "__main__":
    main()
