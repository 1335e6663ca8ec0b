#!/usr/bin/env python
"""bench.py -- decode tokens/sec of Llama-3.1-8B bf16 on B200 (BASELINE.json metric).

Default workload (SURVEY.md 8d, BASELINE.json configs[1]): random-init weights of the 8B architecture, the
fixed 8-token synthetic prompt, SequenceLength 136 -> one prefill call (S=8) that yields token #1 plus 127
S=1 decode calls = exactly 128 generated tokens (src/inference/inference.go:194-253).  ONE STEP = one such
generation.

  value  = 127*K / (device time of the K*127 decode steps), CUDA events on the launching stream inside
           lnb_decode_run; inputs (weights, KV cache, token) resident in HBM.
  e2e    = the same metric through the reference-facing API with HOST buffers: inference.GenerateTokens
           (use_reference_api=True), i.e. per iteration Transformer.Forward (token ids H2D from pinned memory)
           -> Slice(last row) -> ml.Argmax (4-byte D2H of the result); the [S, vocab] f32 logits stay in HBM
           behind the returned tensor's handle and are only copied when the caller reads them.
  roofline = the dominant kernel (w1|w3 GEMV, 54 % of the step's bytes) timed alone.
  cpu_baseline / parity = the CPU oracle ("port" of the Go path) on this box's host cores: the same 128-token
           generation (bounded: --parity-tokens), timed, and its logits compared with the GPU arm's for EVERY
           generated token, teacher-forced.

ONE accumulation mode per scaling curve: `value` is LNB_ACC_STRICT at every N (bit-identical to the oracle
evaluated in the matching order: the reference's order at N=1, per-shard reference order + rank-order sum of the
shards under tensor parallelism); LNB_ACC_FAST is timed and parity-checked beside it under `other_acc_mode` at
every N.  --acc fast swaps the two roles.

Other BASELINE configs (not driver-run; results are committed under profiles/):
  --config prefill2048   configs[2]: one S=2048 prompt-processing call on the tcgen05 GEMM path (tokens/s)
  --config batch8        configs[4]: 8 concurrent prompts, 128-token decode, one pass over the weights per step

`--impl reference` times only the CPU restatement (the Go toolchain does not exist in this image, so the reference
binary itself cannot run; see DESIGN.md).  Multi-GPU (torchrun, one rank per GPU): tensor parallel, "strong".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PROMPT, SEQ_LEN = 8, 136
N_DECODE = SEQ_LEN - N_PROMPT - 1  # 127 S=1 steps
METRIC = "decode tokens/sec Llama-3.1-8B bf16"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = int(float(self.rows[0][1])) if self.rows else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- the CPU oracle (checker / cpu_baseline only; never on the product path) ---------------------------------
def cpu_oracle_setup(args=None):
    """host copy of the synthetic checkpoint (oracle's generator, the product's published scales) + oracle model"""
    import numpy as np
    import lnb_b200 as L
    from oracle import oracle as O
    args = dict(args or L.synth.LLAMA31_8B)
    t0 = time.time()
    tensors = {}
    for name, shape in L.synth.tensor_shapes(args).items():
        sc, off = L.synth.spec(args, name)
        tensors[name] = O.synth_fill(L.synth.SEED, name, sc, off, int(np.prod(shape))).reshape(shape)
    oargs = dict(dim=args["dim"], n_layers=args["n_layers"], n_heads=args["n_heads"], n_kv_heads=args["n_kv_heads"],
                 head_dim=args["head_dim"], ffn_dim=args["ffn_dim"], vocab=args["vocab_size"], max_seq_len=args["max_seq_len"],
                 norm_eps=args["norm_eps"], rope_theta=args["rope_theta"], use_scaled_rope=args["use_scaled_rope"])
    om = O.OracleModel(oargs, tensors)
    return om, tensors, time.time() - t0, np


def cpu_sample(om, np, n_decode: int, prompt=None, forced=None, tp: int = 1):
    """one bounded sample of the workload on the CPU: prefill the 8-token prompt, then n_decode S=1 steps.
    forced: feed these tokens instead of the oracle's own argmax (teacher forcing); tp > 1: the oracle's emulation of
    the tensor-parallel order (per-shard sums in reference order, shards added in rank order).
    returns (prefill_s, decode_s, tokens, last-row logits per call)"""
    import lnb_b200 as L
    from oracle import oracle as O
    prompt = np.array(prompt if prompt is not None else L.synth.PROMPT_8, np.int32)
    sess = om.new_session(SEQ_LEN)
    toks, logits = [], []
    t0 = time.perf_counter()
    lg = sess.forward(prompt, 0, all_rows=False, tp=tp)
    t_prefill = time.perf_counter() - t0
    nxt = O.argmax_f32(lg[0])
    toks.append(nxt); logits.append(lg[0].copy())
    t0 = time.perf_counter()
    for i in range(n_decode):
        feed = forced[i] if forced is not None else nxt
        lg = sess.forward(np.array([feed], np.int32), len(prompt) + i, all_rows=False, tp=tp)
        nxt = O.argmax_f32(lg[0])
        toks.append(nxt); logits.append(lg[0].copy())
    t_decode = time.perf_counter() - t0
    sess.close()
    return t_prefill, t_decode, toks, logits


def dump_outputs(out_dir, arrays, np):
    """--dump-outputs: write what the timed path returned in its last step as <name>.npy (float64 holds every
    token id exactly), so that two builds run with the same arguments can be compared output for output"""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def bf16_ulps(a, b, np):
    """distance in bf16 ulps between two arrays of bf16-valued float32 (monotone integer map of the bit patterns)"""
    def key(x):
        u = (np.ascontiguousarray(x, np.float32).view(np.uint32) >> 16).astype(np.int64)
        return np.where(u & 0x8000, 0x8000 - u, u)
    return np.abs(key(a) - key(b))


class ParityAcc:
    """running comparison of GPU last-row logits with oracle logits over teacher-forced steps"""

    def __init__(self, np, vs: str, tol: float = 1e-2):
        self.np, self.vs, self.tol = np, vs, tol
        self.maxabs, self.n, self.ndiff, self.agree, self.steps = 0.0, 0, 0, 0, 0
        self.hist = [0, 0, 0, 0, 0]  # |diff| = 0 / <= 2^-8 / <= 2^-7 (one bf16 ulp of a logit in [1,2)) / <= 2^-6 / larger
        self.max_logit = 0.0
        self.first_bad_step = None

    def add(self, g, o, g_tok, o_tok):
        np = self.np
        d = np.abs(g - o)
        m = float(d.max())
        if m > self.tol and self.first_bad_step is None:
            self.first_bad_step = self.steps
        self.maxabs = max(self.maxabs, m)
        self.ndiff += int((d > 0).sum())
        self.n += d.size
        self.hist[0] += int((d == 0).sum()); self.hist[1] += int(((d > 0) & (d <= 2.0 ** -8)).sum())
        self.hist[2] += int(((d > 2.0 ** -8) & (d <= 2.0 ** -7)).sum()); self.hist[3] += int(((d > 2.0 ** -7) & (d <= 2.0 ** -6)).sum())
        self.hist[4] += int((d > 2.0 ** -6).sum())
        self.max_logit = max(self.max_logit, float(np.abs(o).max()))
        self.agree += int(g_tok == o_tok)
        self.steps += 1

    def block(self, acc: str, free_equal=None):
        return {"vs": self.vs, "acc": acc, "tokens_compared": self.steps, "logits_max_abs": round(self.maxabs, 6),
                "logits_differing": self.ndiff, "logits_compared": self.n,
                "abs_diff_histogram": {"0": self.hist[0], "<=2^-8": self.hist[1], "<=2^-7": self.hist[2], "<=2^-6": self.hist[3],
                                       ">2^-6": self.hist[4], "note": "2^-7 = one bf16 ulp of a logit in [1, 2)"},
                "max_abs_logit": round(self.max_logit, 4), "argmax_agree": f"{self.agree}/{self.steps}",
                "free_running_tokens_equal": free_equal, "tolerance": self.tol,
                "within_tolerance": bool(self.maxabs <= self.tol),
                "first_step_over_tolerance": self.first_bad_step}


def run_reference(a):
    """--impl reference: the CPU restatement of the Go path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    t_begin = time.perf_counter()
    om, _, t_setup, np = cpu_oracle_setup()
    print(f"[reference arm] host weights ready in {t_setup:.1f} s, {O.lib().orc_num_threads()} threads", file=sys.stderr, flush=True)
    n_dec = 4
    cpu_sample(om, np, 1)   # CPU steps cost seconds: one warm-up sample regardless of --warmup
    t_dec_total, t_pre_total = 0.0, 0.0
    t0 = time.perf_counter()
    done = 0
    for _ in range(a.steps):
        tp, td, toks, _ = cpu_sample(om, np, n_dec)
        t_dec_total += td
        t_pre_total += tp
        done += 1
        print(f"[reference arm] step {done}/{a.steps}: prefill {tp:.2f} s, {n_dec} decode tokens {td:.2f} s", file=sys.stderr, flush=True)
        if time.perf_counter() - t_begin > 150 and done < a.steps:   # keep the whole arm within a few minutes
            print("[reference arm] time budget reached, stopping early", file=sys.stderr, flush=True)
            break
    a.steps = done
    wall = time.perf_counter() - t0
    val = a.steps * n_dec / t_dec_total
    cores = O.lib().orc_num_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": round(val, 4), "unit": "tokens/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(1000 * wall / a.steps, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "Llama-3.1-8B bf16 random-init, 8-token prompt, seq_len=1 decode over KV cache "
                               "(configs[1]); each step = prefill + %d decode tokens (bounded sample)" % n_dec,
                   "seq_len": SEQ_LEN, "prompt_tokens": N_PROMPT},
        "cpu_baseline": {"value": round(val, 4), "unit": "tokens/s", "cores": cores, "kind": "port",
                         "sample": f"{a.steps} x (prefill 8 + {n_dec} decode steps) of the same workload; C restatement of "
                                   "the Go goroutine path (Go toolchain absent)",
                         "prefill_s": round(t_pre_total / a.steps, 3)},
        "e2e": {"value": round(val, 4), "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"tokens": toks}, np)
    print(json.dumps(line), flush=True)


class Env:
    """process group, model and helpers shared by the configs"""

    def __init__(self, a):
        import numpy as np
        import torch
        import lnb_b200 as L
        self.np, self.torch, self.L, self.a = np, torch, L, a
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != a.gpus:
            raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={self.world}: launch with torchrun --nproc-per-node {a.gpus}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
        torch.cuda.set_device(self.local)
        self.dist, nccl_id = None, None
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if self.rank == 0:
                import ctypes
                raw = ctypes.create_string_buffer(128)
                L._capi.check(L._capi.lib.lnb_nccl_unique_id(raw))
                buf = torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8).cuda()
            dist.broadcast(buf, 0)
            nccl_id = bytes(buf.cpu().numpy().tobytes())
        self.args = dict(L.synth.LLAMA31_8B)
        t0 = time.time()
        self.model = L.model.LoadSyntheticModel(self.args, seed=L.synth.SEED, device=self.local, tp_rank=self.rank,
                                                tp_size=self.world, nccl_id=nccl_id)
        self.t_load = time.time() - t0
        self.tf = self.model.Transformer
        self.peak_hbm, self.peak_tf, self.peak_kind = load_peaks()

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def all_gather_bytes(self, b: bytes):
        torch = self.torch
        t = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        out = [torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [bytes(o.cpu().numpy().tobytes()) for o in out]

    def max_over_ranks(self, *vals):
        if self.dist is None:
            return [float(v) for v in vals]
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def bcast_ints(self, ints, n):
        """rank 0's list of n ints to every rank"""
        if self.dist is None:
            return list(ints)
        t = self.torch.zeros(n, dtype=self.torch.int64, device="cuda")
        if self.rank == 0:
            t = self.torch.tensor(list(ints), dtype=self.torch.int64, device="cuda")
        self.dist.broadcast(t, 0)
        return [int(x) for x in t.cpu()]

    def context(self, acc, collective, max_rows=8, n_seq=1, seq_len=SEQ_LEN):
        L = self.L
        ctx = L.model.InferenceContext(self.tf, L.model.InferenceArgs(seq_len), max_rows=max_rows, acc_mode=acc, n_seq=n_seq)
        self.hook(collective)(ctx)
        return ctx

    def hook(self, collective):
        def h(ctx):
            if self.world > 1 and collective == "p2p":
                ctx.enable_peer_allreduce(self.all_gather_bytes)
                ctx.pre_close_hook = lambda c: self.barrier()   # peers may still be storing into this rank's region
        return h

    def close(self):
        self.model.Free()
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def acc_code(L, name):
    return L._capi.LNB_ACC_FAST if name == "fast" else L._capi.LNB_ACC_STRICT


def timed_generations(env, ctx, prompt, n_gen):
    """n_gen x (prefill + device-resident 127-step decode); returns (tokens of the last one, decode ms, prefill s, graphed)"""
    dec_ms, pre_s, toks, first, graphed = 0.0, 0.0, None, None, False
    for _ in range(n_gen):
        t0 = time.perf_counter()
        first, _ = env.tf.forward_argmax(ctx, prompt, 0)                       # prefill, token #1
        pre_s += time.perf_counter() - t0
        toks, ms, graphed = ctx.decode_run(first, N_PROMPT, N_DECODE, use_graph=True)
        dec_ms += ms
    return [int(first)] + [int(t) for t in toks], dec_ms, pre_s, graphed


def teacher_forced_gpu(env, acc, collective, prompt, forced):
    """last-row logits + greedy token of the GPU arm for the prompt and then every forced token (host-driven Forward)"""
    np = env.np
    ctx = env.context(acc, collective)
    out = []
    nxt, lg = env.tf.forward_argmax(ctx, prompt, 0, want_logits="last")
    out.append((int(nxt), lg[0].copy()))
    for i, t in enumerate(forced):
        nxt, lg = env.tf.forward_argmax(ctx, np.array([t], np.int32), N_PROMPT + i, want_logits="last")
        out.append((int(nxt), lg[0].copy()))
    ctx.close()
    return out


def run_decode(a):
    env = Env(a)
    np, torch, L = env.np, env.torch, env.L
    rank, world = env.rank, env.world
    prompt = np.array(L.synth.PROMPT_8, np.int32)
    head, other_name = a.acc, ("fast" if a.acc == "strict" else "strict")
    collective = a.collective if world > 1 else None
    notes = []

    # ---- device-resident arm (`value`) -----------------------------------------------------
    def device_arm(acc_name, coll, n_warm, n_steps, sample_clocks):
        ctx = env.context(acc_code(L, acc_name), coll)
        gen, _, _, graphed = timed_generations(env, ctx, prompt, n_warm)
        launches0 = ctx.launch_count()
        sampler = ClockSampler(env.local) if sample_clocks else None
        if sampler:
            sampler.start()
        env.barrier()
        wall0 = time.perf_counter()
        gen_k, dec_ms, pre_s, graphed = timed_generations(env, ctx, prompt, n_steps)
        env.barrier()
        wall = time.perf_counter() - wall0
        clocks = sampler.summary() if sampler else None
        launches = ctx.launch_count() - launches0
        assert gen_k == gen, "generation is not reproducible run to run"
        dec_ms, wall = env.max_over_ranks(dec_ms, wall)
        return dict(ctx=ctx, tokens=gen_k, dec_ms=dec_ms, wall=wall, pre_s=pre_s, graphed=graphed, clocks=clocks, launches=launches,
                    value=n_steps * N_DECODE / (dec_ms / 1e3), engine=ctx.uses_engine())

    try:
        arm = device_arm(head, collective, a.warmup, a.steps, True)
    except L._capi.LnbError as e:
        if world > 1 and collective == "p2p" and e.code == -6:   # LNB_ETIMEOUT: a peer never delivered -> NCCL, and say so
            notes.append("peer all-reduce timed out (%s); fell back to --collective nccl" % str(e)[:160])
            collective = "nccl"
            arm = device_arm(head, collective, a.warmup, a.steps, True)
        else:
            raise
    ctx = arm["ctx"]
    gen_tokens, value = arm["tokens"], arm["value"]
    stop_hit = any(t in L.synth.STOP_IDS for t in gen_tokens)

    # ---- roofline of the dominant kernel (w1|w3 GEMV), timed alone ----------------------------
    kinds = {0: "wqkv", 1: "wo", 2: "w13", 3: "w2", 4: "lm_head"}
    kern = {}
    for k, nm in kinds.items():
        ms, nb, nl = ctx.bench_kernel(k, reps=3)
        kern[nm] = {"us": round(ms * 1e3, 2), "bytes": nb, "gbs": round(nb / (ms * 1e-3) / 1e9, 1), "launches": nl}
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("w13_dram_bytes_per_launch"), tj.get("source")
        except Exception:
            traffic = None
    dom = kern["w13"]
    path = ("persistent decode engine (csrc/engine.cuh): one launch per 127-step run; the dominant kernel is timed as an engine "
            "launch that runs only the w1|w3 phases of all 32 layers (RMSNorm prologue incl. the reference-order sum of squares, "
            "weight stream, SwiGLU epilogue), CUDA events around the launch / phases") if arm["engine"] else \
           "kernel chain: one launch per projection, the w1|w3 GEMV launched back to back over all 32 layers' weights"
    roofline = {"bound": "hbm", "kernel": "w1|w3 GEMV (rmsnorm prologue, SwiGLU epilogue), acc=%s" % head, "measured_as": path,
                "achieved": dom["gbs"], "peak": env.peak_hbm, "unit": "GB/s", "frac": round(dom["gbs"] / env.peak_hbm, 4),
                "traffic": traffic, "traffic_source": traffic_src, "peak_kind": env.peak_kind + " (burst copy bandwidth)",
                "bytes_per_launch": dom["bytes"], "us_per_launch": dom["us"]}
    per_gpu_bytes = (13_958_643_712 + 1_050_673_152) / world + 524_288 + 16_384 + 131_072 / world * 72
    step_s = arm["dec_ms"] / 1e3 / (a.steps * N_DECODE)
    roofline_step = {"bytes_per_token_per_gpu": int(per_gpu_bytes), "achieved": round(per_gpu_bytes / step_s / 1e9, 1),
                     "peak": env.peak_hbm, "unit": "GB/s", "frac": round(per_gpu_bytes / step_s / 1e9 / env.peak_hbm, 4),
                     "roofline_tokens_per_s": round(env.peak_hbm * 1e9 / per_gpu_bytes, 1)}
    ctx.close()

    # ---- e2e arm: the reference-facing API with host buffers ----------------------------------
    eng = L.inference.InferenceEngine(env.model, L.model.InferenceArgs(SEQ_LEN), acc_mode=acc_code(L, head))
    eng.context_hook = env.hook(collective)
    saved_stop = env.model.Vocabulary.StopTokenIds
    env.model.Vocabulary.StopTokenIds = () if stop_hit else saved_stop
    for _ in range(2):
        list(eng.GenerateTokens(list(prompt), use_reference_api=True))
    times, e2e_tokens = [], None
    env.barrier()
    for _ in range(a.steps):
        st = []
        e2e_tokens = [t for _, t in eng.GenerateTokens(list(prompt), use_reference_api=True, step_times=st)]
        times.append(st)
    env.barrier()
    dec = sum(sum(st[1:]) for st in times)
    ndec = sum(len(st) - 1 for st in times)
    (dec,) = env.max_over_ranks(dec)
    e2e = {"value": round(ndec / dec, 2), "unit": "tokens/s",
           "h2d_bytes_per_step": (N_PROMPT + N_DECODE) * 4,               # token ids, from the session's pinned buffer
           "d2h_bytes_per_step": (N_DECODE + 1) * 4 * (2 if world > 1 and collective == "p2p" else 1),   # greedy ids (+ peer health word)
           "api": "inference.GenerateTokens -> Transformer.Forward (host token ids in; the f32 logits [S,V] stay in HBM behind "
                  "the returned tensor's handle) -> Slice(last row) -> ml.Argmax (device argmax of the kept row, 4 bytes back)",
           "tokens_equal_device_loop": e2e_tokens == gen_tokens[:len(e2e_tokens)],
           "prefill_ms": round(1e3 * sum(st[0] for st in times) / len(times), 2)}
    # the same loop when the caller reads every logits tensor on the host (all S rows, f32): what round 1 timed
    st = []
    ctx_h = env.context(acc_code(L, head), collective)
    V = env.args["vocab_size"]
    t_all = []
    for rep in range(2):
        t_all = []
        cur = prompt
        pos = 0
        for i in range(1 + N_DECODE):
            t0 = time.perf_counter()
            nxt, lg = env.tf.forward_argmax(ctx_h, cur, pos, want_logits="all")
            t_all.append(time.perf_counter() - t0)
            pos += len(cur)
            cur = np.array([nxt], np.int32)
    ctx_h.close()
    (dec_h,) = env.max_over_ranks(sum(t_all[1:]))
    e2e["host_logits_every_step"] = {"value": round(N_DECODE / dec_h, 2), "unit": "tokens/s",
                                     "d2h_bytes_per_step": (N_PROMPT + N_DECODE) * V * 4 + (N_DECODE + 1) * 4}
    env.model.Vocabulary.StopTokenIds = saved_stop

    # ---- the other collective, same session parameters (TP only) ----------------------------------
    other_coll = None
    if world > 1:
        oc = "nccl" if collective == "p2p" else "p2p"
        try:
            arm2 = device_arm(head, oc, 1, 1, False)
            other_coll = {"collective": oc, "value": round(arm2["value"], 2), "unit": "tokens/s", "acc": head,
                          "tokens_equal": arm2["tokens"] == gen_tokens}
            arm2["ctx"].close()
        except L._capi.LnbError as e:
            other_coll = {"collective": oc, "error": str(e)[:200]}

    # ---- the other accumulation mode, timed the same way (every N) -----------------------------------
    arm3 = device_arm(other_name, collective, 1, max(1, min(a.steps, 2)), False)
    arm3["ctx"].close()
    o_tokens = arm3["tokens"]
    n_same = next((i for i, (x, y) in enumerate(zip(o_tokens, gen_tokens)) if x != y), len(gen_tokens))
    other = {"acc": other_name, "value": round(arm3["value"], 2), "unit": "tokens/s", "tokens_equal_to_headline_arm": n_same,
             "decode_path": "engine" if arm3["engine"] else "kernel chain", "parity": None}

    # ---- cpu_baseline + parity against the oracle, every generated token, teacher-forced --------------------
    cpu, parity = None, None
    if not a.no_cpu:
        n_par = max(1, min(a.parity_tokens, N_DECODE + 1))      # tokens compared (1 prefill + n_par-1 decode steps)
        om = None
        o_toks, o_logits, t_pre, t_dec, t_setup = [0] * n_par, None, 0.0, 0.0, 0.0
        if rank == 0:
            from oracle import oracle as O
            om, _, t_setup, _ = cpu_oracle_setup()
            if world == 1:
                cpu_sample(om, np, 1)                               # warm-up (page the 16 GB of host weights in)
            t_pre, t_dec, o_toks, o_logits = cpu_sample(om, np, n_par - 1)
            if world == 1:
                cpu = {"value": round((n_par - 1) / t_dec, 4), "unit": "tokens/s", "cores": O.lib().orc_num_threads(),
                       "kind": "port", "sample": f"prefill 8 tokens ({t_pre:.2f} s) + {n_par - 1} S=1 decode steps ({t_dec:.1f} s) of the "
                       "same workload; C restatement of the Go goroutine path (Go toolchain absent)", "host_weight_gen_s": round(t_setup, 1)}
        o_toks = env.bcast_ints(o_toks, n_par)
        forced = o_toks[:-1]
        g_head = teacher_forced_gpu(env, acc_code(L, head), collective, prompt, forced)
        g_other = teacher_forced_gpu(env, acc_code(L, other_name), collective, prompt, forced)
        if rank == 0:
            def cmp(g, ref_logits, ref_toks, vs):
                p = ParityAcc(np, vs)
                for (gt, gl), ol, ot in zip(g, ref_logits, ref_toks):
                    p.add(gl, ol, gt, ot)
                return p
            free_eq = lambda toks: next((i for i, (x, y) in enumerate(zip(toks, o_toks)) if x != y), min(len(toks), len(o_toks)))
            vs_ref = "cpu oracle in the REFERENCE order (orc_forward), teacher-forced, every generated token"
            parity = cmp(g_head, o_logits, o_toks, vs_ref).block(head, free_eq(gen_tokens))
            other["parity"] = cmp(g_other, o_logits, o_toks, vs_ref).block(other_name, free_eq(o_tokens))
            if world > 1:
                # the order tensor parallelism imposes (north_star: K split over ranks, one all-reduce after Wo and w2):
                # per-shard sums in reference order, shards added in rank order
                _, _, t_toks, t_logits = cpu_sample(om, np, n_par - 1, forced=forced, tp=world)
                vs_tp = f"cpu oracle in the TENSOR-PARALLEL order (orc_forward_tp, tp={world}), teacher-forced with the same tokens"
                parity = {"vs_tp_order": cmp(g_head, t_logits, t_toks, vs_tp).block(head), "vs_reference_order": parity}
                other["parity"] = {"vs_tp_order": cmp(g_other, t_logits, t_toks, vs_tp).block(other_name),
                                   "vs_reference_order": other["parity"]}
            om.close()
        env.barrier()

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "tokens/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(1e3 * arm["wall"] / a.steps, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "Llama-3.1-8B bf16 random-init, 8-token prompt, 128-token generation, seq_len=1 decode "
                                   "over KV cache (BASELINE.json configs[1]%s)" % ("" if world == 1 else f", tensor-parallel x{world}"),
                       "seq_len": SEQ_LEN, "prompt_tokens": N_PROMPT, "decode_steps_per_generation": N_DECODE,
                       "parallelism": "tp%d" % world, "acc": head, "decode_path": "engine" if arm["engine"] else "kernel chain",
                       "cuda_graph": bool(arm["graphed"]) and not arm["engine"],
                       "collective": collective,
                       "l2": "working set 15 GB per token >> 126 MB L2 (no flush needed)",
                       "stop_id_generated": stop_hit, "notes": notes},
            "decode_ms_per_token": round(arm["dec_ms"] / (a.steps * N_DECODE), 4),
            "prefill_ms": round(1e3 * arm["pre_s"] / a.steps, 3),
            "gpu_launches": int(arm["launches"]),
            "clocks": arm["clocks"],
            "roofline": roofline, "roofline_step": roofline_step, "kernels_alone": kern,
            "e2e": e2e, "other_acc_mode": other, "other_collective": other_coll, "cpu_baseline": cpu, "parity": parity,
            "model_load_s": round(env.t_load, 2),
        }
        if a.dump_outputs:
            # the generation of the last timed step: token #1 from the prefill, then the 127 decoded tokens
            dump_outputs(a.dump_outputs, {"tokens": gen_tokens}, np)
        print(json.dumps(line), flush=True)
    env.close()


def run_prefill(a):
    """BASELINE configs[2]: one Forward of S=2048 prompt tokens on 1xB200 (tcgen05 GEMM path, LNB_ACC_FAST)."""
    env = Env(a)
    np, torch, L = env.np, env.torch, env.L
    if env.world != 1:
        raise SystemExit("--config prefill2048 is a 1-GPU config (BASELINE.json configs[2])")
    S = 2048
    ctx = L.model.InferenceContext(env.tf, L.model.InferenceArgs(S + 1), max_rows=S, acc_mode=L._capi.LNB_ACC_FAST)
    rng = np.random.default_rng(0)
    toks = rng.integers(0, 128000, size=S).astype(np.int32)
    for _ in range(max(3, a.warmup)):
        env.tf.forward_argmax(ctx, toks, 0)
    sampler = ClockSampler(env.local)
    sampler.start()
    env.barrier()
    l0 = ctx.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    t0 = time.perf_counter()
    nxt = None
    for _ in range(a.steps):
        nxt, _ = env.tf.forward_argmax(ctx, toks, 0)      # synchronous: H2D tokens (pinned), forward, D2H token
    wall = time.perf_counter() - t0
    env.barrier()
    clocks = sampler.summary()
    launches = ctx.launch_count() - l0
    per = wall / a.steps
    # algorithmic flops of what this call computes: every projection for all S rows, the LM head for the last row only,
    # causal attention (QK^T and PV over the S(S+1)/2 visible (query, key) pairs of 32 heads x 32 layers, 128 MACs each)
    flops = 2 * 6_979_321_856 * S + 2 * 128256 * 4096 + 32 * 32 * (S * (S + 1) // 2) * 128 * 2 * 2
    parity = None
    if a.parity and env.rank == 0:
        om, _, _, _ = cpu_oracle_setup()
        sess = om.new_session(S + 1)
        t0 = time.perf_counter()
        lo = sess.forward(toks, 0, all_rows=False)
        t_cpu = time.perf_counter() - t0
        _, lg = env.tf.forward_argmax(ctx, toks, 0, want_logits="last")
        p = ParityAcc(np, "cpu oracle (reference order), last row of the S=2048 prefill")
        from oracle import oracle as O
        p.add(lg[0], lo[0], int(np.argmax(lg[0])), O.argmax_f32(lo[0]))
        parity = p.block("fast")
        parity["cpu_prefill_s"] = round(t_cpu, 1)
        sess.close(); om.close()
    line = {"metric": "prefill tokens/sec Llama-3.1-8B bf16 (S=2048)", "value": round(S / per, 1), "unit": "tokens/s", "n_gpus": 1,
            "steps": a.steps, "warmup": max(3, a.warmup), "ms_per_step": round(per * 1e3, 3), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "Llama-3.1-8B bf16 random-init, one prefill call of S=2048 random token ids at position 0, "
                                   "last-row LM head + greedy argmax (BASELINE.json configs[2])", "acc": "fast (tensor-core order)",
                       "l2": "weights 15 GB >> 126 MB L2"},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": round(flops / per / 1e12, 1), "peak": env.peak_tf, "unit": "TFLOP/s",
                         "frac": round(flops / per / 1e12 / env.peak_tf, 4), "traffic": None,
                         "what": "whole call: linears + causal SDPA + last-row LM head, algorithmic flops / wall time (H2D/D2H included)"},
            "e2e": {"value": round(S / per, 1), "unit": "tokens/s", "h2d_bytes_per_step": S * 4, "d2h_bytes_per_step": 4},
            "cpu_baseline": None, "parity": parity, "next_token": int(nxt)}
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"next_token": [nxt]}, np)
    print(json.dumps(line), flush=True)
    ctx.close()
    env.close()


def run_batch8(a):
    """BASELINE configs[4]: 8 concurrent prompts, 128-token decode; weights streamed once per step for all 8 sequences."""
    env = Env(a)
    np, torch, L = env.np, env.torch, env.L
    B = 8
    coll = a.collective if env.world > 1 else None
    prompts = [L.synth.batch_prompt(b) for b in range(B)]

    def generation(ctx, n_steps):
        cur, pos = [], []
        t0 = time.perf_counter()
        for b in range(B):
            ctx.set_active_sequence(b)
            nxt, _ = env.tf.forward_argmax(ctx, np.array(prompts[b], np.int32), 0)
            cur.append(int(nxt)); pos.append(N_PROMPT)
        t_pre = time.perf_counter() - t0
        out = [[c] for c in cur]
        t0 = time.perf_counter()
        for _ in range(n_steps):
            nxt, _ = ctx.forward_batch(cur, pos)       # host loop: token ids + positions H2D, greedy ids D2H, per step
            cur = [int(t) for t in nxt]; pos = [p + 1 for p in pos]
            for b in range(B):
                out[b].append(cur[b])
        return out, time.perf_counter() - t0, t_pre

    res = {}
    for name in (a.acc, "fast" if a.acc == "strict" else "strict"):
        ctx = env.context(acc_code(L, name), coll, max_rows=8, n_seq=B)
        generation(ctx, 8)
        l0 = ctx.launch_count()
        sampler = ClockSampler(env.local) if name == a.acc else None
        if sampler:
            sampler.start()
        env.barrier()
        tot, toks = 0.0, None
        for _ in range(a.steps):
            toks, dt, _ = generation(ctx, N_DECODE)
            tot += dt
        env.barrier()
        (tot,) = env.max_over_ranks(tot)
        res[name] = dict(value=B * N_DECODE * a.steps / tot, ms=1e3 * tot / (a.steps * N_DECODE), toks=toks,
                         clocks=sampler.summary() if sampler else None, launches=ctx.launch_count() - l0)
        ctx.close()
    parity = None
    if not a.no_cpu:
        n_par = max(2, min(a.parity_tokens, 16))
        if env.rank == 0:
            om, _, _, _ = cpu_oracle_setup()
        rows = []
        for b in range(B if env.rank == 0 else 0):
            _, _, ot, _ = cpu_sample(om, np, n_par - 1, prompt=prompts[b], tp=env.world)
            got = res["strict"]["toks"][b][:n_par]
            rows.append({"sequence": b, "oracle_tokens_equal": next((i for i, (x, y) in enumerate(zip(got, ot)) if x != y), n_par), "of": n_par})
        if env.rank == 0:
            om.close()
            parity = {"vs": "cpu oracle, one independent context per sequence, free-running greedy ids (strict arm; "
                            + ("reference order" if env.world == 1 else f"tensor-parallel order tp={env.world}") + ")", "per_sequence": rows}
        env.barrier()
    if env.rank == 0:
        h = res[a.acc]
        per_gpu_bytes = (13_958_643_712 + 1_050_673_152) / env.world
        line = {"metric": "decode tokens/sec Llama-3.1-8B bf16, 8 concurrent sequences (aggregate)", "value": round(h["value"], 1),
                "unit": "tokens/s", "n_gpus": env.world, "steps": a.steps, "warmup": 1, "ms_per_step": round(h["ms"] * N_DECODE, 3),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "Llama-3.1-8B bf16 random-init, 8 concurrent 8-token prompts, 128-token decode each, one pass over "
                                       "the weights per step (BASELINE.json configs[4])", "acc": a.acc, "parallelism": "tp%d" % env.world,
                           "collective": coll, "loop": "host-driven (lnb_forward_batch per step)"},
                "decode_ms_per_step": round(h["ms"], 4), "gpu_launches": int(h["launches"]), "clocks": h["clocks"],
                "roofline": {"bound": "hbm", "achieved": round(per_gpu_bytes / (h["ms"] * 1e-3) / 1e9, 1), "peak": env.peak_hbm, "unit": "GB/s",
                             "frac": round(per_gpu_bytes / (h["ms"] * 1e-3) / 1e9 / env.peak_hbm, 4), "traffic": None,
                             "what": "whole step: weight bytes per GPU / step time"},
                "e2e": {"value": round(h["value"], 1), "unit": "tokens/s", "h2d_bytes_per_step": 64 * N_DECODE, "d2h_bytes_per_step": 32 * N_DECODE},
                "other_acc_mode": {"acc": [k for k in res if k != a.acc][0], "value": round([v for k, v in res.items() if k != a.acc][0]["value"], 1)},
                "cpu_baseline": None, "parity": parity}
        if a.dump_outputs:
            # [8 sequences, 128 tokens] of the headline arm's last timed generation
            dump_outputs(a.dump_outputs, {"tokens": h["toks"]}, np)
        print(json.dumps(line), flush=True)
    env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="lnb", choices=["lnb", "reference"])
    ap.add_argument("--config", default="decode", choices=["decode", "prefill2048", "batch8"])
    ap.add_argument("--acc", default=os.environ.get("LNB_BENCH_ACC", "strict"), choices=["fast", "strict"],
                    help="accumulation order of the headline arm at EVERY N (the other one is timed and parity-checked beside it): "
                         "strict = the reference's k order (per shard under tensor parallelism), fast = interleaved partial sums")
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="tensor-parallel reduction after Wo / w2: fused peer-memory all-reduce over NVLink (default) "
                         "or ncclAllReduce; the other one is timed too and reported under other_collective")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity legs")
    ap.add_argument("--parity-tokens", type=int, default=128, help="generated tokens compared with the oracle (teacher-forced)")
    ap.add_argument("--parity", action="store_true", help="prefill2048: also run the oracle's S=2048 prefill (minutes of CPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the token ids the timed path returned in its last step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference":
        return run_reference(a)
    a.warmup = max(a.warmup, 3)
    if a.config == "prefill2048":
        return run_prefill(a)
    if a.config == "batch8":
        return run_batch8(a)
    return run_decode(a)


if __name__ == "__main__":
    main()
