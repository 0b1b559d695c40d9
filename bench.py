#!/usr/bin/env python
"""bench.py — sequences/sec for ESM-2 650M bulk embedding extraction at L=1024 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --steps K --warmup W     # the reference algorithm on the host CPU cores

A "step" is one pass of the hot path (embed -> 33 x TransformerLayer -> final LayerNorm -> per-sequence mean, and for
N > 1 one NCCL all-gather of the per-sequence representations) over one synthetic batch:
BASELINE.json configs[1] = esm2_t33_650M_UR50D, 256 sequences of 1024 tokens (<cls> + 1022 residues + <eos>, no
padding, generator seed 1234), seeded random-init weights (checkpoints are unreachable offline).  For N > 1 the same
256-sequence batch is sharded over the ranks (configs[2], strong scaling).

`value`  : device-timed (CUDA events), tokens already resident in HBM, result left in HBM; nothing but the K steps is
           inside the timed region (no per-launch events: those run in a separate profiling pass).
`e2e`    : the same workload through the public host-facing call esm_b200.extract.BulkEmbedder.embed(): tokens start
           in pinned HOST memory, per-token [B,T,E] fp32 and per-sequence mean representations end in pinned HOST
           memory; H2D and D2H copies are inside the timed region.
`kernels` / `roofline`: a separate pass of the same step with every launch bracketed by CUDA events on the launch
           stream (esmb200_profile_enable); the dominant kernel against the measured cuBLAS bf16 peak in
           MEASURED_PEAKS.json.
`configs`: BASELINE.json configs[3] (3B, L=512, contacts) and configs[4] (MSA Transformer, 128 x 512 MSA), N=1 only.
`gpu_eager_baseline`: the UNMODIFIED reference (baseline/_ref, else the oracle port: same ATen ops) in eager fp32 on
           the same GPU — what scripts/extract.py:70-72 gives a user today.
`cpu_baseline`: the reference on the box's host cores, on a bounded sample (N=1, rank 0 only): the unmodified
           reference when baseline/_ref is present (kind "reference"), else the oracle port (kind "port").
Only the baseline legs and --impl reference import oracle/ or baseline/_ref; the product path never does.

--dump-outputs DIR writes what the last timed step returned, the per-sequence mean representations [batch, E], as
DIR/mean_representations.npy (float32; above 64 MB a fixed seeded sample of its rows).  Tokens (seed 1234) and weights
(seed 0, or the local checkpoint) are the same on every run with the same arguments, so two builds can be compared
output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = "esm2_t33_650M_UR50D"
L_LAYERS, E, H, F = 33, 1280, 20, 5120
GLOBAL_BATCH, SEQ_LEN = 256, 1024
TAGS = ["ln1_f16", "gemm_qkv_rope", "attention", "gemm_out_residual", "ln2_f16", "gemm_fc1_gelu", "gemm_fc2_residual",
        "key_bits", "embed", "layernorm_f32", "attention_probs", "convert", "gemm_other", "mean_pool",
        "tied_row_logits", "tied_row_softmax", "tied_row_update"]


def flops_per_seq(T=SEQ_LEN):
    """SURVEY §8(d): per layer 8TE^2 + 4T^2E + 4TEF, plus the LM head (not executed for embedding extraction)."""
    return L_LAYERS * (8 * T * E * E + 4 * T * T * E + 4 * T * E * F)


def make_tokens(B, T, seed=1234):
    g = torch.Generator().manual_seed(seed)
    tok = torch.randint(4, 24, (B, T), generator=g, dtype=torch.int64)
    tok[:, 0] = 0
    tok[:, -1] = 2
    return tok


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"tensor_burst": d["bf16_tflops"], "tensor_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "hbm": d["hbm_gbs"], "source": "MEASURED_PEAKS.json (of measured)"}
    return {"tensor_burst": 1590.0, "tensor_sustained": 1400.0, "hbm": 6650.0, "source": "B200_PROFILING.md (of fallback)"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                r = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.rows.append([c.strip() for c in r.stdout.strip().split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def import_reference():
    """The unmodified reference package from baseline/_ref (offline `pip install --target`, DESIGN.md §6) or None."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "esm")):
        return None
    if ref not in sys.path:
        sys.path.insert(0, ref)
    try:
        import esm  # noqa: F401
        import esm.model.esm2  # noqa: F401
        return esm
    except Exception:
        return None


class RefRunner:
    """The reference's ESM2.forward(tokens, repr_layers=[33]) (esm2.py:77-144) on a device: the real reference when it
    is installed, else the oracle port of the same ATen ops."""

    def __init__(self, state_dict, device):
        self.device = torch.device(device)
        esm = import_reference()
        self.kind = "reference" if esm is not None else "port"
        if esm is not None:
            self.model = esm.model.esm2.ESM2(num_layers=L_LAYERS, embed_dim=E, attention_heads=H, alphabet="ESM-1b")
            self.model.load_state_dict(state_dict, strict=True)
            self.model = self.model.eval().to(self.device)
        else:
            from oracle import esm2_oracle
            self.oracle = esm2_oracle
            self.sd = {k: v.to(self.device) for k, v in state_dict.items()}

    def layer(self, x):
        """one TransformerLayer on x [B,T,E] (thread-count probe)"""
        if self.kind == "reference":
            return self.model.layers[0](x.transpose(0, 1))[0]
        return self.oracle.transformer_layer(x, self.sd, "layers.0.", H, None, False)[0]

    @torch.no_grad()
    def __call__(self, tokens):
        if self.kind == "reference":
            return self.model(tokens, repr_layers=[L_LAYERS])["representations"][L_LAYERS]
        if self.device.type == "cuda":
            # the oracle's rope/position helpers build CPU tensors: run its functional forward on the device copies
            return self.oracle.esm2_forward(self.sd, L_LAYERS, H, tokens, repr_layers=[L_LAYERS])["representations"][L_LAYERS]
        return self.oracle.esm2_forward(self.sd, L_LAYERS, H, tokens, repr_layers=[L_LAYERS])["representations"][L_LAYERS]


def pick_cpu_threads(runner, T=SEQ_LEN):
    """All host threads are available to the CPU arm; PyTorch's intra-op scaling is not monotonic on many-core hosts
    (on the 128-thread B200 host 128 threads run this model SLOWER than 32), so time one TransformerLayer per candidate
    count and keep the fastest — the reference gets its best configuration."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu // 2, ncpu) if 1 <= c <= ncpu})
    x = torch.randn(1, T, E)
    best, best_t = cands[-1], float("inf")
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            runner.layer(x)
            t0 = time.perf_counter()
            runner.layer(x)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
    return best


def cpu_reference_seq_per_s(state_dict, n_seq, steps, warmup, T=SEQ_LEN):
    """The reference on the host cores; returns (seq/s, ms per step, cores, kind)."""
    runner = RefRunner(state_dict, "cpu")
    cores = pick_cpu_threads(runner)
    torch.set_num_threads(cores)
    tok = make_tokens(n_seq, T, seed=1234)
    runner(tok[:1, :128])  # thread-pool warm-up
    for _ in range(warmup):
        runner(tok)
    t0 = time.perf_counter()
    for _ in range(steps):
        runner(tok)
    dt = time.perf_counter() - t0
    return n_seq * steps / dt, dt / steps * 1e3, torch.get_num_threads(), runner.kind


def gpu_eager_reference(state_dict, dev, n_seq=8, reps=2, T=SEQ_LEN):
    """scripts/extract.py:70-72 as users run it: the reference's model.cuda() in eager fp32 (TF32 off), same tokens."""
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        runner = RefRunner(state_dict, dev)
        tok = make_tokens(n_seq, T, seed=1234).to(dev)
        runner(tok)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            out = runner(tok)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        del out, runner
        torch.cuda.empty_cache()
        return {"value": round(n_seq / ms * 1e3, 3), "unit": "sequences/s", "kind": "reference" if import_reference() else "port",
                "dtype": "f32 (TF32 off)", "sample": f"{n_seq} of the {GLOBAL_BATCH} sequences (L={T}) per pass, eager "
                f"PyTorch {torch.__version__} on the same B200, {ms:.1f} ms per pass"}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from esm_b200 import pretrained
    model, _ = pretrained.load_model_and_alphabet(MODEL, allow_random_init=True)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    n_seq = args.ref_seqs
    v, ms, cores, kind = cpu_reference_seq_per_s(sd, n_seq, args.steps, args.warmup)
    impl = "the unmodified reference (baseline/_ref)" if kind == "reference" else "the oracle port of the reference"
    sample = (f"{n_seq} of the {GLOBAL_BATCH} sequences (L={SEQ_LEN}) per step, {impl}, fp32, torch {torch.__version__} "
              f"CPU, {cores} threads (fastest of the counts tried on {os.cpu_count()} logical cores)")
    print(json.dumps({
        "impl": "reference", "metric": "sequences/sec ESM-2 650M L=1024 embedding extract", "value": v,
        "unit": "sequences/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{MODEL} bulk embedding, batch={GLOBAL_BATCH} synthetic L={SEQ_LEN} (configs[1])",
                   "weights": "seeded random init", "sample": sample},
        "cpu_baseline": {"value": v, "unit": "sequences/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def timed(fn, reps, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """arrays {name: tensor} -> path/<name>.npy in float32, together at most DUMP_BYTES: a larger array keeps a fixed
    seeded sample of its rows (leading dimension)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    cap = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        t = t.detach().float()
        row_bytes = t[0].numel() * 4
        if t.numel() * 4 > cap:
            keep = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:cap // row_bytes]
            t = t[keep.sort().values.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def extra_configs(dev, peaks):
    """BASELINE.json configs[3] and configs[4] on this GPU (N=1): seeded random init built on the device."""
    from esm_b200 import pretrained
    out = {}
    # ---- configs[3]: esm2_t36_3B contact-prediction forward, L=512, B=16 (SURVEY §8d)
    B3, T3, L3, E3, H3 = 16, 512, 36, 2560, 40
    model, _ = pretrained.load_model_and_alphabet("esm2_t36_3B_UR50D", allow_random_init=True, device=dev)
    tok = make_tokens(B3, T3, seed=1234).to(dev)
    ms_embed = timed(lambda: model(tok, repr_layers=[L3]), 3, 2)
    ms_contacts = timed(lambda: model(tok, repr_layers=[L3], return_contacts=True), 3, 2)
    fl = L3 * (8 * T3 * E3 * E3 + 4 * T3 * T3 * E3 + 4 * T3 * E3 * 4 * E3)
    att_bytes = B3 * L3 * H3 * T3 * T3 * 4
    out["3B_L512_contacts"] = {
        "workload": "esm2_t36_3B_UR50D forward, need_head_weights/return_contacts, batch=16 synthetic L=512 (configs[3])",
        "value": round(B3 / ms_contacts * 1e3, 2), "unit": "sequences/s", "ms_per_batch": round(ms_contacts, 2),
        "embed_only": {"value": round(B3 / ms_embed * 1e3, 2), "ms_per_batch": round(ms_embed, 2),
                       "model_tflops": round(B3 * fl / ms_embed / 1e9, 1),
                       "roofline": {"bound": "tensor", "achieved": round(B3 * fl / ms_embed / 1e9, 1),
                                    "peak": peaks["tensor_sustained"], "unit": "TFLOP/s",
                                    "frac": round(B3 * fl / ms_embed / 1e9 / peaks["tensor_sustained"], 4)}},
        "attention_stack_bytes": att_bytes,
        "roofline": {"bound": "hbm", "what": "attention maps + contact head on top of the embedding forward: "
                     "4*B*L*H*T^2 bytes written once and read once", "achieved": round(2 * att_bytes / max(ms_contacts - ms_embed, 1e-3) / 1e6, 1),
                     "peak": peaks["hbm"], "unit": "GB/s",
                     "frac": round(2 * att_bytes / max(ms_contacts - ms_embed, 1e-3) / 1e6 / peaks["hbm"], 4)}}
    del model
    torch.cuda.empty_cache()
    # ---- configs[4]: esm_msa1b_t12_100M axial attention forward on a 128 x 512 MSA
    R, C, E4, H4, F4, L4 = 128, 512, 768, 12, 3072, 12
    msa, _ = pretrained.load_msa_model_and_alphabet("esm_msa1b_t12_100M_UR50S", allow_random_init=True, device=dev)
    g = torch.Generator().manual_seed(1234)
    tokens = torch.randint(4, 24, (1, R, C), generator=g)
    tokens[:, :, 0] = 0
    tokens = tokens.to(dev)
    ms_msa = timed(lambda: msa(tokens, repr_layers=[L4]), 5, 2)
    M = R * C
    fl4 = L4 * (8 * 2 * M * E4 * E4 + 2 * 2 * M * E4 * F4 + 2 * 2 * H4 * C * C * R * 64 + 4 * C * H4 * R * R * 64)
    out["msa_128x512"] = {
        "workload": "esm_msa1b_t12_100M_UR50S forward (row + column axial attention), synthetic MSA 128 x 512 (configs[4])",
        "value": round(1e3 / ms_msa, 2), "unit": "MSAs/s", "ms_per_msa": round(ms_msa, 3),
        "model_tflops": round(fl4 / ms_msa / 1e9, 1),
        "roofline": {"bound": "tensor", "achieved": round(fl4 / ms_msa / 1e9, 1), "peak": peaks["tensor_burst"],
                     "unit": "TFLOP/s", "frac": round(fl4 / ms_msa / 1e9 / peaks["tensor_burst"], 4),
                     "peak_source": "burst (a 20 ms forward does not reach the sustained power state)"}}
    del msa
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=GLOBAL_BATCH)
    ap.add_argument("--micro-batch", type=int, default=128)
    ap.add_argument("--ref-seqs", type=int, default=2, help="sequences per step of the CPU reference arm")
    ap.add_argument("--cpu-baseline-seqs", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip configs[3]/[4] and the GPU eager baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries ONE JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION and above (WARN
        # included), so nothing is set here; a caller who exports NCCL_DEBUG=INFO gets NCCL's lines, then the JSON line last
        dist.init_process_group("nccl", device_id=dev)

    from esm_b200 import _lib, pretrained
    from esm_b200.extract import BulkEmbedder, all_gather_rows, mean_pool, residue_lengths, shard_range
    lib = _lib.load()

    model, alphabet = pretrained.load_model_and_alphabet(MODEL, allow_random_init=True)
    model = model.to(dev)
    tokens_host = make_tokens(args.batch, SEQ_LEN, seed=1234)
    s, e = shard_range(args.batch, world, rank)
    local_host = tokens_host[s:e].contiguous().pin_memory()
    local_dev = local_host.to(dev)
    n_local = e - s

    def step_device():
        out = model(local_dev, repr_layers=[L_LAYERS])["representations"][L_LAYERS]
        m = mean_pool(out, residue_lengths(local_dev, alphabet))
        if world > 1:
            m = all_gather_rows(m, args.batch)
        return m

    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)

    # ---- value: W warm-up steps, then exactly K steps between two events; nothing else in the timed region
    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    launches0 = lib.esmb200_launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        mean = step_device()
    ev1.record()
    torch.cuda.synchronize()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = lib.esmb200_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"mean_representations": mean})

    # ---- per-kernel pass: the same step with every launch bracketed by events (breaks PDL overlap, so it is separate)
    prof_steps = min(2, args.steps)
    max_rec = 260 * prof_steps
    _lib.check(lib.esmb200_profile_enable(max_rec))
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(prof_steps):
        step_device()
    p1.record()
    torch.cuda.synchronize()
    ms_prof = p0.elapsed_time(p1)
    tags = (ctypes.c_int32 * max_rec)()
    mss = (ctypes.c_float * max_rec)()
    nrec = lib.esmb200_profile_read(tags, mss, max_rec)
    _lib.check(lib.esmb200_profile_enable(0))

    # ---- e2e: host tokens -> host representations through the public API
    emb = BulkEmbedder(model, include=("mean", "per_tok"), micro_batch=args.micro_batch)
    for _ in range(2):
        emb.embed(local_host)
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = emb.embed(local_host)
        if world > 1:
            all_gather_rows(res["mean"].to(dev, non_blocking=True), args.batch)
    e1.record()
    torch.cuda.synchronize()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    sampler.stop_flag.set()
    sampler.join(timeout=2)

    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = float(t[0]), float(t[1])
    ms_step = ms_total / args.steps
    value = args.batch / (ms_step / 1e3)
    e2e_value = args.batch / (ms_e2e / args.steps / 1e3)

    # ---- per-kernel table + roofline of the dominant kernel
    per = {}
    for i in range(nrec):
        d = per.setdefault(TAGS[tags[i]], [0, 0.0])
        d[0] += 1
        d[1] += mss[i]
    M = n_local * SEQ_LEN
    work = {  # algorithmic FLOPs (tensor) or bytes (hbm) per launch, SURVEY §8(d)
        "gemm_qkv_rope": ("tensor", 2.0 * M * E * 3 * E), "gemm_out_residual": ("tensor", 2.0 * M * E * E),
        "gemm_fc1_gelu": ("tensor", 2.0 * M * E * F), "gemm_fc2_residual": ("tensor", 2.0 * M * F * E),
        "attention": ("tensor", 4.0 * n_local * H * SEQ_LEN * SEQ_LEN * 64),
        "ln1_f16": ("hbm", 6.0 * M * E), "ln2_f16": ("hbm", 6.0 * M * E), "layernorm_f32": ("hbm", 8.0 * M * E),
        "mean_pool": ("hbm", 4.0 * M * E), "embed": ("hbm", 4.0 * M * E),
    }
    peaks = measured_peaks()
    kernels = {}
    for name, (cnt, tot) in per.items():
        avg = tot / cnt
        row = {"launches": cnt, "avg_ms": round(avg, 4), "share": round(tot / ms_prof, 4)}
        if name in work:
            kind, amount = work[name]
            if kind == "tensor":
                row["TFLOP/s"] = round(amount / avg / 1e9, 1)
                row["frac_of_peak"] = round(amount / avg / 1e9 / peaks["tensor_sustained"], 3)
            else:
                row["GB/s"] = round(amount / avg / 1e6, 1)
                row["frac_of_peak"] = round(amount / avg / 1e6 / peaks["hbm"], 3)
        kernels[name] = row
    dom = max(per.items(), key=lambda kv: kv[1][1])[0] if per else None
    roofline = None
    if dom and dom in work:
        kind, amount = work[dom]
        avg = per[dom][1] / per[dom][0]
        if kind == "tensor":
            ach, peak, unit = amount / avg / 1e9, peaks["tensor_sustained"], "TFLOP/s"
        else:
            ach, peak, unit = amount / avg / 1e6, peaks["hbm"], "GB/s"
        traffic, traffic_src = None, None
        for fname in ("r02_traffic.json", "r01_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", fname)
            if os.path.exists(tpath):  # DRAM bytes per token of this kernel from a committed ncu --set full capture
                bpt = json.load(open(tpath))["bytes_per_token"].get(dom)
                if bpt:
                    traffic = round(bpt * M)
                    traffic_src = f"static: profiles/{fname} (ncu --set full dram__bytes of this kernel per token x {M} tokens)"
                    break
        roofline = {"kernel": dom, "bound": kind, "achieved": round(ach, 1), "peak": peak, "unit": unit,
                    "frac": round(ach / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["source"] + (", sustained (kernel timed inside a long step)" if kind == "tensor" else ""),
                    "avg_launch_ms": round(avg, 4), "algorithmic_per_launch": amount}

    out = {
        "metric": "sequences/sec ESM-2 650M L=1024 embedding extract", "value": round(value, 2),
        "unit": "sequences/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f16 operands, f32 accumulate/residual/LayerNorm/softmax", "data": "synthetic",
        "config": {"workload": f"{MODEL} bulk embedding, batch={args.batch} synthetic L={SEQ_LEN} (BASELINE.json "
                               f"configs[{1 if world == 1 else 2}])",
                   "global_batch": args.batch, "seq_len": SEQ_LEN, "per_gpu_batch": n_local,
                   "parallelism": f"dp{world} (sequence sharding, one all-gather of [B,E] means)",
                   "weights": "seeded random init (no checkpoints offline)", "repr_layers": [L_LAYERS],
                   "l2": "activations per step (>1 GB/GPU) exceed the 126 MB L2; no explicit flush"},
        "model_tflops": round(value * flops_per_seq() / 1e12, 1),
        "tensor_frac_whole_step": round(value * flops_per_seq() / 1e12 / world / peaks["tensor_sustained"], 4),
        "e2e": {"value": round(e2e_value, 2), "unit": "sequences/s", "h2d_bytes_per_step": emb.h2d_bytes * world,
                "d2h_bytes_per_step": emb.d2h_bytes * world, "ms_per_step": round(ms_e2e / args.steps, 3),
                "api": "esm_b200.extract.BulkEmbedder.embed (mean + per_tok to pinned host memory)"},
        "gpu_launches": int(launches), "kernels": kernels,
        "kernels_note": f"separate pass of {prof_steps} step(s) with per-launch CUDA events ({ms_prof / prof_steps:.1f} ms per "
                        f"step; the timed value above has no events inside)",
        "roofline": roofline, "clocks": sampler.summary(),
    }
    if rank == 0 and world == 1 and not args.no_extra:
        del emb, res
        sd = {k: v.detach() for k, v in model.state_dict().items()}
        try:
            out["gpu_eager_baseline"] = gpu_eager_reference({k: v.clone() for k, v in sd.items()}, dev)
        except Exception as ex:  # a baseline leg must never take the contract line down
            out["gpu_eager_baseline"] = {"unavailable": repr(ex)[:200]}
        model_cpu_sd = {k: v.cpu() for k, v in sd.items()}
        del model, sd
        torch.cuda.empty_cache()
        try:
            out["configs"] = extra_configs(dev, peaks)
        except Exception as ex:
            out["configs"] = {"unavailable": repr(ex)[:200]}
    else:
        model_cpu_sd = {k: v.detach().cpu() for k, v in model.state_dict().items()} if (rank == 0 and world == 1) else None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = args.cpu_baseline_seqs
        v, ms, cores, kind = cpu_reference_seq_per_s(model_cpu_sd, n, steps=1, warmup=0)
        impl = "the unmodified reference (baseline/_ref)" if kind == "reference" else "fp32 oracle port of the reference"
        out["cpu_baseline"] = {"value": round(v, 4), "unit": "sequences/s", "cores": cores, "kind": kind,
                               "sample": f"one pass over {n} of the {args.batch} sequences (L={SEQ_LEN}), {impl} on the "
                                         f"host CPU, fp32, {ms / 1e3:.1f} s"}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
