#!/usr/bin/env python
"""bench.py -- MemVul batch-inference hot path on B200 (BASELINE.json metric: issue-reports/sec).

    python bench.py --gpus N --steps K --warmup W [--config c2|c3|c4|c5]   # this repo's sm_100a path
    python bench.py --impl reference --gpus N ...                          # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR     # also write the last timed step's results as DIR/<name>.npy

Workloads (BASELINE.json configs; ``--config``, default c2 = the configuration the metric is quoted on):
  c2  predict_memory full CWE memory, bert-base, seq_len 512, 64 issue reports / GPU, 129 anchors
  c3  the same at 128 issue reports / GPU (1024 over 8 GPUs)
  c4  anchor-bank stress: 256 issue reports x 16,384 synthetic anchors, seq_len 512 (1 GPU; tiled match)
  c5  mixed seq_len {128,256,512} stream in DATA ORDER, 64 issue reports / GPU (512 over 8 GPUs), token-balanced over
      ranks, packed (var-len) execution so padded tokens cost nothing
Synthetic ids / seeded random weights (no checkpoint or dataset exists offline).  A step = one batch through the test
branch of ``ModelMemory.forward``: encoder (12 layers) + fused pool/header/match/softmax/argmax.  N > 1: one process
per GPU (torchrun), weak scaling, weights and bank replicated, ONE NCCL all-gather of the shard results per step,
issued on a side stream so that it overlaps the next step's encoder.

One JSON line on rank 0:
  value      issues/s over all GPUs, device-timed (CUDA events, max over ranks), inputs resident in HBM
  e2e        same metric through ``ModelMemory.forward`` with HOST (pinned) inputs: H2D of ids/mask/type ids/labels and
             D2H of probs [B,G,2] + best probs/idx inside the timed region (N > 1: the all-gather too)
  roofline   the dominant kernel (largest share of the step): EXECUTED flops per launch / live CUDA-event time
  kernels    per-kernel table from the live run (CUDA events around every launch): launches, avg us, executed flops,
             algorithmic bytes, achieved TFLOP/s and GB/s and their fractions of the measured peaks
  parity     SURVEY 8d gates of THIS run on the rows the CPU baseline leg computed (max logit error, label identity,
             decision margins, rows excluded)
  anchor_match  the match kernel alone on the bank-streaming regime (HBM GB/s) and on BASELINE config 4
  cpu_baseline  the CPU oracle (port of the reference's PyTorch path) timed on this box's host cores
The timed region is preceded by an untimed pre-heat (default 3 s of the same step) so that the K timed steps run in
the sustained clock/power regime; the roofline denominators are then MEASURED_PEAKS.json's sustained figures.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (which may be read-only)

SEQ, SEED = 512, 2021
METRIC, UNIT = "issue-reports/sec, bert-base seq512 + CWE memory", "issues/s"
# which attention kernel the C ABI launches (memvul_abi.cu: MEMVUL_ATT_V, default 3)
ATT_KERNEL = {"1": "attention_tcgen05_kernel", "2": "attention_tcgen05_v2_kernel"}.get(
    os.environ.get("MEMVUL_ATT_V", "3"), "attention_tcgen05_v3_kernel<%s>" % os.environ.get("MEMVUL_ATT_POLY", "0"))

CONFIGS = {
    "c2": {"B": 64, "G": 129, "lens": "full", "name": "C2 predict_memory: bert-base S=512, 64 issue reports/GPU, 129-anchor CWE memory"},
    "c3": {"B": 128, "G": 129, "lens": "full", "name": "C3 predict_memory: bert-base S=512, 128 issue reports/GPU (1024 over 8 GPUs), 129 anchors"},
    "c4": {"B": 256, "G": 16384, "lens": "full", "name": "C4 anchor-bank stress: bert-base S=512, 256 issue reports, 16,384 synthetic anchors"},
    "c5": {"B": 64, "G": 129, "lens": "mixed", "name": "C5 mixed seq_len {128,256,512} stream in data order, 64 issue reports/GPU (512 over 8 GPUs)"},
}
H, I, D = 768, 3072, 512


def flops_per_issue(s: int) -> float:
    """SURVEY.md 8d / BASELINE.md 4: algorithmic FLOPs of the reference per issue report of length s."""
    return 12.0 * (14155776.0 * s + 3072.0 * s * s) + 2 * 768 ** 2 + 2 * 768 * 512


def kernel_work(lens, G, cls_only=True):
    """EXECUTED flops and ALGORITHMIC bytes per launch of every kernel class for one batch with these token counts
    (packed execution: M = sum(lens) token rows; the CLS-only last layer runs its three tail GEMMs on B rows, which are
    accounted under ``cls_tail``, not under the full-size classes)."""
    B, T = len(lens), float(sum(lens))
    att = sum(4.0 * l * l * 64 * 12 for l in lens)
    att_cls = sum(4.0 * min(128, l) * l * 64 * 12 for l in lens)
    w = {
        "embed_ln": {"flops": 0.0, "bytes": T * H * 4 + T * H * 6},
        "gemm_qkv": {"flops": 2 * T * H * 3 * H, "bytes": T * H * 2 + 3 * H * H * 2 + T * 3 * H * 2},
        "attention": {"flops": att, "bytes": T * 3 * H * 2 + T * H * 2},
        "attention_cls": {"flops": att_cls, "bytes": T * 2 * H * 2 + B * 128 * H * 4},
        "gemm_attn_out": {"flops": 2 * T * H * H, "bytes": T * H * 2 + H * H * 2 + T * H * 4 + T * H * 6},
        "gemm_ffn_up": {"flops": 2 * T * H * I, "bytes": T * H * 2 + I * H * 2 + T * I * 2},
        "gemm_ffn_down": {"flops": 2 * T * I * H, "bytes": T * I * 2 + H * I * 2 + T * H * 4 + T * H * 6},
        "cls_tail": {"flops": 2.0 * B * (H * H + 2 * H * I) / 3.0, "bytes": (H * H + 2 * H * I) * 2 / 3.0},   # mean of its 3 GEMMs
        "pool_match": {"flops": 2.0 * B * (H * H + H * D + 2 * D) + 8.0 * B * G * D / 2 * 2,
                       "bytes": 4.0 * (G * D + B * D + 2 * B * G) + 4.0 * 2 * B * G + 4.0 * (H * H + D * H)},
    }
    return w


def executed_flops_per_step(lens, G):
    """All flops the step executes (11 full layers + QKV of layer 12 + first-tile attention + B-row tail + head)."""
    k = kernel_work(lens, G)
    B = len(lens)
    full = k["gemm_attn_out"]["flops"] + k["gemm_ffn_up"]["flops"] + k["gemm_ffn_down"]["flops"] + k["attention"]["flops"]
    return 12 * k["gemm_qkv"]["flops"] + 11 * full + k["attention_cls"]["flops"] + 2.0 * B * (H * H + 2 * H * I) \
        + k["pool_match"]["flops"]


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"src": "MEASURED_PEAKS.json", "tflops_sustained": d.get("bf16_tflops_sustained"), "tflops": d.get("bf16_tflops"),
                "hbm_gbs": d.get("hbm_gbs")}
    return {"src": "fallback (B200_PROFILING.md)", "tflops_sustained": 1400.0, "tflops": 1590.0, "hbm_gbs": 6650.0}


def ncu_traffic():
    """DRAM bytes per launch from the committed `ncu --set full` captures (profiles/ncu_traffic.json); None when absent."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return {}
    with open(p) as f:
        return json.load(f).get("kernels", {})


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark(self):
        return time.time()

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if (t0 is None or t >= t0 - 0.05) and (t1 is None or t <= t1 + 0.1)] or [r for _, r in self.rows]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": statistics.median(pw) if pw else None, "reasons": reasons, "samples": len(sm),
                "window": "timed region of the resident-input leg"}


def pick_cpu_threads(probe) -> int:
    """Use as many host threads as actually help: time a 2-sample probe at several thread counts (the box may
    expose more logical CPUs than it lets a tenant use) and keep the fastest."""
    import torch
    n = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, n) if c <= n})
    best, best_t = cands[0], float("inf")
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            probe()
            t0 = time.perf_counter()
            probe()
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def anchor_match_bench(dev, peaks):
    """BASELINE metric part 2 ("anchor-match HBM GB/s"): memvul_pool_match (fused pool + header + match + softmax +
    arg-max, one cooperative launch) timed alone, L2 evicted with clean lines between launches.
      streaming : 1 query x 262,144 anchors (537 MB bank > L2) -- the HBM-bound regime (SURVEY.md 8d)
      config4   : 256 queries x 16,384 anchors (BASELINE configs[3]) -- FP32-ALU bound, reported for completeness
    Algorithmic bytes = 4*(G*512 + B*512 + 2*B*G) + 4*2*B*G (logits and probs are both written)."""
    import torch
    from memvul_b200 import native as N
    out = {}
    flush = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    sink = torch.zeros(1, dtype=torch.float32, device=dev)
    g = torch.Generator(device="cpu").manual_seed(SEED)
    for name, (B, G) in {"streaming": (1, 262144), "config4": (256, 16384)}.items():
        cls = torch.randn(B, H, generator=g).to(dev)
        wp, bp = (torch.randn(H, H, generator=g) * 0.03).to(dev), (torch.randn(H, generator=g) * 0.02).to(dev)
        wh, bh = (torch.randn(D, H, generator=g) * 0.03).to(dev), (torch.randn(D, generator=g) * 0.02).to(dev)
        wproj = (torch.randn(2, 3 * D, generator=g) * 0.03).to(dev)
        bank = torch.relu(torch.randn(G, D, device=dev))
        vterm = N.bank_prepare(bank, wproj)
        ts = []
        for i in range(8):
            sink.copy_(flush[:1] + flush.sum())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            N.pool_match(cls, H, B, wp, bp, wh, bh, wproj, bank, vterm)
            e1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1))
        t = sorted(ts)[len(ts) // 2] * 1e-3
        nbytes = 4 * (G * D + B * D + 2 * B * G) + 4 * 2 * B * G
        out[name] = {"queries": B, "anchors": G, "us": t * 1e6, "algorithmic_MB": nbytes / 1e6, "hbm_GBps": nbytes / t / 1e9,
                     "frac_of_hbm_peak": nbytes / t / 1e9 / peaks["hbm_gbs"], "fp32_lane_Tinstr_per_s": 3.0 * B * G * D / t / 1e12,
                     "frac_of_fp32_lane_peak": 3.0 * B * G * D / t / 1e12 / 37.2}
        del bank, vterm
    out["peak_hbm_GBps"] = peaks["hbm_gbs"]
    out["peak_fp32_lane_Tinstr_per_s"] = 37.2
    out["peak_src"] = peaks["src"] + "; FP32 lane peak = 148 SM x 128 lanes x 1.965 GHz"
    return out


def host_cpu() -> str:
    """`lscpu`-style identification of the host the CPU baseline ran on: model name x logical CPUs."""
    model = "unknown CPU"
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    return f"{model} x {os.cpu_count()} logical CPUs"


def single_thread_figure(O, sd, ids, mask, tids, bank, same_idx, restore_threads: int):
    """SURVEY.md 8(d): the single-thread figure next to the multi-thread one -- ONE issue report of the sample on one
    host thread (a few seconds at S = 512)."""
    import torch
    S1 = max(1, int(mask[0].sum()))
    torch.set_num_threads(1)
    try:
        with torch.no_grad():
            t0 = time.perf_counter()
            O.memory_forward(sd, ids[:1, :S1].contiguous(), mask[:1, :S1].contiguous(), tids[:1, :S1].contiguous(), bank, same_idx)
            dt = time.perf_counter() - t0
    finally:
        torch.set_num_threads(restore_threads)
    return {"value": 1.0 / dt, "unit": UNIT, "sample": f"1 issue report, S={S1}, G={bank.shape[0]}, 1 thread, {dt:.1f}s"}


def cpu_oracle_throughput(ids, mask, tids, bank, same_idx, budget_s: float = 14.0, batch: int = 8):
    """The reference's CPU path (oracle port) on this box's host cores: a bounded sample of the SAME workload (the
    first rows of the benchmarked batch, in batches of 8).  Returns the timing record and the oracle outputs of the
    sampled rows (the checker for this run's parity gates)."""
    import torch
    from oracle import memvul_oracle as O          # the ONE place the product benchmark touches the oracle: the baseline leg
    sd = O.synthetic_state_dict(O.BERT_BASE, SEED)
    cores = pick_cpu_threads(lambda: O.memory_forward(sd, ids[:2], mask[:2], tids[:2], bank[:129], same_idx))
    refs = []
    with torch.no_grad():
        t0 = time.perf_counter()
        n = 0
        while n < ids.shape[0]:
            sl = slice(n, min(ids.shape[0], n + batch))
            S_b = int(mask[sl].sum(1).max())                       # the reference pads a batch to its longest member
            refs.append(O.memory_forward(sd, ids[sl, :S_b].contiguous(), mask[sl, :S_b].contiguous(), tids[sl, :S_b].contiguous(),
                                         bank, same_idx))
            n = sl.stop
            dt = time.perf_counter() - t0
            if dt > budget_s:
                break
    rec = {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"{n} issue reports of this run's batch (batches of {batch}, padded to the batch maximum, G={bank.shape[0]}) in {dt:.1f}s, "
                     f"torch {torch.__version__} fp32 CPU, {torch.get_num_threads()} threads",
           "note": "a stated baseline, not a target: ~0.3 TFLOP/s of fp32 eager PyTorch on host cores",
           "single_thread": single_thread_figure(O, sd, ids, mask, tids, bank, same_idx, cores), "host": host_cpu()}
    ref = {k: torch.cat([r[k] for r in refs]) for k in ("logits", "p")}
    return rec, ref, n


DUMP_BYTES = 64_000_000            # --dump-outputs: all files together stay within 64 MB


def write_outputs(out_dir, arrays):
    """``--dump-outputs``: one ``out_dir/<name>.npy`` per result array, float32 (integer arrays as float64, which holds
    them exactly), so that two builds can be compared output for output on the same seeded inputs.  When the
    [B, G, 2] arrays (logits, probs) would take the total over DUMP_BYTES (config c4), they keep a seeded random subset
    of the anchors, the same one in every run with the same arguments, listed in ``anchor_index.npy``."""
    import numpy as np
    import torch
    out = {k: v.numpy().astype(np.float32 if v.is_floating_point() else np.float64) for k, v in arrays.items()}
    wide = [k for k, a in out.items() if a.ndim == 3]
    budget = DUMP_BYTES - 256 * (len(out) + 1)                        # .npy headers
    total = sum(a.nbytes for a in out.values())
    if wide and total > budget:
        G = out[wide[0]].shape[1]
        per_anchor = sum(out[k][:, :1].nbytes for k in wide) + 8      # + its entry in anchor_index
        keep = max(1, (budget - (total - G * (per_anchor - 8))) // per_anchor)
        idx = torch.randperm(G, generator=torch.Generator().manual_seed(SEED))[:keep].sort().values.numpy()
        out = {k: (a[:, idx] if k in wide else a) for k, a in out.items()}
        out["anchor_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(a))
    written = sum(os.path.getsize(os.path.join(out_dir, k + ".npy")) for k in out)
    if written > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs wrote {written} bytes, more than {DUMP_BYTES}")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = args.steps or 20, max(args.warmup, 0)
    import torch
    from oracle import memvul_oracle as O
    cfg = CONFIGS[args.config]
    sd = O.synthetic_state_dict(O.BERT_BASE, SEED)
    b = 8                                             # bounded sample of the batch per step
    lens = make_lens(cfg, 64, 0)[:b]
    ids, mask, tids = O.synthetic_ids(b, max(lens), lens=lens, seed=SEED + 100)
    g = torch.Generator().manual_seed(SEED)
    G = min(cfg["G"], 129) if args.config != "c4" else cfg["G"]
    bank = torch.relu(torch.randn(G, 512, generator=g) * 0.3)
    cores = pick_cpu_threads(lambda: O.memory_forward(sd, ids[:2], mask[:2], tids[:2], bank[:129], 0))
    with torch.no_grad():
        for _ in range(min(warm, 2)):
            O.memory_forward(sd, ids, mask, tids, bank, 0)
        t0 = time.perf_counter()
        for _ in range(steps):
            last = O.memory_forward(sd, ids, mask, tids, bank, 0)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, last)
    v = steps * b / dt
    single = single_thread_figure(O, sd, ids, mask, tids, bank, 0, cores)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": min(warm, 2), "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{cfg['name']}; CPU sample of {b} issue reports per step (G={G})",
                       "note": "reference = CPU fp32 PyTorch restatement of ModelMemory.forward (oracle port); AllenNLP is not installable offline"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{steps} steps x {b} issue reports, S<={SEQ}, {torch.get_num_threads()} threads",
                             "single_thread": single, "host": host_cpu()},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def make_lens(cfg, n, seed_off):
    """Token counts of n issue reports: all 512 (c2-c4) or a uniform draw from {128,256,512} (c5, SURVEY 8d)."""
    import torch
    if cfg["lens"] == "full":
        return [SEQ] * n
    g = torch.Generator().manual_seed(SEED + 7 + seed_off)
    return [int((128, 256, 512)[i]) for i in torch.randint(0, 3, (n,), generator=g)]


def run_native(args):
    import torch
    import torch.distributed as dist
    from memvul_b200 import native
    from memvul_b200.dist import AsyncGather, balanced_assignment
    from memvul_b200.parity import gate_report
    from memvul_b200.synthetic import BERT_BASE, build_memory_model, synthetic_ids

    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (memvul_b200 has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warm = max(args.warmup, 3)
    B_PER_GPU = int(os.environ.get("MEMVUL_BENCH_B", str(cfg["B"])))       # env override: experiments only
    G = cfg["G"]

    model, _ = build_memory_model(BERT_BASE, SEED, device=dev)
    with torch.no_grad():
        if args.config == "c4":
            # SURVEY 8d: the config-4 bank is relu(N(0,1))-distributed fp32 [16384,512] (post-ReLU header outputs), which
            # decouples the stress test from 1.58 PFLOP of bank encoding
            g = torch.Generator().manual_seed(SEED + 1)
            model._golden_instances_embeddings = torch.relu(torch.randn(G, 512, generator=g) * 0.3).to(dev)
            model._golden_instances_labels = [f"CWE-{i}" for i in range(G)]
        else:
            # 129 synthetic anchors (len 64..512) encoded by the model itself, in the reference's 128 + rest chunks
            g = torch.Generator().manual_seed(SEED + 1)
            a_lens = torch.randint(64, SEQ + 1, (G,), generator=g).tolist()
            for c0, c1 in ((0, 128), (128, G)):
                lens_c = a_lens[c0:c1]
                ids, mask, tids = synthetic_ids(len(lens_c), max(lens_c), lens=lens_c, seed=SEED + 2 + c0)
                model.forward_gold_instances({"tokens": {"token_ids": ids.to(dev), "mask": mask.to(dev), "type_ids": tids.to(dev)}},
                                             [{"type": "golden", "instance": [{"label": f"CWE-{c0 + i}"}]} for i in range(len(lens_c))])
    # ---- this rank's batch
    total = B_PER_GPU * world
    lens_all = make_lens(cfg, total, 0)
    if cfg["lens"] == "mixed" and world > 1:
        mine = balanced_assignment(lens_all, world)[rank]                 # token-balanced shards of the global batch
    else:
        mine = list(range(rank * B_PER_GPU, (rank + 1) * B_PER_GPU))
    lens = [lens_all[i] for i in mine]
    B = len(lens)
    counts = [B] * world
    if world > 1:
        ct = torch.tensor([B], device=dev)
        allc = [torch.zeros_like(ct) for _ in range(world)]
        dist.all_gather(allc, ct)
        counts = [int(c.item()) for c in allc]
    ids_c, mask_c, tids_c = synthetic_ids(B, max(lens), lens=lens, seed=SEED + 100 + rank)
    ids_h, mask_h, tids_h = (t.pin_memory() for t in (ids_c, mask_c, tids_c))
    label_h = (torch.arange(B) % 301 == 0).long().pin_memory()          # ~1:300 CIR:NCIR, labels do not change compute
    meta = [{"type": "unlabel", "instance": [{"label": "neg", "Issue_Url": f"synthetic/{rank}/{i}"}]} for i in range(B)]
    ids_d, mask_d, tids_d = ids_h.to(dev), mask_h.to(dev), tids_h.to(dev)
    sample_d = {"tokens": {"token_ids": ids_d, "mask": mask_d, "type_ids": tids_d}}
    gather = AsyncGather(counts, dev) if world > 1 else None
    if gather is not None:
        model.shard_capacity = max(counts)           # results in one flat buffer: the all-gather needs no packing

    def step_resident():
        res = model.match_batch(sample_d)
        if gather is not None:
            gather.submit(res)                       # side stream: overlaps the next step's encoder
        return res

    def step_e2e():
        s = {"tokens": {"token_ids": ids_h.to(dev, non_blocking=True), "mask": mask_h.to(dev, non_blocking=True),
                        "type_ids": tids_h.to(dev, non_blocking=True)}}
        out = model(sample1=s, label=label_h.to(dev, non_blocking=True), metadata=meta)
        if gather is not None:
            gather.submit(out["native"]["device"])
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n, after=None):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.time()
        e0.record()
        last = None
        for _ in range(n):
            last = fn()
        if after is not None:
            after(last)
        if gather is not None:
            gather.wait()                            # the last step's collective completes inside the timed region
        e1.record()
        barrier()
        t1 = time.time()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, t0, t1, last

    with torch.no_grad():
        for _ in range(warm):
            step_resident()
        if gather is not None:
            gather.wait()
        torch.cuda.synchronize()
        # ---- calibrate: step time -> number of pre-heat steps and (when --steps is not given) of timed steps
        ms_cal = timed(step_resident, 3)[0]
        step_ms = ms_cal / 3
        steps = args.steps if args.steps else max(20, int(3200.0 / step_ms) + 1)      # default: >= 3 s timed region
        preheat_steps = int(args.preheat_s * 1e3 / step_ms) if args.preheat_s > 0 else 0
        if world > 1:                                     # every rank must run the same number of steps
            t = torch.tensor([steps, preheat_steps], device=dev)
            dist.broadcast(t, 0)
            steps, preheat_steps = int(t[0]), int(t[1])
        for _ in range(preheat_steps):
            step_resident()
        if gather is not None:
            gather.wait()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
            time.sleep(0.06)
        l0 = native.launch_count()
        ms_res, t0, t1, res_timed = timed(step_resident, steps)
        launches = native.launch_count() - l0
        clocks = sampler.stop(t0, t1) if rank == 0 else None
        # what a caller of match_batch received from the last timed step (rank 0's shard when N > 1)
        dumped = {k: v.cpu() for k, v in res_timed.items() if not k.startswith("_")} \
            if args.dump_outputs and rank == 0 else None

        for _ in range(2):
            step_e2e()["probs"].numpy()

        def drain(last):                      # the step's result is read on the host inside the timed region
            last["probs"].numpy()
            model.get_metrics(reset=False)
        ms_e2e = timed(step_e2e, steps, after=drain)[0]
        model.get_metrics(reset=True)

        # live per-kernel timing: same step with CUDA events around every launch, right after ~1 s of un-instrumented
        # steps so that the table is taken in the same sustained clock regime as `value` (r02c: profiled cold, FFN-up
        # showed 1.00 of the SUSTAINED peak)
        for _ in range(max(3, preheat_steps // 3)):
            model.match_batch(sample_d)
        native.profile_enable(True)
        native.profile_read()
        prof_steps = 10
        for _ in range(prof_steps):
            model.match_batch(sample_d)
        prof = native.profile_read()
        native.profile_enable(False)
        res_last = model.match_batch(sample_d)
        got = {k: res_last[k].cpu() for k in ("logits", "probs", "best_idx")}
        bank_cpu = model._golden_instances_embeddings.cpu()
        same_idx = model._same_idx

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    n_total = sum(counts)
    value = n_total * steps / (ms_res / 1e3)
    e2e_v = n_total * steps / (ms_e2e / 1e3)
    peaks = measured_peaks()
    region_s = ms_res / 1e3
    sustained = (region_s + preheat_steps * step_ms / 1e3) >= 2.0
    pk_t = peaks["tflops_sustained"] if sustained else peaks["tflops"]
    pk_name = ("bf16_tflops_sustained" if sustained else "bf16_tflops (burst)") + f" from {peaks['src']}"
    work = kernel_work(lens, G)
    traffic = ncu_traffic()
    step_ms_prof = sum(v["ms"] for v in prof.values()) / prof_steps
    kernels = {}
    kname = {"embed_ln": "embed_layernorm_kernel", "gemm_qkv": "gemm_f16_tcgen05_2cta_kernel<BIAS_F16>",
             "attention": ATT_KERNEL, "attention_cls": ATT_KERNEL + " (first query tile, last layer)",
             "gemm_attn_out": "gemm_ln_f16_tcgen05_kernel (K=768)", "gemm_ffn_up": "gemm_f16_tcgen05_2cta_kernel<BIAS_GELU_F16>",
             "gemm_ffn_down": "gemm_ln_f16_tcgen05_kernel (K=3072)", "cls_tail": "gemm_f16_tcgen05_kernel<128,*> + layernorm_rows (B rows)",
             "pool_match": "pool_match_kernel", "layernorm": "layernorm_rows_kernel", "other": "mask_to_lens / row_start / gather_cls"}
    for k, v in prof.items():
        if not v["launches"]:
            continue
        n_l = v["launches"] / prof_steps
        avg_ms = v["ms"] / v["launches"]
        row = {"kernel": kname.get(k, k), "launches_per_step": round(n_l, 2), "avg_us": round(avg_ms * 1e3, 2),
               "ms_per_step": round(v["ms"] / prof_steps, 4), "share": round(v["ms"] / prof_steps / step_ms_prof, 4)}
        if k in work:
            fl, by = work[k]["flops"], work[k]["bytes"]
            row.update({"flops_per_launch": fl, "bytes_per_launch": by,
                        "tflops": round(fl / avg_ms / 1e9, 1) if fl else None,
                        "frac_tensor": round(fl / avg_ms / 1e9 / pk_t, 4) if fl else None,
                        "gbps": round(by / avg_ms / 1e6, 1), "frac_hbm": round(by / avg_ms / 1e6 / peaks["hbm_gbs"], 4)})
        kernels[k] = row
    dom = max((k for k in kernels if k in ("gemm_qkv", "attention", "gemm_attn_out", "gemm_ffn_up", "gemm_ffn_down")),
              key=lambda k: kernels[k]["ms_per_step"])
    dk = kernels[dom]
    tr_key = {"gemm_qkv": "gemm_qkv", "gemm_ffn_up": "gemm_ffn_up", "gemm_attn_out": "ln_attn_out", "gemm_ffn_down": "ln_ffn_down",
              "attention": "attention"}[dom]
    h2d = ids_h.numel() * 8 + tids_h.numel() * 8 + mask_h.numel() + label_h.numel() * 8
    d2h = B * G * 2 * 4 + B * 2 * 4 + B * 4 + 4
    alg_flops = sum(flops_per_issue(l) for l in lens_all) if world > 1 and cfg["lens"] == "mixed" else sum(flops_per_issue(l) for l in lens) * world
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
        "ms_per_step": ms_res / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands, f32 accumulate/residual (reference: f32)", "data": "synthetic",
        "config": {"workload": cfg["name"], "config": args.config, "global_batch": n_total, "seq_len": SEQ, "anchors": G,
                   "tokens_per_step": int(sum(lens)) * world if cfg["lens"] == "full" else int(sum(lens_all)),
                   "parallelism": f"batch-shard x{world}", "execution": "packed var-len (token-major), device-side row count",
                   "l2": "per-step working set ~650 MB > 126 MB L2 (no flush needed)", "weights": f"seeded random, seed {SEED}",
                   "preheat_s": round(preheat_steps * step_ms / 1e3, 2), "preheat_steps": preheat_steps,
                   "timed_region_s": round(region_s, 3)},
        "e2e": {"value": e2e_v, "unit": UNIT, "ms_per_step": ms_e2e / steps, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "ModelMemory.forward(sample1, label, metadata) with pinned host inputs; probs read on host"
                       + ("; the per-step NCCL all-gather of the shard results is inside the region" if world > 1 else "")},
        "gpu_launches": int(launches),
        "tensor_utilisation": {"algorithmic_tflops": alg_flops * steps / (ms_res / 1e3) / 1e12,
                               "executed_tflops": executed_flops_per_step(lens, G) * world * steps / (ms_res / 1e3) / 1e12,
                               "frac_of_peak": alg_flops * steps / (ms_res / 1e3) / 1e12 / world / pk_t,
                               "peak": pk_t, "peak_src": pk_name,
                               "note": "algorithmic = SURVEY 8d F(len) per issue report (the reference's full 12 layers); executed = what the CLS-only last layer actually runs"},
        "roofline": {"kernel": dk["kernel"], "class": dom, "bound": "tensor", "achieved": dk["tflops"], "peak": pk_t, "unit": "TFLOP/s",
                     "frac": dk["frac_tensor"], "peak_src": pk_name,
                     "flops_per_launch": dk["flops_per_launch"], "avg_launch_ms": dk["avg_us"] / 1e3,
                     "launches_per_step": dk["launches_per_step"], "share_of_step": dk["share"],
                     "hbm": {"achieved_GBps": dk["gbps"], "peak_GBps": peaks["hbm_gbs"], "frac": dk["frac_hbm"],
                             "algorithmic_bytes_per_launch": dk["bytes_per_launch"]},
                     "traffic": (traffic.get(tr_key) or {}).get("dram_traffic_bytes"),
                     "traffic_src": "profiles/ncu_traffic.json: dram__bytes_read+write per launch (ncu --set full) of this kernel at C2"},
        "kernels": kernels,
        "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        n_cpu = B if args.config != "c4" else 16
        cpu, ref, n_ref = cpu_oracle_throughput(ids_c[:n_cpu], mask_c[:n_cpu], tids_c[:n_cpu], bank_cpu, same_idx,
                                                budget_s=14.0 if args.config != "c4" else 25.0)
        line["cpu_baseline"] = cpu
        rep = gate_report(got["logits"][:n_ref].numpy(), got["probs"][:n_ref].numpy(), got["best_idx"][:n_ref].numpy(),
                          ref["logits"].numpy(), ref["p"].numpy(), same_idx, thresholds=(0.5,))
        rep["checker"] = ("CPU oracle on the first %d rows of this run's batch; bank = the device-built bank copied to the host "
                          "(bank parity itself is gated in tests/test_configs_gpu.py)" % n_ref)
        line["parity"] = rep
    if world == 1 and not args.no_anchor_bench:
        del model
        torch.cuda.empty_cache()
        line["anchor_match"] = anchor_match_bench(dev, peaks)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: enough for a >= 3 s timed region)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--preheat-s", type=float, default=3.0, help="untimed pre-heat before the timed steps (sustained clocks)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-anchor-bench", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (<= 64 MB in all)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1 and args.impl == "native":
        # convenience: re-launch under torchrun when called directly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
