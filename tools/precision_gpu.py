"""On-hardware precision evidence (VERDICT r01 item 10): the GPU path (fp16 operands, fp32 accumulate / residual stream)
against the CPU oracle over 768 S=512 issue reports x 129 anchors, with the match head (``_projector``) scaled x1, x4
and x16 -- the logit error grows with the head scale, the 1e-3 gate of BASELINE.json's north_star does not.

    python tools/precision_gpu.py [--out profiles/r02_precision.json]

The oracle's header outputs come from tests/golden/precision_u768.npz (made on the CPU by oracle/make_precision_fixture.py);
the match itself is re-evaluated here in float64 for every scale from (u, bank)."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from config_inputs import c2_inputs, split_threshold  # noqa: E402
from memvul_b200 import native as N  # noqa: E402
from memvul_b200.synthetic import BERT_BASE, build_memory_model, synthetic_ids  # noqa: E402


def match64(u, bank, w, same):
    """model_memory.py:135-147 in float64 (separable form; identical to the concat form up to fp64 rounding)."""
    u, bank, w = u.double(), bank.double(), w.double()
    D = u.shape[1]
    wu, wv, wd = w[:, :D], w[:, D:2 * D], w[:, 2 * D:]
    logits = (u @ wu.T)[:, None, :] + (bank @ wv.T)[None] + torch.einsum("bgk,ck->bgc", (u[:, None] - bank[None]).abs(), wd)
    return logits, torch.softmax(logits, -1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "split_fp16"],
                    help="split_fp16 = the opt-in accuracy mode (MEMVUL_ENC_PRECISE)")
    ap.add_argument("--rows", type=int, default=0, help="use only the first N rows of the fixture (the accuracy mode is slow)")
    args = ap.parse_args()
    z = np.load(os.path.join(ROOT, "tests", "golden", "precision_u768.npz"))
    u_ref, bank_ref = torch.from_numpy(z["u"]), torch.from_numpy(z["bank"])
    seed, n_rows = int(z["seed"]), int(z["rows"])
    if args.rows:
        n_rows = min(n_rows, args.rows // 64 * 64)
        u_ref = u_ref[:n_rows]
    dev = torch.device("cuda:0")
    model, sd = build_memory_model(BERT_BASE, device=dev, precision=args.precision)
    a_ids, a_mask, alens, *_ = c2_inputs()
    us = []
    with torch.no_grad():
        for c0 in (0, 128):
            ids, mask = a_ids[c0:c0 + 128], a_mask[c0:c0 + 128]
            if ids.shape[0] == 0:
                continue
            S = int(mask.sum(1).max())
            model.forward_gold_instances({"tokens": {"token_ids": ids[:, :S].contiguous().to(dev), "mask": mask[:, :S].contiguous().to(dev),
                                                     "type_ids": torch.zeros_like(ids[:, :S]).contiguous().to(dev)}},
                                         [{"type": "golden", "instance": [{"label": f"CWE-{c0 + i}"}]} for i in range(ids.shape[0])])
        for b in range(n_rows // 64):
            ids, mask, tids = synthetic_ids(64, 512, seed=seed + b)
            us.append(model.match_batch({"tokens": {"token_ids": ids.to(dev), "mask": mask.to(dev), "type_ids": tids.to(dev)}})["u"].clone())
    u_dev = torch.cat(us)
    bank_dev = model._golden_instances_embeddings
    same = model._same_idx
    rep = {"rows": n_rows, "anchors": int(bank_ref.shape[0]), "seq_len": 512,
           "arithmetic": ("fp16 operands (kind::f16), fp32 TMEM accumulation, fp32 residual stream / LayerNorm / softmax statistics; pooler, header and match in fp32"
                          if args.precision == "fp16" else
                          "accuracy mode: split-fp16 operands (3 partial products per GEMM on the kind::f16 kernels), fp32 attention / GELU / LayerNorm; pooler, header and match in fp32"),
           "u_err": {"max": float((u_dev.cpu() - u_ref).abs().max()), "p999": float(torch.quantile((u_dev.cpu() - u_ref).abs().flatten()[::7], 0.999)),
                     "mean": float((u_dev.cpu() - u_ref).abs().mean())},
           "bank_err": {"max": float((bank_dev.cpu() - bank_ref).abs().max())}, "scales": {}}
    w0 = sd["_projector.weight"]
    H = 768
    dummy_w, dummy_b = torch.zeros(H, H, device=dev), torch.zeros(H, device=dev)
    for scale in (1.0, 4.0, 16.0):
        w = w0 * scale
        wd = w.to(dev).contiguous()
        out = N.pool_match(None, 0, n_rows, dummy_w, dummy_b, torch.zeros(512, H, device=dev), None, wd, bank_dev.contiguous(),
                           N.bank_prepare(bank_dev.contiguous(), wd), same_idx=same,
                           phase_mask=N.PM_UTERM | N.PM_MATCH | N.PM_FINAL, u=u_dev.contiguous())
        lg_ref, p_ref = match64(u_ref, bank_ref, w, same)
        lg = out["logits"].cpu().double()
        p = out["probs"].cpu().double()
        err = (lg - lg_ref).abs().flatten()
        vote_ref, vote = p_ref[:, :, same].max(1).values, p[:, :, same].max(1).values
        thr, margin = split_threshold(vote_ref)
        srt = torch.sort(p_ref[:, :, same], dim=1).values
        gap = srt[:, -1] - srt[:, -2]
        idx_ref = p_ref[:, :, same].argmax(1)
        idx = out["best_idx"].cpu().long()
        rep["scales"][f"x{scale:g}"] = {
            "logit_abs_max_ref": float(lg_ref.abs().max()),
            "logit_err": {"max": float(err.max()), "p999": float(torch.quantile(err[::3], 0.999)), "mean": float(err.mean())},
            "within_1e-3": bool(err.max() <= 1e-3),
            "vote_spread": [float(vote_ref.min()), float(vote_ref.max())],
            "label_flips": {"thr_0.5": int(((vote >= 0.5) != (vote_ref >= 0.5)).sum()),
                            f"thr_split_{thr:.4f}": int(((vote >= thr) != (vote_ref >= thr)).sum()), "split_margin": margin,
                            "rows_within_1e-3_of_0.5": int(((vote_ref - 0.5).abs() <= 1e-3).sum()),
                            "rows_within_1e-3_of_split": int(((vote_ref - thr).abs() <= 1e-3).sum())},
            "argmax": {"flips": int((idx != idx_ref).sum()), "flips_where_gap_gt_2e-3": int(((idx != idx_ref) & (gap > 2e-3)).sum()),
                       "rows_gap_gt_2e-3": int((gap > 2e-3).sum())}}
        print(f"x{scale:g}:", json.dumps(rep["scales"][f"x{scale:g}"]), flush=True)
    print(json.dumps(rep))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
