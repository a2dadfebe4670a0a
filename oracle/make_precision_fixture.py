"""Oracle side of the on-hardware precision study (VERDICT r01 item 10): the CPU fp32 restatement's header outputs u for
768 synthetic S=512 issue reports and the 129-anchor bank, written to tests/golden/precision_u768.npz (float32, < 1 MB).
The match logits for ANY projector scale follow from (u, bank) in milliseconds, so tools/precision_gpu.py can compare
the GPU path against the oracle at head scales x1, x4, x16 without re-running the 12-layer CPU encoder on the GPU box.
Run here (build container, ~12 min on 8 cores); test infrastructure only."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from config_inputs import c2_inputs  # noqa: E402
from oracle import memvul_oracle as O  # noqa: E402

N_ROWS, SEED = 768, 4242


def rows(n=N_ROWS, seed=SEED):
    """``n`` full-length (512-token) synthetic issue reports, in batches of 64 with per-batch seeds."""
    out = []
    for b in range(n // 64):
        ids, mask, tids = O.synthetic_ids(64, 512, seed=seed + b)
        out.append((ids, mask, tids))
    return out


def main():
    sd = O.synthetic_state_dict(O.BERT_BASE, 2021)
    a_ids, a_mask, alens, *_ = c2_inputs()
    t0 = time.time()
    with torch.no_grad():
        bank = O.build_bank(sd, [(a_ids[i][a_mask[i]], a_mask[i][a_mask[i]]) for i in range(len(alens))])
        us = []
        for k, (ids, mask, tids) in enumerate(rows()):
            for c in range(0, 64, 16):
                us.append(O.instance_forward(sd, ids[c:c + 16], mask[c:c + 16], tids[c:c + 16]))
            print(f"batch {k + 1}/{N_ROWS // 64} done, {time.time() - t0:.0f}s", flush=True)
    u = torch.cat(us).numpy().astype(np.float32)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "precision_u768.npz"), u=u, bank=bank.numpy().astype(np.float32),
                        seed=np.int64(SEED), rows=np.int64(N_ROWS))
    print("wrote precision_u768.npz", u.shape, bank.shape)


if __name__ == "__main__":
    main()
