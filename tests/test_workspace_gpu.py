"""Encoder results must not depend on what the workspace (or the output tensor) held before the call.

The packed (var-len) execution computes whole GEMM tiles: up to round_up(T, 128) or round_up(T, 256) rows, where
T = row_start[B] is the token count the kernels read on the device, and the attention's last key block of the last
sequence loads up to 63 rows past T.  Those rows are multiplied by P = 0 (masked keys), but 0 * NaN = NaN, so a
non-finite value there poisons the last sequence of the batch.  A workspace reused for a batch of another shape is
carved at other offsets, so its rows past T can hold any bits an earlier call wrote (fp32 values read as fp16 are
NaN or Inf about once in 32).

Every check here compares with the same call on a freshly zeroed workspace (the path the oracle tests pin) and must
agree bit for bit on the rows the call defines; those rows must be finite."""
import os
import random
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILLS = [0xFF, 0x7B]       # every byte 0xFF: NaN as fp16 and fp32; 0x7B: 6.1e4 as fp16, 1.3e36 as fp32 (finite, huge)


@pytest.fixture(scope="module")
def N():
    from memvul_b200 import native
    native.build()
    return native


@pytest.fixture(scope="module")
def weights(N):
    from memvul_b200.synthetic import BERT_BASE, BERT_TINY, EMB, synthetic_state_dict
    cache = {}

    def get(name, precise=False):
        if (name, precise) not in cache:
            shape = BERT_TINY if name == "tiny" else BERT_BASE
            cache[(name, precise)] = N.PackedBert(synthetic_state_dict(shape), EMB, torch.device("cuda"), precise=precise)
        return cache[(name, precise)]
    return get


# ------------------------------------------------------------------------------------------------ helpers
def _up(n):
    return (n + 1023) & ~1023


def carve_layout(N, hidden, inter, B, S, flags):
    """Python mirror of carve() / carve_precise() (memvul_b200/csrc/memvul_abi.cu): ({buffer: (byte offset, bytes)},
    total bytes).  Every test that relies on it checks the total against memvul_encoder_workspace_bytes."""
    M, H, I = B * S, hidden, inter
    if flags & N.ENC_PRECISE:
        parts = [("x32", M * H * 4), ("xs", M * 3 * H * 2), ("qkv32", M * 3 * H * 4), ("ctx32", M * H * 4),
                 ("h32", M * I * 4), ("hs", M * 3 * I * 2)]
    else:
        parts = [("x16", M * H * 2), ("qkv", M * 3 * H * 2), ("ctx", M * H * 2), ("ffn", M * I * 2),
                 ("x32_cls", B * H * 4), ("x16_cls", B * H * 2), ("ctx_cls", B * H * 2), ("ffn_cls", B * I * 2)]
        if (flags & N.ENC_PACKED) and not (flags & N.ENC_CLS_ONLY):
            parts.append(("x32_packed", M * H * 4))
    lay, off = {}, 0
    for name, n in parts:
        lay[name] = (off, n)
        off += _up(n)
    return lay, off


def _layout(N, w, B, S, flags):
    lay, total = carve_layout(N, w.hidden, w.intermediate, B, S, flags)
    assert total == w.workspace_bytes(B, S, flags), (B, S, flags)
    return lay


def _ids(lens, S, vocab, seed):
    """Prefix-masked ids like synthetic_ids, but lengths of 1 are allowed."""
    g = torch.Generator().manual_seed(seed)
    B = len(lens)
    lo = 1000 if vocab > 2000 else vocab // 2
    ids = torch.randint(lo, vocab, (B, S), generator=g, dtype=torch.int64)
    L = torch.tensor(lens, dtype=torch.int64)
    assert int(L.min()) >= 1 and int(L.max()) <= S
    mask = torch.arange(S)[None, :] < L[:, None]
    ids[:, 0] = 101
    ids[torch.arange(B), L - 1] = torch.where(L > 1, 102, 101)
    return (ids * mask).cuda(), mask.cuda()


def _split(T, B, S, seed):
    """B uneven lengths in [1, S] summing to T, the last not a multiple of 64 (its key block is ragged)."""
    g = random.Random(seed)
    lens = [T // B + (i < T % B) for i in range(B)]
    for _ in range(4 * B):
        i, j = g.randrange(B), g.randrange(B)
        d = g.randint(0, min(lens[i] - 1, S - lens[j]))
        lens[i] -= d
        lens[j] += d
    if lens[-1] % 64 == 0:
        k = next(i for i in range(B - 1) if (lens[i] > 1 if lens[-1] < S else lens[i] < S))
        step = 1 if lens[-1] < S else -1
        lens[k] -= step
        lens[-1] += step
    assert sum(lens) == T and min(lens) >= 1 and max(lens) <= S and lens[-1] % 64 != 0
    return lens


def _encode(N, w, ids, mask, packed, cls_only, fill=None):
    """encoder_forward with a workspace AND an output tensor whose every byte is ``fill`` (None: a fresh zeroed
    workspace and output).  Returns the output after checking the deferred error flag."""
    B, S = ids.shape
    if packed:
        lens, rs, bad = N.mask_to_lens(mask, with_row_start=True)
    else:
        (lens, bad), rs = N.mask_to_lens(mask), None
    flags = N.encoder_flags(w, cls_only, packed)
    nbytes = w.workspace_bytes(B, S, flags)
    ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.zeros(B, S, w.hidden, dtype=torch.float32, device="cuda")
    if fill is not None:
        ws.fill_(fill)
        out.view(torch.uint8).fill_(fill)
    out = N.encoder_forward(w, ids, lens, workspace=ws, out=out, cls_only=cls_only, row_start=rs, bad=bad)
    assert int(bad) == 0
    return out


def _assert_same(got, want, mask, packed, cls_only, what):
    """``got`` is finite on the rows the interface defines ([CLS] rows for cls_only, else every row: padded positions
    are zero in the packed layout and unspecified but finite in the padded one) and equals ``want`` on the valid ones."""
    g, r = (got[:, 0], want[:, 0]) if cls_only else (got, want)
    assert bool(torch.isfinite(g).all()), (what, "non-finite rows", torch.nonzero(~torch.isfinite(g).all(-1))[:8].tolist())
    if cls_only:
        ok = torch.equal(g, r)
        bad_rows = torch.nonzero((g != r).any(-1)).flatten()[:8].tolist()
    else:
        ok = torch.equal(got[mask], want[mask])
        bad_rows = torch.nonzero(((got != want).any(-1) & mask).any(-1)).flatten()[:8].tolist()
        if packed:
            assert float(got[~mask].abs().max() if (~mask).any() else 0.0) == 0.0, (what, "padded positions not zero")
    assert ok, (what, "differs from the zeroed-workspace run in sequences", bad_rows)


# ------------------------------------------------------------------------------------------------ dirty workspace
# lens: the last sequence is ragged (len % 64 != 0) and T mod 256 >= 194, so its last key block reaches past the last
# 256-row GEMM tile.  tiny: B*S = 1200, T = 706.  base: B*S = 2048 (QKV on the 128-row kernel, FFN-up on the CTA-pair
# kernel, fused LayerNorms), T = 1250.
DIRTY = {"tiny": (200, [200, 130, 7, 64, 133, 172]), "base": (256, [256, 200, 31, 255, 100, 256, 90, 62])}


@pytest.mark.parametrize("cls_only", [False, True], ids=["full", "cls_only"])
@pytest.mark.parametrize("packed", [True, False], ids=["packed", "padded"])
@pytest.mark.parametrize("shape", ["tiny", "base"])
def test_dirty_workspace_gives_the_zeroed_result(N, weights, shape, packed, cls_only):
    w = weights(shape)
    S, lens = DIRTY[shape]
    _layout(N, w, len(lens), S, N.encoder_flags(w, cls_only, packed))
    ids, mask = _ids(lens, S, w.word.shape[0], seed=len(lens))
    want = _encode(N, w, ids, mask, packed, cls_only)
    for fill in FILLS:
        got = _encode(N, w, ids, mask, packed, cls_only, fill)
        _assert_same(got, want, mask, packed, cls_only, (shape, packed, cls_only, hex(fill)))


@pytest.mark.parametrize("shape,packed,cls_only", [("tiny", True, False), ("tiny", True, True), ("tiny", False, False),
                                                   ("tiny", False, True), ("base", True, True)])
def test_dirty_workspace_accuracy_mode(N, weights, shape, packed, cls_only):
    """MEMVUL_ENC_PRECISE (PackedBert(precise=True)) carves its own workspace: the same guarantee."""
    w = weights(shape, precise=True)
    S, lens = DIRTY[shape]
    _layout(N, w, len(lens), S, N.encoder_flags(w, cls_only, packed))
    ids, mask = _ids(lens, S, w.word.shape[0], seed=len(lens))
    want = _encode(N, w, ids, mask, packed, cls_only)
    got = _encode(N, w, ids, mask, packed, cls_only, 0xFF)
    _assert_same(got, want, mask, packed, cls_only, (shape, "precise", packed, cls_only))


# ------------------------------------------------------------------------------------------------ row-count edges
# bert-base at B*S = 8 x 512: the CTA-pair GEMMs (256-row tiles) and the six-CTA fused LayerNorm run, as in
# production.  T at the 128 / 256-row tile edges, and T mod 256 in [194, 255] (450, 511, 1000, 2000), where the last
# sequence's ragged key block crosses the last GEMM tile.  B*S = 2 x 512: QKV and FFN-up on the 128-row kernel
# (which writes no row past T), the attention-output and FFN-down GEMMs fused with LayerNorm on 256-row tiles.
EDGES = [(8, 512, T) for T in (8, 127, 128, 129, 255, 256, 257, 383, 385, 450, 511, 1000, 2000)] + \
        [(2, 512, T) for T in (2, 129, 200, 255, 257, 450, 511, 706, 1000)]


def _edge_case(B, S, T):
    lens = _split(T, B, S, seed=T * 7 + B)
    return lens, 30522, T + B


def _edge_results(N, w, B, S, T, fill):
    """(packed, padded) x (full, cls_only) outputs of one edge case on a workspace filled with ``fill``."""
    lens, vocab, seed = _edge_case(B, S, T)
    ids, mask = _ids(lens, S, vocab, seed)
    return mask, {(p, c): _encode(N, w, ids, mask, p, c, fill) for p in (True, False) for c in (False, True)}


@pytest.mark.parametrize("B,S,T", EDGES)
def test_packed_equals_padded_at_row_count_edges(N, weights, B, S, T):
    w = weights("base")
    mask, r = _edge_results(N, w, B, S, T, 0xFF)
    for c in (False, True):
        _assert_same(r[(True, c)], r[(False, c)], mask, True, c, ("packed vs padded", B, S, T, c))


_CHILD = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[1] + "/tests")
import test_workspace_gpu as t
from memvul_b200 import native as N
from memvul_b200.synthetic import BERT_BASE, EMB, synthetic_state_dict
w = N.PackedBert(synthetic_state_dict(BERT_BASE), EMB, torch.device("cuda"))
res = []
for B, S, T in t.EDGES:
    mask, r = t._edge_results(N, w, B, S, T, 0xFF)
    row = {}
    for c in (False, True):
        try:
            t._assert_same(r[(True, c)], r[(False, c)], mask, True, c, ("packed vs padded", B, S, T, c))
            row[c] = "ok"
        except AssertionError as e:
            row[c] = repr(e)[:500]
    res.append(((B, S, T), row))
torch.save(res, sys.argv[2])
"""


def test_row_count_edges_without_the_fused_layernorm(N, tmp_path):
    """MEMVUL_FUSED_LN=0 (the operator fallback: GEMM + stand-alone LayerNorm over all B*S rows) keeps the guarantee.
    The switch is read once per process, so the cases run in a child."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("MEMVUL_")}
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(tmp_path / "out.pt")],
                       env=dict(env, MEMVUL_FUSED_LN="0"), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    res = torch.load(tmp_path / "out.pt")
    assert len(res) == len(EDGES)
    failed = [(case, row) for case, row in res if any(v != "ok" for v in row.values())]
    assert not failed, failed


# ------------------------------------------------------------------------------------------------ realistic reuse
def _batch(ids, mask):
    return {"tokens": {"token_ids": ids, "mask": mask, "type_ids": torch.zeros_like(ids)}}


def _lens_with(B, S, T, last, seed):
    """B lengths in [1, S] summing to T, the longest equal to S (batches are padded to their longest member) and the
    last equal to ``last``."""
    lens = _split(T - last - S, B - 2, S, seed) if B > 2 else []
    lens = [S] + lens + [last]
    assert sum(lens) == T and max(lens) == S
    return lens


def test_model_memory_reuses_its_workspace_across_batch_shapes(N):
    """ModelMemory keeps one workspace per embedder and reuses it for every batch shape (the bank in chunks of 128,
    then query batches padded to their own longest member).  Every batch must give what a zeroed workspace gives.

    The stream includes a sequence that places stale fp32 bits under rows the next call reads: 64 x 512 allocates the
    workspace; 64 x 128 (cls_only, packed) writes its fp32 [CLS] residual rows x32_cls; 64 x 256 with T = 8200 then
    has the rows [T, round_up(T, 256)) of its attention output ctx on those bytes, and its last report (100 tokens)
    has a ragged key block that reads rows past T."""
    from memvul_b200.synthetic import BERT_BASE, build_memory_model
    model, _ = build_memory_model(BERT_BASE, device="cuda")
    ref, _ = build_memory_model(BERT_BASE, device="cuda")
    emb, ref_emb = model.embedder, ref.embedder
    flags = N.encoder_flags(emb.packed(), True, True)           # ModelMemory: cls_only, packed

    def fresh_workspace(B, S):
        ref_emb._workspace = torch.zeros(ref_emb.packed().workspace_bytes(B, S, flags), dtype=torch.uint8, device="cuda")

    rng = random.Random(5)
    anchors = [(128, 256), (128, 96), (7, 300)]                 # the bank: 263 anchors in chunks of at most 128
    meta = lambda n: [{"type": "golden", "instance": [{"label": f"CWE-{i}"}]} for i in range(n)]
    with torch.no_grad():
        for i, (B, S) in enumerate(anchors):
            lens = [S] + [rng.randint(1, S) for _ in range(B - 1)]
            ids, mask = _ids(lens, S, 30522, seed=100 + i)
            model.forward_gold_instances(_batch(ids, mask), meta(B))
            fresh_workspace(B, S)
            ref.forward_gold_instances(_batch(ids, mask), meta(B))
    assert torch.equal(model._golden_instances_embeddings, ref._golden_instances_embeddings)

    queries = [(64, 512, _lens_with(64, 512, 20000, 333, 1)),
               (64, 128, _lens_with(64, 128, 5000, 77, 2)),
               (64, 256, _lens_with(64, 256, 8200, 100, 3))]
    for i, (B, S) in enumerate([(16, 384), (64, 64), (8, 512), (33, 200), (64, 256), (5, 40), (64, 128), (17, 511)]):
        queries.append((B, S, [S] + [rng.randint(1, S) for _ in range(B - 1)]))

    # the stale bytes of the second batch lie under ctx rows [T, round_up(T, 256)) of the third
    x32_cls_off, x32_cls_n = _layout(N, emb.packed(), 64, 128, flags)["x32_cls"]
    ctx_off = _layout(N, emb.packed(), 64, 256, flags)["ctx"][0]
    row = 2 * emb.packed().hidden
    lo, hi = ctx_off + 8200 * row, ctx_off + 8448 * row
    assert lo < x32_cls_off + x32_cls_n and x32_cls_off < hi

    ws_ptr = None
    for qi, (B, S, lens) in enumerate(queries):
        _layout(N, emb.packed(), B, S, flags)
        ids, mask = _ids(lens, S, 30522, seed=200 + qi)
        with torch.no_grad():
            got = model.match_batch(_batch(ids, mask))
            fresh_workspace(B, S)
            want = ref.match_batch(_batch(ids, mask))
        if qi < 3:                                              # the first three batches share one allocation
            ws_ptr = ws_ptr or emb._workspace.data_ptr()
            assert emb._workspace.data_ptr() == ws_ptr
        # (a NaN [CLS] row need not show as NaN here: the header's ReLU maps NaN to 0, so compare every value)
        for k in ("logits", "probs", "best_probs"):
            assert bool(torch.isfinite(got[k]).all()), (qi, B, S, k)
            assert torch.equal(got[k], want[k]), \
                (qi, B, S, k, "reports", torch.nonzero((got[k] != want[k]).reshape(B, -1).any(1)).flatten().tolist())
        assert torch.equal(got["best_idx"], want["best_idx"]), (qi, B, S)


def test_embedder_stream_of_random_shapes_tiny(N):
    """About 40 bert-tiny batches of random (B, S, lens, cls_only) through one embedder (one workspace, grown as
    needed) against the same call on a zeroed workspace."""
    from memvul_b200.custom_PTM_embedder import _PACKED_DEFAULT as packed
    from memvul_b200.synthetic import BERT_TINY, build_memory_model
    model, _ = build_memory_model(BERT_TINY, device="cuda")
    emb = model.embedder
    rng = random.Random(2021)
    for i in range(40):
        B, S = rng.choice([1, 2, 3, 7, 16, 33, 64, 100]), rng.randint(1, 512)
        lens = [rng.randint(1, S) for _ in range(B)]
        lens[rng.randrange(B)] = S
        cls_only = rng.random() < 0.5
        ids, mask = _ids(lens, S, 1024, seed=i)
        w = emb.packed()
        _layout(N, w, B, S, N.encoder_flags(w, cls_only, packed))
        with torch.no_grad():
            got = emb(ids, mask, None, cls_only=cls_only)
            emb.check_last_batch()
        want = _encode(N, w, ids, mask, packed, cls_only)
        _assert_same(got, want, mask, packed, cls_only, ("stream", i, B, S, cls_only))
