"""Kernels at adversarial value ranges, against float64 references computed on the same (fp16- or fp32-rounded) inputs.

Attention: Q and K are built so that the scores follow a chosen pattern instead of being random.  With a fixed
fp16-exact direction u (entries +-1, |u|^2 = 64) and q_i = a_i u + noise, k_j = (t_j / 8) u + noise, the score
q_i . k_j / 8 is about a_i t_j natural units.  The patterns reach the soft-max paths random inputs almost never do:
the lazy rescale of O (a row maximum that grows by more than 2^8 = 5.545 natural units over the stale one), rows of
one warp that do and do not grow, probabilities that underflow in fp16, scores of several hundred units, and a
single dominant key in a ragged last block.

Fused GEMM + LayerNorm: rows whose mean is large next to their spread (|mean| / std up to 20,000), where a
one-pass E[x^2] - mean^2 variance cancels catastrophically; the fused kernel must agree with a float64 LayerNorm,
with the unfused gemm_f16 + layernorm path and with the stand-alone LayerNorm kernels to within the cost of rounding
the fp32 pre-LN row itself."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BKV = 64                                              # keys per block of the attention kernels
PATTERNS = ["ramp5", "ramp6", "ramp15", "ramp40", "late_spike", "early_spike", "mixed_rows", "large"]
SEQS = [64, 65, 200, 511, 512]
SENTINEL = -1234.0                                    # fp16-exact; marks ctx rows the kernel must not write


@pytest.fixture(scope="module")
def N():
    from memvul_b200 import native
    native.build()
    return native


# ------------------------------------------------------------------------------------------------ attention inputs
def _lens(S):
    """[S, the longest length <= S with len % 64 == 1, the longest with len % 64 == 63]: one key alone in the last
    block, and a last block with a single masked column."""
    l1 = max(l for l in range(1, S + 1) if l % BKV == 1)
    l63 = max([l for l in range(1, S + 1) if l % BKV == 63] or [S])
    return [S, l1, l63]


def _levels(pattern, B, nH, S, lens, g):
    """(a [B,nH,S] per query row, t [B,nH,S] per key): score(i, j) ~= a_i t_j natural units."""
    j = torch.arange(S, dtype=torch.float64)
    blk = (j // BKV)[None, None, :].expand(B, nH, S)
    U = torch.rand(B, nH, S, generator=g, dtype=torch.float64)
    a = torch.ones(B, nH, S, dtype=torch.float64)
    last = torch.tensor(lens, dtype=torch.long)[:, None, None].expand(B, nH, 1) - 1       # each sequence's last key
    if pattern.startswith("ramp"):
        # block maximum = delta * block: one key per block sits exactly on it (column 17, or the block's first key when
        # the ragged last block is shorter), the rest up to 3 units below.  delta 5 stays under the 5.545 threshold
        # (the stale maximum is kept for one block, then the rescale runs); 6, 15, 40 rescale every block.
        delta = float(pattern[4:])
        top = (j % BKV == 17) | ((j % BKV == 0)[None, None, :] & (j[None, None, :] + 17 > last))
        t = delta * blk - 3.0 * U * (~top)
        a = 1.0 - 0.03 * torch.rand(B, nH, S, generator=g, dtype=torch.float64)          # growth per block in [0.97, 1] delta
    elif pattern == "late_spike":
        # one key, the LAST valid one (alone in its block when len % 64 == 1, next to the masked column when 63),
        # 60 units above all others: ctx ~= that key's V row
        t = torch.randn(B, nH, S, generator=g, dtype=torch.float64)
        t.scatter_(2, last.contiguous(), 60.0)
    elif pattern == "early_spike":
        # the maximum is in block 0; every later key sits >= 17 units below it, so its P underflows in fp16
        t = 20.0 + torch.randn(B, nH, S, generator=g, dtype=torch.float64).clamp(-3, 3)
        t[:, :, :BKV] = torch.randn(B, nH, min(S, BKV), generator=g, dtype=torch.float64).clamp(-3, 3)
        t.scatter_(2, last.clamp(max=5).contiguous(), 40.0)                             # key min(5, len - 1): block 0
    elif pattern == "mixed_rows":
        # ramp of 8 units per block; inside every 32-row warp the rows mix growing (a > 0: growth 0.4 ... 16 per block),
        # shrinking (a < 0: maximum in block 0), flat (a = 0) and tiny (a = 0.05)
        t = 8.0 * blk - 3.0 * U
        choices = torch.tensor([1.0, -1.0, 0.0, 0.05, 0.5, -0.3, 2.0, 0.7], dtype=torch.float64)
        i = torch.arange(S)
        a = choices[(i[None, None, :] * 5 + torch.arange(B)[:, None, None] + 3 * torch.arange(nH)[None, :, None]) % 8]
        a = a.expand(B, nH, S).clone()
    elif pattern == "large":
        # scores of +-300 units with near-ties: every key within 2 units of the maximum
        t = 300.0 - 2.0 * U
        a = torch.tensor([1.0, -1.0, 0.9], dtype=torch.float64)[torch.arange(S) % 3][None, None, :].expand(B, nH, S).clone()
    else:
        raise ValueError(pattern)
    return a, t


def _scored_qkv(pattern, B, S, H, lens, seed):
    """fp16 qkv [B*S, 3H] (padded layout; Q | K | V, heads of 64) with the score pattern of ``_levels`` in every
    (sequence, head); ``pattern`` may also be a list giving one pattern per sequence."""
    g = torch.Generator().manual_seed(seed)
    nH = H // 64
    pats = pattern if isinstance(pattern, list) else [pattern] * B
    a = torch.empty(B, nH, S, dtype=torch.float64)
    t = torch.empty(B, nH, S, dtype=torch.float64)
    for b, p in enumerate(pats):
        a[b:b + 1], t[b:b + 1] = _levels(p, 1, nH, S, lens[b:b + 1], g)
    u = torch.randint(0, 2, (B, nH, 1, 64), generator=g).double() * 2 - 1
    q = a[..., None] * u + 1e-3 * torch.randn(B, nH, S, 64, generator=g, dtype=torch.float64)
    k = (t / 8.0)[..., None] * u + 0.02 * torch.randn(B, nH, S, 64, generator=g, dtype=torch.float64)
    v = torch.randn(B, nH, S, 64, generator=g, dtype=torch.float64).clamp(-2.0, 2.0)
    qkv = torch.stack([q, k, v], 0).permute(1, 3, 0, 2, 4).reshape(B * S, 3 * H)           # [B, S, 3, nH, 64]
    return qkv.to(torch.float16)


def _attn_ref64(qkv, lens, B, S, H):
    """float64 softmax(Q K^T / 8 + (1 - mask) * -10000) V (transformers 4.1.0 key mask) on the given inputs (padded)."""
    nH = H // 64
    q, k, v = qkv.double().view(B, S, 3, nH, 64).permute(2, 0, 3, 1, 4)
    mask = torch.arange(S, device=qkv.device)[None, :] < lens[:, None]
    sc = q @ k.transpose(-1, -2) / 8.0 + (~mask).double()[:, None, None, :] * -10000.0
    ref = (torch.softmax(sc, -1) @ v).permute(0, 2, 1, 3).reshape(B * S, H)
    return ref, mask.reshape(-1), float(sc.masked_fill(~mask[:, None, None, :], 0.0).abs().max())


def _pack(qkv, lens, S):
    """The packed (var-len) layout of the same sequences: rows back to back, the tail of the B*S-row buffer holds
    unrelated finite values.  Returns (packed qkv, row_start int32 [B+1], index of each packed row in ``qkv``)."""
    B = len(lens)
    rows = torch.cat([torch.arange(l) + b * S for b, l in enumerate(lens)]).to(qkv.device)
    packed = (torch.randn(qkv.shape, generator=torch.Generator().manual_seed(7)) * 4).to(qkv.dtype).to(qkv.device)
    packed[:rows.numel()] = qkv[rows]
    rs = torch.zeros(B + 1, dtype=torch.int32)
    rs[1:] = torch.cumsum(torch.tensor(lens), 0)
    return packed, rs.to(qkv.device), rows


def _attention_into(N, fn, qkv, lens, B, S, H, row_start, fill):
    """The ABI call with a ctx buffer pre-filled with ``fill`` (the Python wrappers hand the kernel zeros)."""
    ctx = torch.full((qkv.shape[0], H), fill, dtype=qkv.dtype, device=qkv.device)
    with torch.cuda.device(qkv.device):
        N._check(fn(qkv.data_ptr(), lens.data_ptr(), N._ptr(row_start), ctx.data_ptr(), B, S, H,
                    torch.cuda.current_stream().cuda_stream))
    return ctx


def _check_attention(N, qkv, lens, B, S, H, tol, f32=False, pattern=None):
    """Padded and packed layouts against the float64 reference: finite, within ``tol`` on valid rows, the packed
    output equal bit for bit to the padded one on the same rows, and nothing written past the last packed token."""
    fn = N.lib().memvul_attention_f32 if f32 else N.lib().memvul_attention_f16
    lens_t = torch.tensor(lens, dtype=torch.int32, device="cuda")
    ref, valid, smax = _attn_ref64(qkv, lens_t, B, S, H)
    if f32:     # fp32 scores: one rounding at the score's magnitude, u |s|, moves ctx by up to |v_j - ctx| <= 4
        tol = tol + 4 * 2.0 ** -24 * smax
    ctx = _attention_into(N, fn, qkv, lens_t, B, S, H, None, 0.0)
    assert torch.isfinite(ctx[valid]).all()
    err = float((ctx.double() - ref)[valid].abs().max())
    assert err < tol, (pattern, "padded", err)
    packed, rs, rows = _pack(qkv, lens, S)
    T = rows.numel()
    ctx_p = _attention_into(N, fn, packed, lens_t, B, S, H, rs, SENTINEL)
    assert torch.isfinite(ctx_p[:T]).all()
    err_p = float((ctx_p[:T].double() - ref[rows]).abs().max())
    assert err_p < tol, (pattern, "packed", err_p)
    assert torch.equal(ctx_p[:T], ctx[rows]), (pattern, float((ctx_p[:T].double() - ctx[rows].double()).abs().max()))
    assert bool((ctx_p[T:] == SENTINEL).all()), (pattern, "rows past the last packed token were written")
    return ctx


# fp16 P and fp16 output with |V| <= 2: the bound of tests/test_kernels_gpu.py::test_attention_tcgen05
TOL_F16 = 4e-3
# fp32 scores of 64-term dot products with |score| up to ~10: the bound of tests/test_precise_gpu.py::test_attention_f32;
# _check_attention adds the rounding of larger scores (4 u max|score|: 6.7e-5 at the 280 units of ramp40)
TOL_F32 = 3e-5


@pytest.mark.parametrize("H", [128, 768])
@pytest.mark.parametrize("S", SEQS)
@pytest.mark.parametrize("pattern", PATTERNS)
def test_attention_score_patterns(N, pattern, S, H):
    lens = _lens(S)
    qkv = _scored_qkv(pattern, 3, S, H, lens, seed=S * 31 + H + PATTERNS.index(pattern)).cuda()
    ctx = _check_attention(N, qkv, lens, 3, S, H, TOL_F16, pattern=pattern)
    if pattern == "late_spike":                       # one key dominates by e^58: ctx is that key's V row
        for b, L in enumerate(lens):
            vrow = qkv[b * S + L - 1, 2 * H:].float()
            assert float((ctx[b * S:b * S + L].float() - vrow).abs().max()) < TOL_F16


@pytest.mark.parametrize("H", [128, 768])
@pytest.mark.parametrize("S", SEQS)
@pytest.mark.parametrize("pattern", PATTERNS)
def test_attention_f32_score_patterns(N, pattern, S, H):
    lens = _lens(S)
    qkv = _scored_qkv(pattern, 3, S, H, lens, seed=S * 31 + H + PATTERNS.index(pattern)).cuda().float()
    _check_attention(N, qkv, lens, 3, S, H, TOL_F32, f32=True, pattern=pattern)


def _many_items():
    """B=40, S=512, H=768: 40 x 12 heads x 4 query tiles = 1,920 work items per launch (> 3 x 148 SMs), so every
    persistent CTA runs several items back to back, with the patterns alternating from one sequence to the next."""
    B, S, H = 40, 512, 768
    lens = [[512, 449, 511, 257, 1, 63, 320, 128][b % 8] for b in range(B)]
    pats = [PATTERNS[(b * 3) % len(PATTERNS)] for b in range(B)]
    return pats, B, S, H, lens


@pytest.mark.parametrize("f32", [False, True])
def test_attention_patterns_across_work_items(N, f32):
    pats, B, S, H, lens = _many_items()
    qkv = _scored_qkv(pats, B, S, H, lens, seed=11).cuda()
    _check_attention(N, qkv.float() if f32 else qkv, lens, B, S, H, TOL_F32 if f32 else TOL_F16, f32=f32)


_CHILD = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from memvul_b200 import native as N
cases = torch.load(sys.argv[2])
out = []
for c in cases:
    rs = c["row_start"].cuda() if c["row_start"] is not None else None
    out.append(N.attention_f16(c["qkv"].cuda(), c["lens"].cuda(), c["B"], c["S"], c["H"], row_start=rs).cpu())
torch.save(out, sys.argv[3])
"""


def test_attention_kernel_switch_is_bit_identical(N, tmp_path):
    """MEMVUL_ATT_V=1 (the two-CTA kernel with speculative exponentials) and the default three-stream kernel give the
    same bits on the adversarial patterns.  The switch is read once per process, so each kernel runs in a child."""
    pats, B, S, H, lens = _many_items()
    big = _scored_qkv(pats, B, S, H, lens, seed=11)
    packed, rs, rows = _pack(big, lens, S)
    cases = [dict(qkv=big, lens=torch.tensor(lens, dtype=torch.int32), row_start=None, B=B, S=S, H=H),
             dict(qkv=packed.cpu(), lens=torch.tensor(lens, dtype=torch.int32), row_start=rs.cpu(), B=B, S=S, H=H)]
    for p in ("ramp5", "mixed_rows", "late_spike"):
        l3 = _lens(200)
        cases.append(dict(qkv=_scored_qkv(p, 3, 200, 128, l3, seed=5), lens=torch.tensor(l3, dtype=torch.int32),
                          row_start=None, B=3, S=200, H=128))
    torch.save(cases, tmp_path / "in.pt")
    env = {k: v for k, v in os.environ.items() if not k.startswith("MEMVUL_ATT_")}
    outs = {}
    for ver in ("3", "1"):
        r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(tmp_path / "in.pt"), str(tmp_path / f"out{ver}.pt")],
                           env=dict(env, MEMVUL_ATT_V=ver), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        outs[ver] = torch.load(tmp_path / f"out{ver}.pt")
    for i, c in enumerate(cases):
        lens_t = c["lens"].cuda()
        if c["row_start"] is None:
            ref, valid, _ = _attn_ref64(c["qkv"].cuda(), lens_t, c["B"], c["S"], c["H"])
            valid = valid.cpu()
            for ver in ("3", "1"):
                err = float((outs[ver][i].double() - ref.cpu())[valid].abs().max())
                assert err < TOL_F16, (i, ver, err)
        else:
            T = rows.numel()
            for ver in ("3", "1"):
                assert torch.equal(outs[ver][i][:T], outs[ver][0][rows.cpu()]), (i, ver)
        assert torch.equal(outs["3"][i], outs["1"][i]), \
            (i, float((outs["3"][i].double() - outs["1"][i].double()).abs().max()))


# ------------------------------------------------------------------------------------------------ LayerNorm
MUS = [0.0, 10.0, -10.0, 100.0, -100.0, 1000.0, -1000.0]
SIGMAS = [1.0, 0.05]
U_RND = 2.0 ** -24                                     # fp32 unit roundoff


def _ill_rows(M, H, g):
    """fp32 [M, H]: row r = sigma_r * N(0,1) + mu_r, (mu, sigma) cycling through all 14 pairs every 14 rows, so every
    32-row strip and 256-row tile mixes well- and ill-conditioned rows."""
    r = torch.arange(M)
    mu = torch.tensor(MUS, dtype=torch.float64)[r % len(MUS)]
    sg = torch.tensor(SIGMAS, dtype=torch.float64)[(r // len(MUS)) % len(SIGMAS)]
    return (torch.randn(M, H, generator=g, dtype=torch.float64) * sg[:, None] + mu[:, None]).float()


def _ln64(x, gamma, beta, eps=1e-12):
    x = x.double()
    m = x.mean(1, keepdim=True)
    var = ((x - m) ** 2).mean(1, keepdim=True)
    return (x - m) / torch.sqrt(var + eps) * gamma.double() + beta.double()


def _row_tol(x64):
    """Per-row bound: 2e-4 plus 8 unit roundoffs of |mean| / std -- what rounding the fp32 pre-LN row itself costs
    once it is normalised (an error of u |mean| in any element or in the mean becomes u |mean| / std)."""
    m = x64.mean(1)
    sd = torch.sqrt(((x64 - m[:, None]) ** 2).mean(1))
    return 2e-4 + 8 * U_RND * m.abs() / sd


def _assert_rows(out, ref, tol, what):
    err = (out.double() - ref).abs().amax(1)
    bad = err > tol
    worst = int(torch.argmax(err / tol))
    assert not bool(bad.any()), (what, int(bad.sum()), "rows fail; worst row", worst, float(err[worst]), float(tol[worst]))


@pytest.mark.parametrize("M,K", [(1000, 768), (1000, 3072), (8000, 768), (8000, 3072)])
def test_gemm_layernorm_ill_conditioned_rows(N, M, K):
    """K <= 1024 runs with the third residual buffer, K = 3072 with the four-stage ring; M = 1000 / 8000 end in a ragged
    256-row tile, 8000 gives clusters several tiles each.  The GEMM part is kept small (std ~0.02) so that a row's
    spread is its residual's."""
    g = torch.Generator().manual_seed(M + K)
    a = torch.randn(M, K, generator=g).half().cuda()
    w = (torch.randn(768, K, generator=g) * (0.02 / K ** 0.5)).half().cuda()
    bias = (torch.randn(768, generator=g) * 0.02).cuda()
    resid = _ill_rows(M, 768, g).cuda()
    gamma = (1 + 0.1 * torch.randn(768, generator=g)).cuda()
    beta = (0.1 * torch.randn(768, generator=g)).cuda()
    x64 = a.double() @ w.double().T + bias.double() + resid.double()
    ref = _ln64(x64, gamma, beta)
    tol = _row_tol(x64)
    x32, x16 = N.gemm_ln_f16(a, w, bias, resid, gamma, beta)
    assert torch.isfinite(x32).all() and torch.isfinite(x16.float()).all()
    _assert_rows(x32, ref, tol, "fused x32")
    _assert_rows(x16, ref, 4e-3 + (tol - 2e-4), "fused x16")        # fp16 output rounding at |y| < 8
    # the unfused path of the same operation: fp32 GEMM + residual epilogue, then the two-pass LayerNorm kernel
    y = N.gemm_f16(a, w, bias, N.EPI_BIAS_RESID_F32, resid=resid)
    z32, _ = N.layernorm(y, gamma, beta)
    _assert_rows(x32, z32.double(), tol, "fused vs gemm_f16 + layernorm")
    buf = resid.clone()
    y32, y16 = N.gemm_ln_f16(a, w, bias, buf, gamma, beta, inplace=True)
    assert torch.equal(y32, x32) and torch.equal(y16, x16)          # deterministic, in place == out of place


@pytest.mark.parametrize("H", [768, 128])
def test_layernorm_ill_conditioned_rows(N, H):
    """The stand-alone two-pass kernel meets the same per-row bound on the same kind of rows."""
    g = torch.Generator().manual_seed(H)
    y = _ill_rows(1000, H, g).cuda()
    gamma = (1 + 0.1 * torch.randn(H, generator=g)).cuda()
    beta = (0.1 * torch.randn(H, generator=g)).cuda()
    x32, x16 = N.layernorm(y, gamma, beta)
    ref = _ln64(y, gamma, beta)
    tol = _row_tol(y.double())
    _assert_rows(x32, ref, tol, "layernorm x32")
    _assert_rows(x16, ref, 4e-3 + (tol - 2e-4), "layernorm x16")


def test_embed_layernorm_ill_conditioned_rows(N):
    """Embedding sum + LayerNorm with word-embedding rows of large mean and small spread."""
    from memvul_b200.synthetic import BERT_TINY, EMB, synthetic_state_dict
    sd = synthetic_state_dict(BERT_TINY)
    e = EMB + "embeddings."
    g = torch.Generator().manual_seed(3)
    Hh = BERT_TINY.hidden
    sd[e + "word_embeddings.weight"] = _ill_rows(BERT_TINY.vocab_size, Hh, g)
    sd[e + "position_embeddings.weight"] = torch.randn(BERT_TINY.max_pos, Hh, generator=g) * 0.01
    sd[e + "token_type_embeddings.weight"] = torch.randn(2, Hh, generator=g) * 0.01
    w = N.PackedBert(sd, EMB, torch.device("cuda"))
    B, S = 6, 128
    ids = torch.randint(0, BERT_TINY.vocab_size, (B, S), generator=g)
    tids = torch.randint(0, 2, (B, S), generator=g)
    x32, _ = N.embed_layernorm(w, ids.cuda(), tids.cuda())
    x64 = (sd[e + "word_embeddings.weight"][ids].double() + sd[e + "position_embeddings.weight"][:S][None].double()
           + sd[e + "token_type_embeddings.weight"][tids].double()).reshape(B * S, Hh)
    ref = _ln64(x64, sd[e + "LayerNorm.weight"], sd[e + "LayerNorm.bias"])
    _assert_rows(x32.cpu(), ref, _row_tol(x64), "embed_layernorm x32")
