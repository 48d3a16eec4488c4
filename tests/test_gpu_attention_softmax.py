"""Every attention kernel against a float64 softmax on growing, peaked and masked score patterns.

Random q/k at scale D**-0.5 give scores of about N(0, 1): no row maximum ever moves much, and a key
that leaks past a mask moves the output by about |v| / n, below any practical tolerance.  The
inputs here are built so that those mistakes move the output by a lot.

Score patterns.  Per KV head a unit direction u (a row of the Sylvester-Hadamard matrix over
sqrt(D), so q = +-u * sqrt(D) has entries +-1); key j is ``c_j u + noise``, noise orthogonal to u,
with c_j chosen so that the scaled score ``s * scale * log2(e)`` of a query along +u follows a
chosen shape (units below: log2 of the scaled score):

* ``stair:<step>`` - score = step * floor(key / 64): every 64-key tile beats the previous maximum
  by ``step``: 7.75 stays under the lazy-rescale threshold of the tcgen05 kernel (2^8), 9 and 30
  cross it on every tile (30: earlier tiles underflow to exact zeros).  8 - 1/16 and 8 + 1/16 sit
  on the threshold: bf16 rounding of the keys moves a tile's maximum by about +-0.15, so rows
  land on either side of it from tile to tile.
* ``ramp`` - score = 9/64 * key: each causal row's maximum sits on its own diagonal.
* ``spike:<where>`` - one key +40 above a flat background (tile, page, split and row edges).
* ``sink`` - key 0 and one key of the last tile at +40 / +40.75, the rest flat.
* ``mixed`` - stair:9, with the query heads of a KV group along +u, -u, +u/2 and a direction
  orthogonal to u: growing and non-growing rows in one warp.
* ``hot`` / ``cold`` - every score near +1000 / -1000: no overflow, underflow or NaN.
* ``decoy`` - keys a row must not see score +60 above everything visible and carry V = +-256:
  slots >= ctx of the last page, whole pages past ctx that are still in the block table and, for
  causal prefill, the causal future (a ramp of 1/4 per key: a row's weight sits on its last few
  keys, and a one-key leak takes about 1/6 of it, moving the result by about 40).

The referee, ``attention_fp64``, gathers the pages through the block table and computes scores,
softmax and P V in float64 from the exact bf16 / f32 input values.

Tolerance, per output element, for bf16 outputs (f32 in brackets):

    |got - ref| <= 2^-8 |ref|  +  (2^-8 + n * 2^-23 + E_s) * Vmax        [1e-5 |ref|, 2^-20 Vmax]

* Vmax: the largest |v| over the keys that row may see (decoys the row must not see are left out,
  or a leak would widen its own bound).
* 2^-8 |ref|: one rounding of the output (2^-9) with a factor 2 of margin.
* 2^-8 Vmax: P stored in bf16 before P V (2^-9 per weight, at most 2^-9 Vmax on a weighted mean;
  2^-8 when the row sum is taken from the rounded weights), with margin.
* n * 2^-23 Vmax: the fp32 sums of O and of the row sum over the row's n visible keys
  (n * 2^-24 each; 2^-10 Vmax at the longest table here, 8192 keys).
* E_s = 2.2 ln2 * sum_j w_j delta_j: the fp32 score.  A perturbation delta_j (log2 units) of the
  scores moves a softmax mean by at most 2 ln2 sum_j w_j delta_j Vmax (first order; 2.2 covers the
  rest); ex2.approx adds 2^-22 relative (2^-21.5 log2 units).  With A_j = scale log2(e) sum_i
  |q_i k_ij| and S_j the scaled score:
  - CUDA-core kernels (paged_gqa_kernel, row-wise, dense decode) round q * scale * log2(e), each
    product and each partial sum: delta_j = (D + 2) 2^-24 A_j.
  - Tensor-core kernels (tcgen05, mma.sync, the fused decode) sum the exact bf16 products q_i k_ij
    in fp32.  Every product is a multiple of 2^e, e the sum of the last-bit exponents of the row's
    q and the key's k; where sum_i |q_i k_ij| < 2^(e + 24) (checked per row and key) every addend
    and partial sum is such a multiple below 2^(e + 24), which 24 significant bits aligned at the
    largest addend hold exactly, so the raw score is exact in any summation order.  Only the scale
    and the subtraction of the row maximum round: delta_j = 2^-23 (A_j + max_k A_k).  Keys that fail the check get the
    CUDA-core bound.
  The patterns are shifted so that the keys that carry a +u row's weight score near 0; there E_s is
  2^-13.6.  The cases where E_s is largest, computed from the inputs (the widening of the budget
  this term makes is accepted there):
  - ``hot`` / ``cold`` (every |S| ~ 1000, the largest scores used) on the CUDA-core routes:
    E_s = 2^-6.4 (D 64: 2^-7.4), so their budget is about (2^-8 + 2^-6.4) Vmax = 4 * 2^-8 Vmax.
    These two patterns check for overflow, underflow and NaN, which the budget still catches.  On
    the tensor-core routes the sums are exact and E_s = 2^-11.4.
  - ``mixed`` on the CUDA-core routes: the -u head's weight sits on the earliest keys, at
    |S| = 9 ctx / 64: E_s = 2^-7.2 over 4000 keys (page 16), 2^-9.9 over 700.
  - everything else: at most 2^-10.5 (stair:30 over the 4096-key prefill).
  The f32 routes see the same E_s and n * 2^-23 terms, which dominate their 2^-20.

``decode_attention_fused`` computes q itself (RMSNorm -> RoPE).  Its inputs are +-3 per element
with unit norm weights at position 0: RMSNorm gives +-1 exactly (+-3 / sqrt(9 + eps) rounds to
+-1 in bf16) and RoPE at position 0 is the identity in the kernel (sincosf(0) = (0, 1)) and in the
oracle, so the kernel's q equals the oracle's q bit for bit and the q-rounding term of its bound
is zero; ``test_fused_decode_query_is_exact_at_position_zero`` pins that on the CPU.  Its scores
stay within 64 log2 units.
"""

from __future__ import annotations

import math
import zlib
from dataclasses import dataclass

import pytest
import torch

from oracle import ops as oracle

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
LN2 = math.log(2.0)
LOG2E = 1.0 / LN2
SIGMA = 0.5  # per-element noise of the keys, orthogonal to u
STAIR_STEPS = (7.75, 8 - 1 / 16, 8 + 1 / 16, 9.0, 30.0)


# ------------------------------------------------------------------------------ fp64 referee --
def _quantum_exp(x):
    """Exponent of the last mantissa bit of each bf16 value (x = m 2^e, |m| < 2^8); +inf for zeros."""
    _, e = torch.frexp(x)
    return torch.where(x == 0, torch.full_like(x, math.inf), (e - 8).to(x.dtype))


def _fp64(q, kp, vp, bt, cl, scale, causal, Hkv, Hq, device=None, mma=False):
    """float64 attention plus, per output row, what its error budget needs: (out, Vmax, E_s, n).
    ``mma``: the kernel sums the bf16 products q_i k_i on tensor cores and scales afterwards."""
    device = torch.device(device) if device is not None else q.device
    rows, L, D = q.shape
    B, G, page = rows // Hq, Hq // Hkv, kp.shape[2]
    out = torch.zeros(B, Hq, L, D, dtype=F64, device=device)
    vmax = torch.zeros(B, Hq, L, dtype=F64, device=device)
    e_s = torch.zeros(B, Hq, L, dtype=F64, device=device)
    n_vis = torch.zeros(B, Hq, L, dtype=F64, device=device)
    bt_rows, ctxs = bt.cpu().tolist(), cl.cpu().tolist()
    for b in range(B):
        ctx = int(ctxs[b])
        if ctx == 0:
            continue  # an idle request: exact zeros
        ids = torch.tensor(bt_rows[b][: -(-ctx // page)], dtype=torch.int64, device=kp.device)
        k = kp[ids].to(device=device, dtype=F64).permute(1, 0, 2, 3).reshape(Hkv, -1, D)[:, :ctx]
        v = vp[ids].to(device=device, dtype=F64).permute(1, 0, 2, 3).reshape(Hkv, -1, D)[:, :ctx]
        qb = q[b * Hq : (b + 1) * Hq].to(device=device, dtype=F64).reshape(Hkv, G, L, D)
        s = (qb @ k.transpose(-1, -2)[:, None]) * scale  # [Hkv, G, L, ctx]
        # bottom-right causal alignment: row l sees keys < min(ctx, ctx - L + l + 1)
        vis = torch.full((L,), ctx, device=device)
        if causal:
            vis = torch.clamp(ctx - L + 1 + torch.arange(L, device=device), max=ctx)
        hidden = torch.arange(ctx, device=device)[None, :] >= vis[:, None]  # [L, ctx]
        p = torch.softmax(s.masked_fill(hidden, -math.inf), dim=-1)
        out[b] = (p @ v[:, None]).reshape(Hq, L, D)
        vabs = v.abs().amax(-1)[:, None, None, :].expand(Hkv, G, L, ctx)
        vmax[b] = vabs.masked_fill(hidden, 0).amax(-1).reshape(Hq, L)
        raw = qb.abs() @ k.abs().transpose(-1, -2)[:, None]  # sum_i |q_i k_ij|
        a = raw * (scale * LOG2E)
        delta = (D + 2) * 2.0**-24 * a  # D products and sums rounded in fp32, then the scale
        if mma:
            # every product is a multiple of 2^e (e: last-bit exponents of the row's q and the key's k);
            # with sum_i |q_i k_ij| < 2^(e + 24) every addend and partial sum is such a multiple below
            # 2^(e + 24), which 24 significant bits aligned at the largest addend hold exactly: the raw
            # score is exact in any summation order, and only the scale and the subtraction of the row
            # maximum round (2^-24 |S_j| + 2^-24 |S_j - m| <= 2^-23 (A_j + A_max))
            e = _quantum_exp(qb).amin(-1)[..., None] + _quantum_exp(k).amin(-1)[:, None, None, :]
            exact = raw < torch.exp2(e + 24)
            a_max = a.masked_fill(hidden, 0).amax(-1, keepdim=True)
            delta = torch.where(exact, 2.0**-23 * (a + a_max), delta)
        delta = delta + 2.0**-21.5  # ex2.approx: 2^-22 relative
        e_s[b] = (2.2 * LN2 * (p * delta).sum(-1)).reshape(Hq, L)
        n_vis[b] = vis.to(F64)[None, None, :].expand(Hkv, G, L).reshape(Hq, L)
    return out.reshape(rows, L, D), vmax.reshape(rows, L), e_s.reshape(rows, L), n_vis.reshape(rows, L)


def attention_fp64(q, kp, vp, bt, cl, scale, causal, Hkv, Hq, device=None):
    """softmax(q K^T * scale) V in float64 over the pages of ``bt`` (q [B*Hq, L, D], pages
    [P, Hkv, page, D]); bottom-right causal alignment; idle requests (ctx == 0) give zeros."""
    return _fp64(q, kp, vp, bt, cl, scale, causal, Hkv, Hq, device)[0]


def assert_within_budget(got, q, kp, vp, bt, cl, scale, causal, Hkv, Hq, what="", device=None, mma=False):
    """``got`` [B*Hq, L, D] against the float64 referee within the budget of the module docstring."""
    ref, vmax, e_s, n = _fp64(q, kp, vp, bt, cl, scale, causal, Hkv, Hq, device, mma)
    got = got.to(device=ref.device, dtype=F64).reshape(ref.shape)
    rel, vterm = (1e-5, 2.0**-20) if q.dtype == F32 else (2.0**-8, 2.0**-8)
    bound = rel * ref.abs() + ((vterm + n * 2.0**-23 + e_s) * vmax)[..., None]
    err = (got - ref).abs()
    bad = ~(err <= bound)  # NaN fails too
    if bool(bad.any()):
        worst = int(torch.argmax(torch.where(bad, err - bound, torch.zeros_like(err)).flatten().nan_to_num(math.inf)))
        r, l, d = (worst // (ref.shape[1] * ref.shape[2]), (worst // ref.shape[2]) % ref.shape[1], worst % ref.shape[2])
        raise AssertionError(
            f"{what}: {int(bad.sum())} of {bad.numel()} outputs outside the budget; worst at row {r} (request "
            f"{r // Hq}, head {r % Hq}), l {l}, d {d}: got {float(got[r, l, d]):.6g}, ref {float(ref[r, l, d]):.6g}, "
            f"bound {float(bound[r, l, d]):.3g}, Vmax {float(vmax[r, l]):.3g}"
        )


# ---------------------------------------------------------------------------- score patterns --
def hadamard(n):
    h = torch.ones(1, 1, dtype=F64)
    while h.shape[0] < n:
        h = torch.cat([torch.cat([h, h], 1), torch.cat([h, -h], 1)], 0)
    return h


def pattern_scores(pattern, ctx, L, page, N, causal):
    """Target scaled scores (log2 units) of the N table keys of one request for a query along +u,
    and which keys carry V = +-256."""
    key = torch.arange(N, dtype=F64)
    s = torch.zeros(N, dtype=F64)
    loud = torch.zeros(N, dtype=torch.bool)
    if ctx == 0:
        return s, loud
    top = ctx - 1
    name, _, arg = pattern.partition(":")
    if name in ("stair", "mixed"):
        step = float(arg) if name == "stair" else 9.0
        s = step * torch.floor(key / 64)
        s = s - s[top]
    elif name == "ramp":
        s = 9 / 64 * key
        s = s - s[top]
    elif name == "spike":
        pos = {"last": top, "page-1": page - 1, "page": page}.get(arg)
        pos = int(arg) if pos is None else pos
        assert pos < ctx
        s[pos] = 40.0
    elif name == "sink":
        s[0] = 40.0
        s[top - (top % 64) // 2] = 40.75  # inside the last tile
    elif name in ("hot", "cold"):
        s[:] = 1000.0 if name == "hot" else -1000.0
    elif name == "decoy":
        loud[ctx:] = True  # slots >= ctx of the last page, and whole pages past ctx
        s[ctx:] = 60.0 + L
        if causal and L > 1:  # the causal future: row l must not see keys > ctx - L + l
            fut = key > ctx - L
            loud |= fut & (key < ctx)
            s = torch.where(fut & (key < ctx), 60.0 + (key - (ctx - L)) / 4, s)
    else:
        raise ValueError(pattern)
    return s, loud


def directions(D, Hkv):
    h = hadamard(D)
    u = h[1 : 1 + Hkv] / math.sqrt(D)  # per KV head, unit
    perp = h[1 + Hkv : 1 + 2 * Hkv] / math.sqrt(D)  # orthogonal to every u
    return u, perp


def query_coefs(pattern, G):
    """Coefficient of u for each query head of a group (None: orthogonal to u)."""
    if pattern == "mixed":
        return [(1.0, -1.0, 0.5, None)[g % 4] for g in range(G)]
    return [1.0] * G


def make_keys(scores, u, g):
    """Keys ``c u + noise`` ([..., N, D]) whose score against ``sqrt(D) u`` at scale D**-0.5 is ``scores``."""
    D = u.shape[-1]
    n = SIGMA * torch.randn(*scores.shape, D, generator=g, dtype=F64)
    n -= (n * u).sum(-1, keepdim=True) * u
    return (scores * LN2)[..., None] * u + n


@dataclass(frozen=True)
class Case:
    name: str
    kernel: str  # the __global__ this shape selects (checked by test_each_route_runs_the_kernel_its_cases_target)
    ctxs: tuple
    L: int
    Hq: int = 8
    Hkv: int = 2
    page: int = 128
    width: int = 0  # block-table width in pages (0: just enough for the longest context)
    causal: bool = True
    dtype: torch.dtype = BF16
    D: int = 128
    patterns: tuple = ()  # a subset of the patterns (large inputs); empty: all
    absent: tuple = ()  # kernels this shape must not launch (checked by the route test)

    @property
    def mma(self):
        """The tcgen05 and mma.sync kernels sum bf16 products on tensor cores; the CUDA-core
        kernels (paged_gqa_kernel, row-wise) round q * scale * log2(e) before the products."""
        return self.name.startswith(("tc_", "fa_"))


def build(case, pattern, seed, device="cpu"):
    """(q [B*Hq, L, D], key pages, value pages, block table, context lengths) of ``case``; every
    table slot holds a real page, including the slots past a request's context."""
    g = torch.Generator().manual_seed(seed)
    B, G, D, page = len(case.ctxs), case.Hq // case.Hkv, case.D, case.page
    width = case.width or max(1, max(-(-c // page) for c in case.ctxs))
    N = width * page
    P = B * width + 1
    u, perp = directions(D, case.Hkv)
    s = torch.zeros(B, case.Hkv, N, dtype=F64)
    loud = torch.zeros(B, N, dtype=torch.bool)
    for b, ctx in enumerate(case.ctxs):
        sb, lb = pattern_scores(pattern, ctx, case.L, page, N, case.causal)
        s[b], loud[b] = sb, lb
    k = make_keys(s, u[None, :, None, :], g)  # [B, Hkv, N, D]
    v = torch.randn(B, case.Hkv, N, D, generator=g, dtype=F64)
    sign = torch.where(torch.rand(B, case.Hkv, N, D, generator=g) < 0.5, -1.0, 1.0).to(F64)
    v = torch.where(loud[:, None, :, None], 256.0 * sign, v)
    coefs = query_coefs(pattern, G)
    qh = torch.stack([perp if c is None else c * u for c in coefs], 1) * math.sqrt(D)  # [Hkv, G, D]
    q = qh.reshape(case.Hq, 1, D).expand(B, case.Hq, case.L, D).reshape(B * case.Hq, case.L, D)
    perm = torch.randperm(P, generator=g)
    bt = perm[: B * width].reshape(B, width).to(torch.int32)
    kp = torch.randn(P, case.Hkv, page, D, generator=g, dtype=F64)
    vp = torch.randn(P, case.Hkv, page, D, generator=g, dtype=F64)
    kp[bt.long()] = k.reshape(B, case.Hkv, width, page, D).transpose(1, 2)
    vp[bt.long()] = v.reshape(B, case.Hkv, width, page, D).transpose(1, 2)
    cl = torch.tensor(case.ctxs, dtype=torch.int32)
    dt = case.dtype
    return [t.to(device) for t in (q.to(dt).contiguous(), kp.to(dt), vp.to(dt), bt, cl)]


# ---------------------------------------------------------------------------------- the routes --
# tl::launch_paged_decode / launch_paged_prefill (attention_decode.cu) pick the kernel from the
# shape; each case's comment cites the condition that sends it where ``kernel`` says.
TC, GQA, MERGE, FA, ROW = "paged_prefill_tc_kernel", "paged_gqa_kernel", "paged_gqa_merge_kernel", "paged_prefill_fa_kernel", "paged_rowwise_kernel"
CASES = [
    # L <= 8, bf16, D 128, page % 64 == 0, G | 128, L <= 128 / G and a table of >= 1024 keys
    # (attention_decode.cu:565-569) -> tcgen05 kernel; split count from the cost model
    # (attention_prefill_tc.cu:516-539): one request over 8192 keys splits, 64 x 1024 does not.
    Case("tc_decode_1x8192", MERGE, (8192,), 1),
    Case("tc_decode_16x4096", TC, (4096,) * 13 + (0, 300, 4000), 1, page=64,  # one idle, one much shorter than the table
         patterns=("stair:8.0625", "stair:30", "ramp", "spike:64", "spike:last", "sink", "cold", "decoy")),
    Case("tc_decode_64x1024", TC, (1024,) * 63 + (1000,), 1, Hq=32, Hkv=8, page=256,
         patterns=("stair:9", "stair:30", "spike:last", "hot", "decoy"), absent=(MERGE,)),
    Case("tc_decode_L4_causal", TC, (3000, 1500), 4, page=128, width=24),
    # G = 16: RH = 128 / G = 8 rows per head, so one softmax warp holds the rows of four query heads
    # (+u, -u, +u/2 and orthogonal under ``mixed``)
    Case("tc_decode_G16", TC, (2048, 1111), 1, Hq=32, Hkv=2, page=128, patterns=("mixed", "stair:9", "ramp", "decoy")),
    # L <= 8, bf16, D 128, table < 1024 keys or page % 64 != 0 (:570-572) -> paged_gqa_kernel<RG>,
    # RG = G * L >= 3 ? 4 : G * L (:492); page 16 over 4000 keys splits (+ merge).
    Case("gqa_rg1", GQA, (500, 311), 1, Hq=4, Hkv=4, page=64, width=8),
    Case("gqa_rg2", GQA, (700, 64), 1, Hq=4, Hkv=2, page=32, width=30),
    Case("gqa_rg4_split_page16", MERGE, (4000,), 2, Hq=8, Hkv=2, page=16),
    Case("gqa_L8_causal", GQA, (700, 9), 8, Hq=8, Hkv=2, page=16, width=48),
    # L <= 8 with f32 or D != 128 (:573) -> paged_rowwise_kernel
    Case("rowwise_f32_d128", ROW, (500,), 1, page=64, dtype=F32),
    Case("rowwise_f32_d64", ROW, (300, 130), 2, page=32, width=12, dtype=F32, D=64),
    # L > 8, bf16, D 128, page % 64 == 0, G | 128 (:586-588) -> tcgen05 prefill
    Case("tc_prefill_4096", TC, (4096,), 4096, page=64),
    Case("tc_prefill_noncausal", TC, (300,), 300, page=128, causal=False),
    Case("tc_prefill_chunk_512_of_4096", TC, (4096,), 512, page=256),
    Case("tc_prefill_L100_G4", TC, (100, 350), 100, page=64, width=8),  # L not a multiple of 128 / G = 32
    Case("tc_prefill_G8", TC, (700,), 300, Hq=16, Hkv=2, page=64),  # RH = 16: two query heads per softmax warp
    # L > 8, page not a multiple of 64 or G not dividing 128 (:589-591) -> paged_prefill_fa_kernel
    Case("fa_page16", FA, (700,), 200, page=16),
    Case("fa_page32_noncausal", FA, (333, 200), 200, page=32, width=12, causal=False),
    Case("fa_g3", FA, (700,), 200, Hq=12, Hkv=4, page=64),
    # L > 8 with f32 (:595) -> paged_rowwise_kernel
    Case("rowwise_f32_prefill", ROW, (200,), 40, page=64, dtype=F32),
]
BY_NAME = {c.name: c for c in CASES}
PREFILL_PATTERNS = [f"stair:{s}" for s in STAIR_STEPS] + ["ramp", "mixed", "sink", "hot", "cold", "decoy"]
DECODE_PATTERNS = PREFILL_PATTERNS + ["spike:0", "spike:63", "spike:64", "spike:127", "spike:128", "spike:page-1", "spike:page", "spike:last"]


def patterns_for(case):
    pats = case.patterns or (DECODE_PATTERNS if case.L <= 8 else PREFILL_PATTERNS)
    short = min(c for c in case.ctxs if c > 0)
    keep = []
    for p in pats:
        if p.startswith("spike:") and p != "spike:last":
            pos = {"page-1": case.page - 1, "page": case.page}.get(p[6:])
            if (pos if pos is not None else int(p[6:])) >= short:
                continue
        keep.append(p)
    return keep


PAIRS = [(c.name, p) for c in CASES for p in patterns_for(c)]


# ------------------------------------------------------------------- CPU checks of the referee --
@pytest.mark.parametrize("dtype,causal,L", [(BF16, True, 1), (BF16, True, 16), (BF16, False, 5), (F32, True, 12), (F32, False, 1)])
def test_reference_matches_the_oracle_on_randn(dtype, causal, L):
    """Benign N(0, 1) scores: the float64 referee and the fp32 oracle agree to the oracle's rounding."""
    g = torch.Generator().manual_seed(L * 7 + int(causal))
    Hq, Hkv, D, page = 8, 2, 128, 32
    ctxs = [150, 0, 97]
    bt = torch.randperm(20, generator=g)[:15].reshape(3, 5).to(torch.int32)
    cl = torch.tensor(ctxs, dtype=torch.int32)
    q = torch.randn(3 * Hq, L, D, generator=g).to(dtype)
    kp = torch.randn(20, Hkv, page, D, generator=g).to(dtype)
    vp = torch.randn(20, Hkv, page, D, generator=g).to(dtype)
    got = oracle.paged_attention(q, kp, vp, bt, cl, D**-0.5, causal, Hkv, Hq)
    assert_within_budget(got, q, kp, vp, bt, cl, D**-0.5, causal, Hkv, Hq, "oracle")
    ref = attention_fp64(q, kp, vp, bt, cl, D**-0.5, causal, Hkv, Hq)
    assert torch.count_nonzero(ref[Hq : 2 * Hq]) == 0, "idle request must be exact zeros"


def test_reference_causal_alignment_and_page_gather_by_hand():
    """Two keys per page, pages out of order: row l of L = 2 over ctx = 3 sees keys < 2 + l."""
    D = 4
    kp = torch.zeros(3, 1, 2, D, dtype=F64)
    vp = torch.zeros(3, 1, 2, D, dtype=F64)
    for t, (pid, slot) in enumerate([(2, 0), (2, 1), (0, 0)]):  # logical token -> (page, slot)
        vp[pid, 0, slot] = float(t + 1)
    kp[0, 0, 1] = 1e3  # slot ctx of the last page: never visible
    vp[0, 0, 1] = -1e3
    bt = torch.tensor([[2, 0]], dtype=torch.int32)
    cl = torch.tensor([3], dtype=torch.int32)
    q = torch.zeros(1, 2, D, dtype=F64)
    out = attention_fp64(q, kp, vp, bt, cl, 1.0, True, 1, 1)
    assert out[0, 0].tolist() == [1.5] * D  # mean of tokens 0, 1
    assert out[0, 1].tolist() == [2.0] * D  # mean of tokens 0, 1, 2
    assert attention_fp64(q, kp, vp, bt, cl, 1.0, False, 1, 1)[0, 0].tolist() == [2.0] * D


@pytest.mark.parametrize("pattern", PREFILL_PATTERNS + ["spike:64", "spike:last"])
@pytest.mark.parametrize("causal,L", [(True, 1), (True, 24), (False, 3)])
def test_reference_matches_the_oracle_on_every_pattern(pattern, causal, L):
    """The patterns as the GPU tests use them, at CPU size: the fp32 oracle (the referee of the
    other attention tests) stays within the same budget as the kernels."""
    case = Case("cpu", "", (300, 0, 131), L, Hq=8, Hkv=2, page=64, width=6, causal=causal)
    q, kp, vp, bt, cl = build(case, pattern, seed=len(pattern) + L)
    got = oracle.paged_attention(q, kp, vp, bt, cl, 128**-0.5, causal, 2, 8)
    assert_within_budget(got, q, kp, vp, bt, cl, 128**-0.5, causal, 2, 8, f"oracle, {pattern}")


@pytest.mark.parametrize("pattern", ["stair:9", "ramp", "spike:64", "decoy"])
def test_patterns_have_the_intended_scores(pattern):
    """The scaled scores of the bf16 inputs follow the target shape to within the noise."""
    case = Case("cpu", "", (256,), 1, Hq=2, Hkv=1, page=64, width=5, causal=False)
    q, kp, vp, bt, cl = build(case, pattern, seed=3)
    k = kp[bt[0].long()].to(F64).reshape(-1, 128)
    s = (q[0, 0].to(F64) @ k.T) * 128**-0.5 * LOG2E
    want, loud = pattern_scores(pattern, 256, 1, 64, 320, False)
    assert (s - want).abs().max() < 0.5
    if pattern == "decoy":
        assert loud[256:].all() and not loud[:256].any()
        assert (vp[bt[0].long()].reshape(-1, 128)[256:].abs() == 256).all()


def test_fused_decode_query_is_exact_at_position_zero():
    """+-3 inputs, unit norm weight, position 0: the oracle's RMSNorm -> RoPE gives exactly +-1,
    which is what the fused kernel computes too (no q-rounding term in its bound)."""
    D = 128
    x = (3.0 * hadamard(D)[5]).to(BF16).reshape(1, 1, 1, D)
    w = torch.ones(D, dtype=BF16)
    q = oracle.rope(oracle.rms_norm(x, w, 1e-6), torch.zeros(1, dtype=torch.int32), D, 1e6)
    assert torch.equal(q.reshape(D), hadamard(D)[5].to(BF16))


# ------------------------------------------------------------------------------- GPU: paged --
def _ref_device(case):
    return "cuda" if case.L * max(case.ctxs) >= 1 << 20 else "cpu"


@pytest.mark.gpu
@pytest.mark.parametrize("name,pattern", PAIRS, ids=[f"{n}-{p}" for n, p in PAIRS])
def test_paged_attention_against_fp64(cuda_device, name, pattern):
    case = BY_NAME[name]
    q, kp, vp, bt, cl = build(case, pattern, seed=zlib.crc32(f"{name}/{pattern}".encode()), device=cuda_device)
    scale = case.D**-0.5
    got = ext().paged_attention(q, kp, vp, bt, cl, scale, is_causal=case.causal, num_kv_heads=case.Hkv, num_heads=case.Hq)
    torch.cuda.synchronize()
    dev = _ref_device(case)
    assert_within_budget(got, *(t.to(dev) for t in (q, kp, vp, bt, cl)), scale, case.causal, case.Hkv, case.Hq, f"{name}, {pattern}",
                         mma=case.mma)


@pytest.mark.gpu
def test_spike_after_every_tile_boundary_of_a_long_table(cuda_device):
    """One request over 8192 keys (the split + merge route): a +40 spike on the first key past each
    of the 127 tile boundaries in turn - one spike per KV head, eight heads a call - so every
    split boundary is covered whatever the split policy, with all other splits 40 below."""
    Hkv, G, page, N, D = 8, 4, 128, 8192, 128
    starts = list(range(64, N, 64))
    for first in range(0, len(starts), Hkv):
        pos = starts[first : first + Hkv]
        pos += [pos[-1]] * (Hkv - len(pos))
        g = torch.Generator().manual_seed(first)
        u, _ = directions(D, Hkv)
        s = torch.zeros(Hkv, N, dtype=F64)
        s[torch.arange(Hkv), torch.tensor(pos)] = 40.0
        k = make_keys(s, u[:, None, :], g)
        v = torch.randn(Hkv, N, D, generator=g, dtype=F64)
        bt = torch.randperm(N // page, generator=g).to(torch.int32)[None]
        kp = torch.empty(N // page, Hkv, page, D, dtype=F64)
        vp = torch.empty_like(kp)
        kp[bt[0].long()] = k.reshape(Hkv, N // page, page, D).transpose(0, 1)
        vp[bt[0].long()] = v.reshape(Hkv, N // page, page, D).transpose(0, 1)
        q = (u[:, None, :] * math.sqrt(D)).expand(Hkv, G, D).reshape(Hkv * G, 1, D)
        q, kp, vp = q.to(BF16), kp.to(BF16), vp.to(BF16)
        cl = torch.tensor([N], dtype=torch.int32)
        got = ext().paged_attention(*(t.to(cuda_device) for t in (q, kp, vp, bt, cl)), D**-0.5, is_causal=True, num_kv_heads=Hkv, num_heads=Hkv * G)
        assert_within_budget(got.cpu(), q, kp, vp, bt, cl, D**-0.5, True, Hkv, Hkv * G, f"spikes at {pos}", mma=True)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["stair:9", "decoy"])
def test_token_major_prefill_against_fp64(cuda_device, pattern):
    """paged_attention_token_major (tcgen05 prefill storing [B * L, Hq * D]) on a staircase and on decoys."""
    case = Case("token_major", TC, (1000, 700), 256, page=128, width=9)
    q, kp, vp, bt, cl = build(case, pattern, seed=11, device=cuda_device)
    got = ext().paged_attention_token_major(q, kp, vp, bt, cl, 128**-0.5, True, case.Hkv, case.Hq)
    B, L, Hq = 2, case.L, case.Hq
    got = got.view(B, L, Hq, 128).transpose(1, 2).reshape(B * Hq, L, 128)
    assert_within_budget(got.cpu(), *(t.cpu() for t in (q, kp, vp, bt, cl)), 128**-0.5, True, case.Hkv, Hq, f"token-major, {pattern}", mma=True)


# -------------------------------------------------------------------------- GPU: fused decode --
FUSED_PATTERNS = ["stair:7.75", "stair:9", "stair:30", "spike:0", "spike:64", "spike:last", "sink", "decoy"]


def build_fused(ctx, pattern, seed):
    """Inputs of one decode_attention_fused step for two requests (ctx and ctx - 37) at position 0,
    and the oracle's page contents after the append."""
    g = torch.Generator().manual_seed(seed)
    Hq, Hkv, D, page = 8, 2, 128, 64
    ctxs = [ctx, ctx - 37]
    width = -(-ctx // page) + 1
    B, P, N = 2, 2 * width + 1, width * page
    u, perp = directions(D, Hkv)
    s = torch.zeros(B, Hkv, N, dtype=F64)
    loud = torch.zeros(B, N, dtype=torch.bool)
    for b, c in enumerate(ctxs):
        sb, lb = pattern_scores(pattern, c, 1, page, N, True)
        s[b], loud[b] = sb.clamp(min=-64.0), lb  # keep the score range within 64 log2 units
    k = make_keys(s, u[None, :, None, :], g)
    v = torch.randn(B, Hkv, N, D, generator=g, dtype=F64)
    sign = torch.where(torch.rand(B, Hkv, N, D, generator=g) < 0.5, -1.0, 1.0).to(F64)
    v = torch.where(loud[:, None, :, None], 256.0 * sign, v)
    bt = torch.randperm(P, generator=g)[: B * width].reshape(B, width).to(torch.int32)
    kp = torch.randn(P, Hkv, page, D, generator=g, dtype=F64)
    vp = torch.randn(P, Hkv, page, D, generator=g, dtype=F64)
    kp[bt.long()] = k.reshape(B, Hkv, width, page, D).transpose(1, 2)
    vp[bt.long()] = v.reshape(B, Hkv, width, page, D).transpose(1, 2)
    kp, vp = kp.to(BF16), vp.to(BF16)
    # qkv: q heads along +u, the new key along the pattern's direction at ctx - 1 (its norm weight
    # carries the magnitude: RMSNorm of +-3 is +-1), the new value from the pattern's V row
    h = hadamard(D)
    top = [s[b, :, c - 1] for b, c in enumerate(ctxs)]
    assert all(bool(((t == 0) | (t == 40)).all()) for t in top), "the new key scores 0 or +40"
    qkv = torch.zeros(B, (Hq + 2 * Hkv) * D, dtype=F64)
    for b, c in enumerate(ctxs):
        for hq in range(Hq):
            qkv[b, hq * D : (hq + 1) * D] = 3.0 * h[1 + hq // (Hq // Hkv)]
        for hk in range(Hkv):
            spike = bool(top[b][hk] == 40)
            qkv[b, (Hq + hk) * D : (Hq + hk + 1) * D] = 3.0 * (h[1 + hk] if spike else h[1 + Hkv + hk])
            qkv[b, (Hq + Hkv + hk) * D : (Hq + Hkv + hk + 1) * D] = v[b, hk, c - 1]
    qw = torch.ones(D, dtype=BF16)
    kw = torch.full((D,), 40.0 * LN2 / math.sqrt(D), dtype=F64).to(BF16) if pattern == "spike:last" else torch.ones(D, dtype=BF16)
    qkv = qkv.to(BF16)
    cl = torch.tensor(ctxs, dtype=torch.int32)
    offsets = torch.zeros(B, dtype=torch.int32)
    # the oracle's operator sequence: RMSNorm -> RoPE (position 0) -> append at ctx - 1
    q_ref = oracle.rope(oracle.rms_norm(qkv[:, : Hq * D].reshape(B, 1, Hq, D), qw, 1e-6), offsets, D, 1e6)
    k_ref = oracle.rope(oracle.rms_norm(qkv[:, Hq * D : (Hq + Hkv) * D].reshape(B, 1, Hkv, D), kw, 1e-6), offsets, D, 1e6)
    v_in = qkv[:, (Hq + Hkv) * D :].reshape(B, 1, Hkv, D)
    kp_ref, vp_ref = kp.clone(), vp.clone()
    for b, c in enumerate(ctxs):
        pid = int(bt[b, (c - 1) // page])
        oracle.paged_cache_update(kp_ref, k_ref[b : b + 1].transpose(1, 2).contiguous(), pid, (c - 1) % page)
        oracle.paged_cache_update(vp_ref, v_in[b : b + 1].transpose(1, 2).contiguous(), pid, (c - 1) % page)
    q_ref = q_ref.transpose(1, 2).reshape(B * Hq, 1, D).contiguous()
    return dict(qkv=qkv, qw=qw, kw=kw, offsets=offsets, bt=bt, cl=cl, kp=kp, vp=vp, kp_ref=kp_ref, vp_ref=vp_ref, q_ref=q_ref,
                Hq=Hq, Hkv=Hkv, D=D)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", FUSED_PATTERNS)
@pytest.mark.parametrize("ctx", [200, 700, 4100])  # one round, two splits, many splits (decode_attention_fused.cu:388-394)
def test_fused_decode_attention_against_fp64(cuda_device, ctx, pattern):
    f = build_fused(ctx, pattern, seed=ctx + len(pattern))
    dev = cuda_device
    kd, vd = f["kp"].to(dev), f["vp"].to(dev)
    D = f["D"]
    got = ext().decode_attention_fused(f["qkv"].to(dev), f["qw"].to(dev), f["kw"].to(dev), f["offsets"].to(dev), f["bt"].to(dev),
                                       f["cl"].to(dev), ext().rope_inv_freq_table(D, 1e6, dev), kd, vd, f["Hq"], f["Hkv"], 1e-6,
                                       D**-0.5, ctx)
    assert torch.equal(kd.cpu(), f["kp_ref"]) and torch.equal(vd.cpu(), f["vp_ref"]), "appended K/V differ from the oracle's"
    got = got.cpu().reshape(-1, 1, D)
    assert_within_budget(got, f["q_ref"], f["kp_ref"], f["vp_ref"], f["bt"], f["cl"], D**-0.5, True, f["Hkv"], f["Hq"], f"fused, ctx {ctx}, {pattern}",
                         mma=True)  # mma.sync on bf16 q and K


# -------------------------------------------------------------------- GPU: dense week-2 decode --
def dense_inputs(pattern, causal, seed, L=3, S=700):
    """decode_attention q [Hq, L, D], k / v [Hkv, S, D] and an fp32 mask with -inf and -1e4 entries
    (no row fully masked)."""
    g = torch.Generator().manual_seed(seed)
    Hq, Hkv, D = 8, 2, 128
    u, _ = directions(D, Hkv)
    s, _ = pattern_scores(pattern, S, L, 64, S, causal)
    k = make_keys(s.expand(Hkv, S).clone(), u[:, None, :], g)
    v = torch.randn(Hkv, S, D, generator=g, dtype=F64)
    q = (u[:, None, None, :] * math.sqrt(D)).expand(Hkv, Hq // Hkv, L, D).reshape(Hq, L, D)
    r = torch.rand(Hq, L, S, generator=g)
    mask = torch.where(r < 0.2, -math.inf, torch.where(r < 0.3, -1e4, 0.0)).to(F32)
    mask[..., S - L :] = 0.0  # every row keeps its diagonal key
    return q.to(BF16), k.to(BF16), v.to(BF16), mask, Hq, Hkv, D


def dense_fp64(q, k, v, mask, scale, causal, Hq, Hkv):
    """(out, Vmax, E_s, n) of decode_attention in float64 (additive mask, bottom-right causality)."""
    L, S, D = q.shape[1], k.shape[1], q.shape[2]
    G = Hq // Hkv
    q64, k64, v64 = q.to(F64).reshape(Hkv, G, L, D), k.to(F64)[:, None], v.to(F64)[:, None]
    s = (q64 @ k64.transpose(-1, -2)) * scale + mask.to(F64).reshape(Hkv, G, L, S)
    if causal:
        s = s.masked_fill(torch.arange(S)[None, :] > (S - L + torch.arange(L))[:, None], -math.inf)
    p = torch.softmax(s, -1)
    seen = torch.isfinite(s)
    vmax = torch.where(seen, v64.abs().amax(-1)[:, :, None, :], 0.0).amax(-1)
    a = (q64.abs() @ k64.abs().transpose(-1, -2)) * scale * LOG2E
    e_s = 2.2 * LN2 * (p * ((D + 2) * 2.0**-24 * a + 2.0**-19)).sum(-1)  # __expf: 2^-21 + argument rounding
    return (p @ v64).reshape(Hq, L, D), vmax.reshape(Hq, L), e_s.reshape(Hq, L), seen.sum(-1).to(F64).reshape(Hq, L)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["spike:64", "spike:last", "stair:9", "stair:30", "ramp"])
@pytest.mark.parametrize("causal", [False, True])
def test_dense_decode_attention_with_mask_against_fp64(cuda_device, pattern, causal):
    q, k, v, mask, Hq, Hkv, D = dense_inputs(pattern, causal, seed=len(pattern) + int(causal))
    scale = D**-0.5
    got = ext().decode_attention(q.to(cuda_device), k.to(cuda_device), v.to(cuda_device), mask.to(cuda_device), scale, causal, True, Hq, Hkv)
    ref, vmax, e_s, n = dense_fp64(q, k, v, mask, scale, causal, Hq, Hkv)
    bound = 2.0**-8 * ref.abs() + ((2.0**-8 + n * 2.0**-23 + e_s) * vmax)[..., None]
    err = (got.cpu().to(F64) - ref).abs()
    assert bool((err <= bound).all()), f"{pattern}: {int((~(err <= bound)).sum())} outputs outside the budget, max error {float(err.max()):.3g}"


# ------------------------------------------------------------------------------ route check --
def _kernels_launched(fn):
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


@pytest.mark.gpu
def test_each_route_runs_the_kernel_its_cases_target(cuda_device):
    """Each case above, once, under torch.profiler (kernel tracing only): the __global__ its comment
    names is launched - a change of a routing threshold cannot move a case off its kernel unnoticed."""
    missing = []
    for case in CASES:
        q, kp, vp, bt, cl = build(case, "stair:9", seed=1, device=cuda_device)
        names = _kernels_launched(lambda: ext().paged_attention(q, kp, vp, bt, cl, case.D**-0.5, is_causal=case.causal,
                                                                num_kv_heads=case.Hkv, num_heads=case.Hq))
        want = [case.kernel] + ([TC] if case.kernel == MERGE and case.name.startswith("tc") else [])
        want += [GQA] if case.kernel == MERGE and case.name.startswith("gqa") else []
        for w in want:
            if not any(w in n for n in names):
                missing.append(f"{case.name}: {w} not in {sorted(names)}")
        for w in case.absent:
            if any(w in n for n in names):
                missing.append(f"{case.name}: {w} launched ({sorted(names)})")
    tm = Case("token_major", TC, (1000,), 256, page=128)
    q, kp, vp, bt, cl = build(tm, "stair:9", seed=1, device=cuda_device)
    names = _kernels_launched(lambda: ext().paged_attention_token_major(q, kp, vp, bt, cl, 128**-0.5, True, 2, 8))
    if not any(TC in n for n in names):
        missing.append(f"token-major: {TC} not in {sorted(names)}")
    fused, merge = "decode_attention_fused_kernel", "decode_attention_merge_kernel"
    for ctx, want, absent in ((200, [fused], [merge]), (700, [fused, merge], []), (4100, [fused, merge], [])):
        f = build_fused(ctx, "stair:9", seed=1)
        dev = cuda_device
        args = (f["qkv"].to(dev), f["qw"].to(dev), f["kw"].to(dev), f["offsets"].to(dev), f["bt"].to(dev), f["cl"].to(dev),
                ext().rope_inv_freq_table(128, 1e6, dev), f["kp"].to(dev), f["vp"].to(dev), f["Hq"], f["Hkv"], 1e-6, 128**-0.5, ctx)
        names = _kernels_launched(lambda: ext().decode_attention_fused(*args))
        missing += [f"fused ctx {ctx}: {w} not in {sorted(names)}" for w in want if not any(w in n for n in names)]
        missing += [f"fused ctx {ctx}: {w} launched ({sorted(names)})" for w in absent if any(w in n for n in names)]
    q, k, v, mask, Hq, Hkv, D = (t.to(cuda_device) if torch.is_tensor(t) else t for t in dense_inputs("stair:9", True, 1))
    names = _kernels_launched(lambda: ext().decode_attention(q, k, v, mask, D**-0.5, True, True, Hq, Hkv))
    if not any("decode_attention_kernel" in n for n in names):
        missing.append(f"dense decode: decode_attention_kernel not in {sorted(names)}")
    assert not missing, "\n".join(missing)


def ext():
    from extensions_b200 import tiny_llm_ext_b200

    return tiny_llm_ext_b200
