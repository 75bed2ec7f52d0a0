"""Every attention kernel path against a float64 reference, with a per-element error bound, on adversarial scores.

Reference and bound
-------------------
From the exact 16-bit inputs, in float64 on the device:  s = q k^T hd^-1/2 (+ key_bias),  p = softmax(s),  ref = p v,
E = p |v| (the softmax-weighted magnitude of V).  Every output element must satisfy  |got - ref| <= 2 * bound  with

    bound = u |ref| + u E + sigma_i E + N f max_j |v_j|

  * u = 2^-11 (fp16) or 2^-8 (bf16) is the unit roundoff of the 16-bit type.
  * u |ref|: the output O / l is rounded to 16 bits once.
  * u E: P is rounded to 16 bits before P V, each weight with relative error <= u, while l sums the unrounded exponentials,
    so nothing cancels: the error is at most sum_j u p_j |v_j| = u E.  (The fp32 accumulation of P V and the rescaling by
    alpha add O(2^-24) relative terms, well inside the factor 2.)
  * sigma_i E: the fp32 score of row i carries an absolute error of a few fp32 ulps of the largest magnitude that went into
    it, sigma_i = 2^-22 (scale max_j sum_d |q_id k_jd| + max_j |bias_j| + |max_j s_ij|) nats.  A score error d changes
    the weight by the factor e^d, i.e. p_j by |d| p_j: at most sigma_i E on the output.  ex2.approx (2^-22 relative) and the
    polynomial exponential (2.8e-6 relative, spatial tiles of 256 keys and the streaming kernel) are of this size or less.
  * N f max_j |v_j|: a weight at the bottom of the range carries an absolute error f on each of the N keys; l >= 1 only
    shrinks it.  fp16 weights below 2^-14 are subnormal, rounded to 2^-25 absolute (f = 2^-25); bf16 has the fp32 exponent
    range, where the exponentials flush below 2^-126 (f = 2^-126, negligible here but not in the backward, whose outputs
    can themselves be that small).
The factor 2 is the only free constant.  Every call must also be free of NaN, and three calls must be bit-identical.

Input families (all built from 16-bit-representable values; scores are designed in log2 units through "control"
dimensions: q holds 1 there and k holds the wanted level / (hd^-1/2 log2 e), split into three 16-bit terms so that the
score is exact to ~2^-30; the other dimensions carry small noise)
  F1 random      q, k ~ 1.5 N(0,1) (the existing tests' inputs).
  F2 growth      chunks of 128 keys.  Rows r % 4 == 0: the row maximum grows by TAU + 0.5 at the first key of every later
                 chunk; every key of the intermediate chunks sits at that chunk's maximum, the last chunk's other keys far
                 below, so the rescaled history keeps >= 20 % of the final weight.  Rows r % 4 == 2: the same, except
                 that the chunk before the last sits 3 below the running maximum, so the previous chunk's maximum is not
                 the running maximum when the last jump comes.  Odd rows never grow.  Growing and non-growing rows
                 alternate inside every warp.
  F3 stale max   the same with jumps of TAU - 0.5 over chunk 0 and keys spread below: the lazy running maximum stays at
                 chunk 0 and the exponentials reach 2^7.5 (ex2_poly with positive arguments).
  F4 peaked      one key per row sits >= 30 nat above the rest, at key 0, 127, 128, 255, 256 or N-1 (by row): out = v[j*].
  F5 flat        q = 0: out = the mean of V.
  F6 wide range  q, k ~ 6 N(0,1): most weights are below 2^-126 and flush.
  F7 mask leak   keys the row must not see score >= 100 nat above its own: packed: the first sequence of every 128-row
                 tile; temporal: the first token group of every tile; cross: odd samples, whose K rows the 128-row box of
                 the previous sample reads past kv_len.  A row maximum taken over them underflows every valid weight.

Coverage (test ids without the [attn_v2|attn_v3] and [fp16|bf16] parts; impl 2 = attn_pipe / attn_long, impl 3 =
attn_v3 / attn_stream; hd 64 = TAIL false, hd 72 / 80 = TAIL true; every id runs both dtypes, i.e. both BF16 values)
  launch_{pipe,v3}<*, *, MODE_PACKED>    test_self_attention[packed-n{1,2,4,8,32}-hd{64,80}]       F1 F4 F5 F6 F7
  launch_{pipe,v3}<*, *, MODE_FULL>      test_self_attention[full-n128-hd{64,80}, full-n256-hd{64,72,80}]  F1 F4 F5 F6
                                         (+ F2 F3 at n256; v3 runs n128 on 128-key tiles, n256 on 256-key tiles + ex2_poly)
  launch_{pipe,v3}<*, *, MODE_TEMPORAL>  test_self_attention[temporal-f{4,16,64,128}-hd{64,72,80}]    F1 F4 F5 F6 F7 (F7 not
                                         at f128: one token per tile, nothing is masked; f16 is v3's one-pass 8-token path)
  launch_{pipe,v3}<*, *, MODE_CROSS>     test_cross_attention[rows{128,384}-kv{1,64,65,127,128}-hd{64,72,80}-{nobias,bias}]
                                         F1 F4 F5 F6 F7 (bias: one sample partly masked, one fully, one with only its last key)
  launch_{long,stream}<*, *>             test_self_attention[long-n512-hd80, long-n768-hd72, long-n2048-hd64]  F1..F6
Backward (b200_attention_bwd): test_attention_backward[spatial-n{64,256,512,1024}-hd{64,72}, temporal-f{4,8,16}-hd72]
on F1 F4 F6 (+ F2 at n >= 512), per element against bwd_reference.

The CPU part (no GPU needed) checks that every generator has its property and that a float32 emulation of the streaming
recurrence passes the bound while four plausible bugs in it fail it: the bound can catch what it is meant to catch.
"""
import math

import pytest
import torch

F64 = torch.float64
TAU = 8.0                 # lazy-maximum threshold of the streaming kernel, log2 units
CHUNK = 128               # keys per chunk of the streaming kernel
LOG2E = 1.4426950408889634
U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}
FLUSH = {torch.float16: 2.0 ** -25, torch.bfloat16: 2.0 ** -126}   # absolute error of a weight near the bottom of the range
SAFETY = 2.0
PEAK = 50.0               # F4: the chosen key, log2 units above the others' [-2, 2] (>= 33 nat margin)
LOUD = 170.0              # F7: log2 units added to the masked keys (118 nat)
DTS = [torch.float16, torch.bfloat16]
DT_IDS = ["fp16", "bf16"]


def _r16(x, dt):
    return x.to(dt).to(F64)


def _split(x, dt, parts=3):
    """x (float64) as `parts` dt-representable terms whose sum is x to ~2^-30 relative."""
    out, r = [], x.clone()
    for _ in range(parts):
        t = _r16(r, dt)
        out.append(t)
        r = r - t
    return out


def _peak_positions(n):
    return sorted(j for j in {0, 127, 128, 255, 256, n - 1} if 0 <= j < n)


def _chunk_levels(fam, S, N, g):
    """F2 / F3 score levels, log2 units, [S, 3 patterns, N]: pattern 0 grows, 1 never grows, 2 grows after a dip."""
    C = N // CHUNK
    lv = torch.empty(S, 3, N, dtype=F64)
    lv[:, 1] = -6 * torch.rand(S, N, generator=g, dtype=F64)
    lv[:, 1, 0] = 0
    for pat in (0, 2):
        lv[:, pat, :CHUNK] = 0
        level = 0.0
        for c in range(1, C):
            ck = slice(c * CHUNK, (c + 1) * CHUNK)
            if fam == "F3":
                lv[:, pat, ck] = -4 + (TAU - 0.5 + 4) * torch.rand(S, CHUNK, generator=g, dtype=F64)
                lv[:, pat, c * CHUNK] = TAU - 0.5
            elif pat == 2 and C >= 3 and c == C - 2:    # the dip right before the last jump
                lv[:, pat, ck] = level - 3
            else:
                level += TAU + 0.5
                lv[:, pat, ck] = level if c < C - 1 else level - 24
                lv[:, pat, c * CHUNK] = level
    return lv


def _pattern_qk(levels, pattern, hd, dt, g, noise=0.125):
    """q [S, R, hd], k [S, N, hd] with q_r . k_j hd^-1/2 log2(e) = levels[s, pattern[r], j] + small noise."""
    S, P, N = levels.shape
    R = pattern.numel()
    kval = levels / (hd ** -0.5 * LOG2E)
    q = torch.zeros(S, R, hd, dtype=F64)
    k = torch.zeros(S, N, hd, dtype=F64)
    for p in range(P):
        for i, part in enumerate(_split(kval[:, p], dt)):
            k[:, :, 3 * p + i] = part
        q[:, pattern == p, 3 * p:3 * p + 3] = 1
    c = 3 * P
    q[..., c:] = _r16(noise * torch.randn(S, R, hd - c, generator=g, dtype=F64), dt)
    k[..., c:] = _r16(noise * torch.randn(S, N, hd - c, generator=g, dtype=F64), dt)
    return q, k


def family(fam, S, R, N, hd, dt, g, loud=None):
    """Inputs of one family for S independent (sequence, head) problems of R query rows and N keys: float64 tensors
    q [S, R, hd], k, v [S, N, hd] holding dt values.  F7 needs `loud` [S] bool: those problems' keys get +LOUD log2 units
    against every query, which only matters to the queries that must not see them (other sequences of the same tile)."""
    rows = torch.arange(R)
    v = _r16(torch.randn(S, N, hd, generator=g, dtype=F64), dt)
    rn = lambda n, a: _r16(a * torch.randn(S, n, hd, generator=g, dtype=F64), dt)  # noqa: E731
    if fam == "F1":
        q, k = rn(R, 1.5), rn(N, 1.5)
    elif fam == "F5":
        q, k = torch.zeros(S, R, hd, dtype=F64), rn(N, 1.5)
    elif fam == "F6":
        q, k = rn(R, 6.0), rn(N, 6.0)
    elif fam in ("F2", "F3"):
        assert N % CHUNK == 0 and N >= 2 * CHUNK
        pattern = torch.where(rows % 2 == 1, 1, torch.where(rows % 4 == 0, 0, 2))
        q, k = _pattern_qk(_chunk_levels(fam, S, N, g), pattern, hd, dt, g)
    elif fam == "F4":
        pos = _peak_positions(N)
        lv = -2 + 4 * torch.rand(S, len(pos), N, generator=g, dtype=F64)
        for p, j in enumerate(pos):
            lv[:, p, j] = PEAK
        q, k = _pattern_qk(lv, rows % len(pos), hd, dt, g)
    elif fam == "F7":
        assert loud is not None
        q, k = rn(R, 0.7), rn(N, 0.7)
        q[..., 0:2] = 1
        k[..., 0:2] = 0
        for i, part in enumerate(_split(torch.full((N,), LOUD / (hd ** -0.5 * LOG2E), dtype=F64), dt, 2)):
            k[loud, :, i] = part
    else:
        raise ValueError(fam)
    return q, k, v


def reference(q, k, v, dt, bias=None):
    """float64 softmax(q k^T hd^-1/2 + bias) v for independent problems q [S, R, hd], k, v [S, N, hd] (bias [S, N],
    natural-log units), and the per-element bound of the module docstring."""
    scale = q.shape[-1] ** -0.5
    s = q @ k.transpose(-1, -2) * scale
    mag = (q.abs() @ k.abs().transpose(-1, -2)).amax(-1) * scale
    bmax = torch.zeros_like(mag)
    if bias is not None:
        s = s + bias[:, None, :]
        bmax = bmax + bias.abs().amax(-1, keepdim=True)
    p = torch.softmax(s, dim=-1)
    ref = p @ v
    E = p @ v.abs()
    sigma = 2.0 ** -22 * (mag + bmax + s.amax(-1).abs())
    u = U[dt]
    bound = u * ref.abs() + u * E + sigma[..., None] * E + k.shape[-2] * FLUSH[dt] * v.abs().amax(-2, keepdim=True)
    return ref, bound


def check(got, ref, bound, what):
    got = got.to(F64)
    assert not torch.isnan(got).any(), f"{what}: NaN in the output"
    err = (got - ref).abs()
    ratio = err / (SAFETY * bound).clamp_min(1e-300)
    bad = err > SAFETY * bound
    if bad.any():
        i = int(ratio.flatten().argmax())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements outside 2 x bound; worst: err "
                             f"{err.flatten()[i].item():.3e} = {ratio.flatten()[i].item():.2f} x (2 x bound), "
                             f"flat index {i} of shape {tuple(got.shape)}")


# ------------------------------------------------------------------------------------------------------------------
# CPU: generators, and a float32 emulation of the streaming recurrence to show the bound's sensitivity

def _levels(q, k):
    return q @ k.transpose(-1, -2) * (q.shape[-1] ** -0.5 * LOG2E)


def _lazy_growth(L):
    """Per chunk c >= 1: its maximum minus the lazy running maximum before it [..., C-1]; and the final running max."""
    C = L.shape[-1] // CHUNK
    cmax = L.unflatten(-1, (C, CHUNK)).amax(-1)
    m = cmax[..., 0]
    growth = []
    for c in range(1, C):
        d = cmax[..., c] - m
        growth.append(d)
        m = torch.where(d > TAU, cmax[..., c], m)
    return torch.stack(growth, -1), m


@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
@pytest.mark.parametrize("hd", [64, 72, 80])
@pytest.mark.parametrize("N", [256, 512, 2048])
def test_growth_generators(dt, hd, N):
    """F2: every growing row grows by (TAU, TAU + 1) at every later chunk (after the dip where there is one) and the
    history keeps >= 20 % of the final weight; F3: no row ever moves its lazy maximum and the exponentials reach 2^7."""
    g = torch.Generator().manual_seed(N + hd)
    R = 128
    rows = torch.arange(R)
    q, k, _ = family("F2", 2, R, N, hd, dt, g)
    L = _levels(q, k)
    growth, _ = _lazy_growth(L)
    grow0, dip, flat = rows % 4 == 0, rows % 4 == 2, rows % 2 == 1
    assert ((growth[:, grow0] > TAU) & (growth[:, grow0] < TAU + 1)).all()
    C = N // CHUNK
    if C >= 3:
        jumps = torch.arange(C - 1) != C - 3
        assert (growth[:, dip, C - 3] < -2).all()
        assert ((growth[:, dip][..., jumps] > TAU) & (growth[:, dip][..., jumps] < TAU + 1)).all()
    else:
        assert ((growth[:, dip] > TAU) & (growth[:, dip] < TAU + 1)).all()
    assert (growth[:, flat] <= 0.5).all()
    w = torch.softmax(L / LOG2E, dim=-1)
    history = w[..., : N - CHUNK].sum(-1)
    assert (history[:, ~flat] >= 0.2).all(), history[:, ~flat].min()

    q, k, _ = family("F3", 2, R, N, hd, dt, g)
    L = _levels(q, k)
    growth, m = _lazy_growth(L)
    assert (growth <= TAU - 0.25).all()
    assert ((growth[:, ~flat] > TAU - 1)).all()
    assert ((L - m[..., None]).amax(-1)[:, ~flat] >= 7).all()


@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
@pytest.mark.parametrize("hd", [64, 80])
@pytest.mark.parametrize("N", [1, 8, 64, 128, 256, 512])
def test_peaked_and_wide_generators(dt, hd, N):
    """F4: the designed key is every row's argmax, >= 30 nat above the next; all peak positions < N are used.
    F5: q = 0.  F6: most weights are below 2^-126."""
    g = torch.Generator().manual_seed(N * 7 + hd)
    q, k, _ = family("F4", 2, N, N, hd, dt, g)
    s = q @ k.transpose(-1, -2) * hd ** -0.5
    pos = torch.tensor(_peak_positions(N))
    want = pos[torch.arange(N) % len(pos)]
    top = s.topk(min(2, N), dim=-1)
    assert (top.indices[..., 0] == want).all()
    if N > 1:
        assert (top.values[..., 0] - top.values[..., 1] >= 30).all()
    assert set(want.tolist()) == set(pos.tolist())
    q, _, _ = family("F5", 2, N, N, hd, dt, g)
    assert (q == 0).all()
    if N >= 256:
        q, k, _ = family("F6", 2, N, N, hd, dt, g)
        p = torch.softmax(q @ k.transpose(-1, -2) * hd ** -0.5, dim=-1)
        assert (p < 2.0 ** -126).double().mean() > 0.5


def _packed_tile(fam, n, hd, dt, g):
    """One 128-row packed tile of 128 / n sequences of n tokens: tile q, k, v [128, hd], block-diagonal validity, and the
    per-sequence inputs.  F7 makes sequence 0 loud."""
    S = 128 // n
    loud = torch.arange(S) == 0
    q, k, v = family(fam, S, n, n, hd, dt, g, loud if fam == "F7" else None)
    r = torch.arange(128)
    valid = (r[:, None] // n) == (r[None, :] // n)
    return q, k, v, valid


@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
@pytest.mark.parametrize("hd", [64, 80])
@pytest.mark.parametrize("n", [1, 8, 32])
def test_mask_leak_generator(dt, hd, n):
    """F7: in every row that must not see the loud sequence, its keys score >= 100 nat above every valid key."""
    g = torch.Generator().manual_seed(n + hd)
    q, k, _, valid = _packed_tile("F7", n, hd, dt, g)
    s = q.reshape(128, hd) @ k.reshape(128, hd).T * hd ** -0.5
    quiet = torch.arange(128) >= n
    top_valid = s.masked_fill(~valid, -math.inf).amax(-1)
    loud_min = s[:, :n].amin(-1)
    assert (loud_min[quiet] - top_valid[quiet] >= 100).all()


def emulate_stream(q, k, v, dt, valid=None, mutation=None):
    """float32 restatement of the streaming kernel's recurrence (attention.cu attn_stream_kernel) on one problem q [R, hd],
    k, v [N, hd]: 128-key chunks, lazy running maximum with TAU = 8, P rounded to dt, l summed from the unrounded
    exponentials, O / l rounded to dt.  `mutation` plants a bug:
      "a" the O rescale skips the head-dim tail columns [64, hd);  "b" the row maximum includes masked keys;
      "c" l is rescaled but O is not;  "d" alpha is taken against the previous chunk's maximum instead of m_run."""
    f32 = torch.float32
    hd = q.shape[-1]
    sl2 = torch.tensor(1.0 / math.sqrt(hd), dtype=f32) * torch.tensor(LOG2E, dtype=f32)
    s = q.to(f32) @ k.to(f32).T
    R, N = s.shape
    if valid is None:
        valid = torch.ones(R, N, dtype=torch.bool)
    m_run = torch.full((R,), -math.inf, dtype=f32)
    prev = torch.full((R,), -math.inf, dtype=f32)
    l_run = torch.zeros(R, dtype=f32)
    O = torch.zeros(R, hd, dtype=f32)
    vf = v.to(f32)
    for c0 in range(0, N, CHUNK):
        sc, vc = s[:, c0:c0 + CHUNK], valid[:, c0:c0 + CHUNK]
        cmax = (sc if mutation == "b" else sc.masked_fill(~vc, -math.inf)).amax(1)
        grow = (cmax - m_run) * sl2 > TAU
        base = prev if mutation == "d" else m_run
        alpha = torch.where(grow, torch.exp2((base - cmax) * sl2), torch.ones_like(cmax))
        m_run = torch.where(grow, cmax, m_run)
        prev = cmax
        l_run = l_run * alpha
        if mutation == "a":
            O[:, :64] *= alpha[:, None]
        elif mutation != "c":
            O *= alpha[:, None]
        e = torch.exp2(sc * sl2 - (m_run * sl2)[:, None])
        e = torch.where(vc, e, torch.zeros_like(e))
        l_run = l_run + e.sum(1)
        O = O + e.to(dt).to(f32) @ vf[c0:c0 + CHUNK]
    return (O / l_run[:, None]).to(dt)


def _emulation_cases(dt):
    """(family, q [R, hd], k, v [N, hd], valid or None, reference, bound) at hd 80 (so the tail exists), N = 512."""
    hd, N, R = 80, 512, 128
    g = torch.Generator().manual_seed(11)
    out = []
    for fam in ("F1", "F2", "F3", "F4", "F5", "F6"):
        q, k, v = family(fam, 1, R, N, hd, dt, g)
        ref, bound = reference(q, k, v, dt)
        out.append((fam, q[0], k[0], v[0], None, ref[0], bound[0]))
    q, k, v, valid = _packed_tile("F7", 8, hd, dt, g)
    ref, bound = reference(q, k, v, dt)
    out.append(("F7", q.reshape(128, hd), k.reshape(128, hd), v.reshape(128, hd), valid,
                ref.reshape(128, hd), bound.reshape(128, hd)))
    return out


@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
def test_emulation_passes_bound(dt):
    for fam, q, k, v, valid, ref, bound in _emulation_cases(dt):
        check(emulate_stream(q, k, v, dt, valid), ref, bound, f"emulation {fam}")


@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
@pytest.mark.parametrize("mutation,catcher", [("a", "F2"), ("b", "F7"), ("c", "F2"), ("d", "F2")])
def test_emulation_mutation_fails_bound(dt, mutation, catcher):
    """Each planted bug breaks the bound on the family designed to expose it: the GPU tests can fail."""
    failed = []
    for fam, q, k, v, valid, ref, bound in _emulation_cases(dt):
        try:
            check(emulate_stream(q, k, v, dt, valid, mutation), ref, bound, fam)
        except AssertionError:
            failed.append(fam)
    assert catcher in failed, f"mutation {mutation} passes {catcher} (fails: {failed})"


def bwd_reference(q, k, v, do, dt, o16=None):
    """float64 dq, dk, dv of softmax(q k^T hd^-1/2) v with delta formed the way the kernel forms it: rowsum(dO . O16) from
    the 16-bit forward output O16 when given (spatial sequences), else rowsum(dO . O) from the float64 output (temporal
    sequences: that kernel sums P dP itself and never reads the forward output).  Per-element bounds u |ref| + 4u T
    (+ the FLUSH terms of the forward bound, for P and dS), with
      T(dv) = p^T |dO|,   T(dq) = scale (p (|dP| + D)) |k|,   T(dk) = scale (p (|dP| + D))^T |q|,   D = rowsum(|dO . O|).
    D bounds the rounding of delta, which is summed from 16-bit products and may cancel where delta itself is small."""
    scale = q.shape[-1] ** -0.5
    p = torch.softmax(q @ k.transpose(-1, -2) * scale, dim=-1)
    if o16 is None:
        o16 = p @ v
    dv = p.transpose(-1, -2) @ do
    dP = do @ v.transpose(-1, -2)
    delta = (do * o16).sum(-1, keepdim=True)
    dS = p * (dP - delta)
    dq = scale * dS @ k
    dk = scale * dS.transpose(-1, -2) @ q
    u = U[dt]
    w = p * (dP.abs() + (do * o16).abs().sum(-1, keepdim=True))
    bounds = [u * dq.abs() + 4 * u * scale * (w @ k.abs()),
              u * dk.abs() + 4 * u * scale * (w.transpose(-1, -2) @ q.abs()),
              u * dv.abs() + 4 * u * (p.transpose(-1, -2) @ do.abs())]
    # P and dS near the bottom of the range (fp16 subnormals; bf16 and the fp32 exponentials flush below 2^-126): an
    # absolute error of FLUSH on each of the N terms, times dO, or times dP - delta and then k or q
    sub = q.shape[-2] * FLUSH[dt]
    amax = lambda t: t.abs().amax(dim=(-2, -1), keepdim=True)  # noqa: E731
    ds_w = 1 + amax(dP) + amax((do * o16).abs().sum(-1, keepdim=True))
    bounds[0] = bounds[0] + sub * scale * amax(k) * ds_w
    bounds[1] = bounds[1] + sub * scale * amax(q) * ds_w
    bounds[2] = bounds[2] + sub * amax(do)
    return (dq, dk, dv), bounds


def test_bwd_reference_matches_autograd():
    """The closed-form backward reference is float64 autograd when delta is formed from the float64 output."""
    g = torch.Generator().manual_seed(3)
    q, k, v = (torch.randn(2, 40, 24, generator=g, dtype=F64) for _ in range(3))
    do = torch.randn(2, 40, 24, generator=g, dtype=F64)
    qa, ka, va = (t.clone().requires_grad_() for t in (q, k, v))
    o = torch.softmax(qa @ ka.transpose(-1, -2) * 24 ** -0.5, dim=-1) @ va
    o.backward(do)
    for o16 in (o.detach(), None):
        (dq, dk, dv), _ = bwd_reference(q, k, v, do, torch.float16, o16)
        for got, want in ((dq, qa.grad), (dk, ka.grad), (dv, va.grad)):
            assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------------------------------
# GPU

@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(params=[2, 3], ids=["attn_v2", "attn_v3"])
def attn_impl(request):
    """Both attention kernels serve the same contract (include/latte_b200.h: b200_set_attention_impl)."""
    from latte_b200 import _lib
    lib = _lib.load()
    _lib.check(lib.b200_set_attention_impl(request.param), "b200_set_attention_impl")
    yield request.param
    lib.b200_set_attention_impl(0)


def _self_problem(fam, b, f, n, h, hd, temporal, dt, seed, dev):
    """qkv [b f n, 3 h hd] for one family, and the per-(sequence, head) q, k, v [S, L, hd] (float64, on dev)."""
    g = torch.Generator().manual_seed(seed)
    if temporal:
        S, L, G = b * n * h, f, 128 // f
        loud = ((torch.arange(S) // h) % n) % G == 0
    else:
        S, L = b * f * h, n
        loud = ((torch.arange(S) // h) % max(1, 128 // n)) == 0
    q, k, v = family(fam, S, L, L, hd, dt, g, loud if fam == "F7" else None)
    x = torch.stack([q, k, v])
    if temporal:
        x = x.reshape(3, b, n, h, f, hd).permute(1, 4, 2, 0, 3, 5)
    else:
        x = x.reshape(3, b * f, h, n, hd).permute(1, 3, 0, 2, 4)
    qkv = x.reshape(b * f * n, 3 * h * hd).to(dt).contiguous().to(dev)
    return qkv, q.to(dev), k.to(dev), v.to(dev)


def _regroup(out, b, f, n, h, hd, temporal):
    """[b f n, h hd] rows -> [S, L, hd] per (sequence, head), the order family() uses."""
    if temporal:
        return out.reshape(b, f, n, h, hd).permute(0, 2, 3, 1, 4).reshape(b * n * h, f, hd)
    return out.reshape(b * f, n, h, hd).permute(0, 2, 1, 3).reshape(b * f * h, n, hd)


def _thrice(fn):
    outs = [fn() for _ in range(3)]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2]), "reruns are not bit-identical"
    return outs[0]


SELF_CASES = (
    [pytest.param("packed", b, f, n, 2, hd, False, id=f"packed-n{n}-hd{hd}")
     for (b, f, n) in ((1, 200, 1), (2, 50, 2), (1, 80, 4), (1, 3, 8), (2, 6, 32)) for hd in (64, 80)]
    + [pytest.param("full", 1, 2, n, 2, hd, False, id=f"full-n{n}-hd{hd}") for n, hd in ((128, 64), (128, 80), (256, 64), (256, 72), (256, 80))]
    + [pytest.param("long", 1, f, n, 2, hd, False, id=f"long-n{n}-hd{hd}") for f, n, hd in ((2, 512, 80), (2, 768, 72), (1, 2048, 64))]
    + [pytest.param("temporal", 2, F, tok, 2, hd, True, id=f"temporal-f{F}-hd{hd}")
       for F, tok in ((4, 96), (16, 24), (64, 6), (128, 3)) for hd in (64, 72, 80)]
)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
@pytest.mark.parametrize("path,b,f,n,h,hd,temporal", SELF_CASES)
def test_self_attention(dev, dt, path, b, f, n, h, hd, temporal, attn_impl):
    from latte_b200 import ops
    L = f if temporal else n
    fams = ["F1", "F4", "F5", "F6"]
    if L >= 2 * CHUNK and not temporal:
        fams += ["F2", "F3"]
    if (temporal and f < 128) or path == "packed":
        fams += ["F7"]
    for i, fam in enumerate(fams):
        qkv, q, k, v = _self_problem(fam, b, f, n, h, hd, temporal, dt, 1000 * i + L + hd + b, dev)
        got = _regroup(_thrice(lambda: ops.attention(qkv, b, f, n, h, temporal)), b, f, n, h, hd, temporal)
        ref, bound = reference(q, k, v, dt)
        check(got, ref, bound, fam)
        if n == 1 and not temporal:
            assert torch.equal(got.to(F64), v), f"{fam}: a one-token sequence must return v"
        if fam == "F4":
            pos = torch.tensor(_peak_positions(L), device=dev)
            vj = v[:, pos[torch.arange(L, device=dev) % len(pos)]]
            assert ((got.to(F64) - vj).abs() <= U[dt] * vj.abs()).all(), "F4: out != v[j*]"


CROSS_CASES = [pytest.param(128 if i % 2 == 0 else 384, L, hd, id=f"rows{128 if i % 2 == 0 else 384}-kv{L}-hd{hd}")
               for i, (L, hd) in enumerate((L, hd) for L in (1, 64, 65, 127, 128) for hd in (64, 72, 80))]


@pytest.mark.gpu
@pytest.mark.parametrize("with_bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
@pytest.mark.parametrize("rows,L,hd", CROSS_CASES)
def test_cross_attention(dev, dt, rows, L, hd, with_bias, attn_impl):
    """Batch 3: sample 0 partly masked, sample 1 fully masked, sample 2 with only its last key valid (bias runs);
    odd samples are F7's loud ones, read by sample 0's 128-row K box past kv_len."""
    from latte_b200 import ops
    b, h = 3, 2
    D = h * hd
    S = b * h
    bias = None
    if with_bias:
        m = torch.ones(b, L)
        m[0, 1::3] = 0
        m[1] = 0
        m[2, :-1] = 0
        bias = torch.full((b, 128), 123.0)          # columns >= kv_len must be ignored
        bias[:, :L] = (1 - m) * -10000.0
        bias = bias.to(dev)
    for i, fam in enumerate(("F1", "F4", "F5", "F6", "F7")):
        g = torch.Generator().manual_seed(100 * i + rows + L + hd)
        loud = (torch.arange(S) // h) % 2 == 1
        q, k, v = family(fam, S, rows, L, hd, dt, g, loud if fam == "F7" else None)
        qd = q.reshape(b, h, rows, hd).permute(0, 2, 1, 3).reshape(b * rows, D).to(dt).contiguous().to(dev)
        kv = torch.stack([k, v]).reshape(2, b, h, L, hd).permute(1, 3, 0, 2, 4).reshape(b * L, 2 * D).to(dt).contiguous().to(dev)
        out = _thrice(lambda: ops.cross_attention(qd, kv, b, rows, L, h, key_bias=bias))
        got = out.reshape(b, rows, h, hd).permute(0, 2, 1, 3).reshape(S, rows, hd)
        q, k, v = q.to(dev), k.to(dev), v.to(dev)
        sb = bias[:, :L].to(F64).repeat_interleave(h, 0) if with_bias else None
        ref, bound = reference(q, k, v, dt, bias=sb)
        check(got, ref, bound, fam)
        if with_bias:
            last = got[2 * h:].to(F64)
            assert torch.equal(last, v[2 * h:, L - 1:L].expand_as(last)), f"{fam}: only the last key is valid: out = v[L-1]"
        if fam == "F4" and not with_bias:
            pos = torch.tensor(_peak_positions(L), device=dev)
            vj = v[:, pos[torch.arange(rows, device=dev) % len(pos)]]
            assert ((got.to(F64) - vj).abs() <= U[dt] * vj.abs()).all(), "F4: out != v[j*]"


BWD_CASES = ([pytest.param(1, 2, n, 2, hd, False, id=f"spatial-n{n}-hd{hd}") for n in (64, 256, 512, 1024) for hd in (64, 72)]
             + [pytest.param(2, F, 32, 2, 72, True, id=f"temporal-f{F}-hd72") for F in (4, 8, 16)])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
@pytest.mark.parametrize("b,f,n,h,hd,temporal", BWD_CASES)
def test_attention_backward(dev, dt, b, f, n, h, hd, temporal):
    """b200_attention_bwd per element against the float64 closed form (bwd_reference), on F1, F4, F6 (+ F2 at N >= 512)."""
    from latte_b200 import ops
    from latte_b200.train_ops import NativeOps
    nat = NativeOps(dt)
    L = f if temporal else n
    D = h * hd
    fams = ["F1", "F4", "F6"] + (["F2"] if not temporal and n >= 512 else [])
    for i, fam in enumerate(fams):
        qkv, q, k, v = _self_problem(fam, b, f, n, h, hd, temporal, dt, 500 * i + L + hd, dev)
        g = torch.Generator().manual_seed(7 + i)
        do = torch.randn(qkv.shape[0], D, generator=g).to(dt).to(dev)
        o = ops.attention(qkv, b, f, n, h, temporal)
        dqkv = _thrice(lambda: nat.attention_bwd(qkv, o, do, b, f, n, h, temporal))
        rg = lambda t: _regroup(t, b, f, n, h, hd, temporal).to(F64)  # noqa: E731
        refs, bounds = bwd_reference(q, k, v, rg(do), dt, None if temporal else rg(o))
        for j, name in enumerate(("dq", "dk", "dv")):
            got = rg(dqkv[:, j * D:(j + 1) * D])
            assert not torch.isnan(got).any(), f"{fam} {name}: NaN"
            err = (got - refs[j]).abs()
            bad = err > bounds[j]
            assert not bad.any(), (f"{fam} {name}: {int(bad.sum())} of {bad.numel()} outside u|ref| + 4u T; worst "
                                   f"{(err / bounds[j].clamp_min(1e-300)).max().item():.2f} x bound")
