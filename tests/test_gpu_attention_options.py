"""GPU: the attention options and edges that tests/test_gpu_attention.py does not reach, against a float64 reference.

Covered here: an explicit `scale` on every kernel family (FA-2, FFPA D-sliced 1-CTA, streaming-Q, CTA pair, O^T), the
[B,H,D,N] V layout at every FA-2 head dim (also masked), bf16 with `seqlens_k`, key-padding lengths on both sides of
every KV-tile edge, keys and values past the length that hold NaN / Inf, row independence under lazy rescaling, the
65535 (batch x head) grid limit and more than 2^31 elements per tensor in the FFPA kernels.

Accuracy is checked per element against a bound derived from the kernels' arithmetic (see `_bound`), not against an
fp32 oracle with a fixed tolerance: at N ~ 1000 one key leaking past a mask moves O by ~|v|/N ~ 1e-3, which a fixed
atol of 1e-3 does not reliably catch.  Where two calls do identical arithmetic they are compared bit for bit.
Each accuracy test records its largest err/bound as the user property `max_err_over_bound` of its report
(written, for example, by --junitxml)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

FA2_D = (32, 64, 96, 128)
# (D, variant): the FFPA kernel families.  256: D-sliced 1-CTA, and the O^T kernel (0x200); 320: D-sliced;
# 576: D-sliced with Q streamed (Q is kept resident only up to D = 512); 512: O^T (default) and the D-sliced CTA pair
# (0x400); 768, 1024: CTA pair.
FFPA = [(256, 0), (256, 0x200), (320, 0), (576, 0), (512, 0), (512, 0x400), (768, 0), (1024, 0)]
RAGGED_N = (1, 129, 300, 777)


def _ops():
    from b200k import ops

    return ops


def _lib():
    from b200k import _loader

    return _loader


def _rand(shape, dtype, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, generator=g, device="cuda", dtype=dtype)


def _scales(D):
    return (0.02, 0.5 / np.sqrt(D), 1.0, 2.0)


def c_default_scale(D):
    """The scale the C side uses for scale <= 0: 1.0f / sqrtf(float(D))."""
    return float(np.float32(1) / np.sqrt(np.float32(D)))


def attn_f64(q, k, v, scale, causal=False, seqlens=None, v_dn=False):
    """softmax(q k^T * scale) v in float64 with no rounding, on q's device.  Also returns absPV = sum_j p_j |v_j| for
    every output element and the number of keys each query row sees.  `scale` should be the fp32 value the kernel
    receives.  v_dn: v is [B,H,D,N]."""
    qd, kd, vd = q.double(), k.double(), v.double()
    if v_dn:
        vd = vd.transpose(-2, -1)
    B, H, N, D = q.shape
    s = (qd @ kd.transpose(-2, -1)) * float(scale)
    key = torch.arange(N, device=q.device)
    masked = torch.zeros(B, 1, N, N, dtype=torch.bool, device=q.device)
    if causal:
        masked |= key.view(1, 1, 1, N) > key.view(1, 1, N, 1)
    if seqlens is not None:
        masked |= key.view(1, 1, 1, N) >= torch.as_tensor(seqlens, device=q.device).view(B, 1, 1, 1)
    p = torch.softmax(s.masked_fill(masked, float("-inf")), dim=-1)
    return p @ vd, p @ vd.abs(), (~masked).sum(-1, keepdim=True)


def _bound(ref, abs_pv, n_keys, vmax, dtype):
    """|o - ref| allowed per element.  The kernels round P once to the I/O type (the row sum l is taken before that
    rounding), keep statistics and accumulators in fp32, round O once, and compute a fraction of the exponentials
    with a degree-3 polynomial (relative error 1e-4).  So:
      fp16: 2^-11 |ref| (output rounding) + 2^-10 absPV (P rounding 2^-11, polynomial and fp32 error within the other
            2^-11) + n_keys 2^-25 max|v| (P below fp16's normal range is rounded to a multiple of 2^-24; l >= 1)
            + 2^-24 (O in fp16's subnormal range);
      bf16: 2^-8 |ref| + 2^-7 absPV + 2^-130 (bf16 has fp32's exponent range)."""
    if dtype == torch.float16:
        return 2.0 ** -11 * ref.abs() + 2.0 ** -10 * abs_pv + n_keys * 2.0 ** -25 * vmax + 2.0 ** -24
    assert dtype == torch.bfloat16
    return 2.0 ** -8 * ref.abs() + 2.0 ** -7 * abs_pv + 2.0 ** -130


def check_f64(o, q, k, v, scale, causal=False, seqlens=None, v_dn=False, what=""):
    """Asserts |o - ref| <= bound everywhere (a NaN fails); returns max err/bound."""
    ref, abs_pv, n_keys = attn_f64(q, k, v, scale, causal, seqlens, v_dn)
    vmax = v.abs().amax(dim=(-2, -1), keepdim=True).double()
    ratio = ((o.double() - ref).abs() / _bound(ref, abs_pv, n_keys, vmax, o.dtype)).max().item()
    assert ratio <= 1.0, "%s: max err/bound = %r" % (what, ratio)
    return ratio


def _record(request, ratio):
    request.node.user_properties.append(("max_err_over_bound", ratio))


def fa2(q, k, v, scale=None, causal=False, seqlens=None, v_dn=False):
    o = torch.full_like(q, float("nan"))
    sl = None if seqlens is None else torch.tensor(seqlens, dtype=torch.int32, device=q.device)
    _ops().fa2_fwd(q, k, v, o, scale=scale, v_is_dn=v_dn, causal=causal, seqlens_k=sl)
    return o


def ffpa(q, k, v, scale=None, variant=0):
    o = torch.full_like(q, float("nan"))
    _ops().ffpa_fwd(q, k, v, o, scale=scale, variant=variant)
    return o


def _mode(mode, B, N):
    """(causal, seqlens) of a mask mode; seqlens cut the keys of each batch at a different, tile-ragged length."""
    lens = [max(1, N - 1 - 37 * b) if b % 2 == 0 else max(1, N // 2 + 1) for b in range(B)]
    return {"plain": (False, None), "causal": (True, None), "seqlens": (False, lens),
            "causal+seqlens": (True, lens)}[mode]


# ------------------------------------------------------------------------------------------------ 1. explicit scale
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("mode", ["plain", "causal", "seqlens"])
@pytest.mark.parametrize("D", FA2_D)
def test_fa2_explicit_scale_vs_f64(D, mode, dtype, request):
    """Scale 2.0 at D = 128 gives nearly one-hot rows and many lazy-rescale events; 0.02 nearly uniform rows."""
    worst = 0.0
    for N in RAGGED_N:
        B, H = 2, 2
        q, k, v = [_rand((B, H, N, D), dtype, 100 * D + N + i) for i in range(3)]
        causal, lens = _mode(mode, B, N)
        for scale in _scales(D):
            s32 = float(np.float32(scale))
            o = fa2(q, k, v, s32, causal, lens)
            worst = max(worst, check_f64(o, q, k, v, s32, causal, lens, what="N=%d scale=%g" % (N, scale)))
    _record(request, worst)


@pytest.mark.parametrize("D,variant", FFPA)
def test_ffpa_explicit_scale_vs_f64(D, variant, request):
    worst = 0.0
    for N in RAGGED_N:
        q, k, v = [_rand((1, 2, N, D), torch.float16, 7 * D + N + i) for i in range(3)]
        for scale in _scales(D):
            s32 = float(np.float32(scale))
            o = ffpa(q, k, v, s32, variant)
            worst = max(worst, check_f64(o, q, k, v, s32, what="N=%d scale=%g" % (N, scale)))
    _record(request, worst)


# ------------------------------------------------------------------------------------------------ 2. exact scale identity
def _scale_identities(run, q, k, D):
    """fwd(q, k, s) == fwd(2q, k, s/2) == fwd(q, 2k, s/2) bit for bit: a power-of-two factor passes exactly through the
    fp32 scores and through scale * log2(e), so every exp2 argument is the same.  And scale None / 0 / negative is the
    C side's default 1.0f / sqrtf(D)."""
    for scale in _scales(D):
        s32 = float(np.float32(scale))
        o = run(q, k, s32)
        assert torch.isfinite(o).all()
        assert torch.equal(run(2 * q, k, s32 / 2), o), "2q, scale/2 (scale %g)" % scale
        assert torch.equal(run(q, 2 * k, s32 / 2), o), "2k, scale/2 (scale %g)" % scale
    o = run(q, k, c_default_scale(D))
    for dflt in (None, 0.0, -1.0):
        assert torch.equal(run(q, k, dflt), o), "scale=%r" % dflt


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("D", FA2_D)
def test_fa2_scale_identity_bitexact(D, dtype):
    N = 300
    q, k, v = [_rand((2, 2, N, D), dtype, 300 + D + i) for i in range(3)]
    for mode in ("plain", "causal", "seqlens"):
        causal, lens = _mode(mode, 2, N)
        _scale_identities(lambda qq, kk, s: fa2(qq, kk, v, s, causal, lens), q, k, D)


@pytest.mark.parametrize("D,variant", FFPA)
def test_ffpa_scale_identity_bitexact(D, variant):
    q, k, v = [_rand((1, 2, 300, D), torch.float16, 400 + D + i) for i in range(3)]
    _scale_identities(lambda qq, kk, s: ffpa(qq, kk, v, s, variant), q, k, D)


# ------------------------------------------------------------------------------------------------ 3. V as [B,H,D,N]
@pytest.mark.parametrize("mode", ["plain", "causal", "seqlens", "causal+seqlens"])
@pytest.mark.parametrize("D", FA2_D)
def test_fa2_v_dn_every_head_dim(D, mode, request):
    """The transposed-V builds (K-major V operand, [D rows x 64 keys] boxes; D = 96 has one box per 64-key tile, D = 128
    the shared-S layout) against fp64, and bit for bit against the same call with V as [B,H,N,D]: the two differ only
    in the shared-memory descriptor of V, the tensor core sums the same products in the same order."""
    worst = 0.0
    for N in (8, 64, 136, 264, 1000, 2048):
        B, H = 2, 2
        q, k, v = [_rand((B, H, N, D), torch.float16, 500 + D + N + i) for i in range(3)]
        v_dn = v.transpose(-2, -1).contiguous()
        causal, lens = _mode(mode, B, N)
        o = fa2(q, k, v_dn, None, causal, lens, v_dn=True)
        worst = max(worst, check_f64(o, q, k, v_dn, c_default_scale(D), causal, lens, v_dn=True, what="N=%d" % N))
        assert torch.equal(o, fa2(q, k, v, None, causal, lens)), "N=%d: [B,H,D,N] V differs from [B,H,N,D] V" % N
    _record(request, worst)


def _fa2_rc(q, k, v, o, v_dn, dtype_enum, B, H, N, D, causal=0):
    L = _lib()
    return L.lib.b200k_fa2_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), B, H, N, D, 0.0, v_dn, dtype_enum,
                               causal, None, 0, None)


def test_fa2_v_dn_rejections_return_before_launch():
    """N % 8 != 0 with V as [B,H,D,N] (rows of V^T would not be 16-byte aligned) -> EALIGN; bf16 with V as [B,H,D,N]
    (built for fp16 only) -> EARG.  Neither may touch O."""
    L = _lib()
    N, D = 12, 64
    q, k = [_rand((1, 1, N, D), torch.float16, i) for i in range(2)]
    v = _rand((1, 1, D, N), torch.float16, 2)
    o = torch.full_like(q, 7.0)
    assert _fa2_rc(q, k, v, o, 1, L.F16, 1, 1, N, D) == L.EALIGN
    assert _fa2_rc(q, k, v, o, 1, L.F16, 1, 1, N, D, causal=1) == L.EALIGN
    with pytest.raises(RuntimeError):
        _ops().fa2_fwd(q, k, v, o, v_is_dn=True)
    qb, kb, vb = q[..., :8, :].bfloat16().contiguous(), k[..., :8, :].bfloat16().contiguous(), v[..., :8].bfloat16()
    vb = vb.contiguous()
    ob = torch.full_like(qb, 7.0)
    assert _fa2_rc(qb, kb, vb, ob, 1, L.BF16, 1, 1, 8, D) == L.EARG
    torch.cuda.synchronize()
    assert bool((o == 7.0).all()) and bool((ob == 7.0).all())


# ------------------------------------------------------------------------------------------------ 4. key padding at tile edges
EDGE_N = 392  # a multiple of 8 (V as [B,H,D,N]) that is ragged against both KV-tile widths (128, and 64 for D = 96)
EDGE_LENS = [1, 63, 64, 65, 127, 128, 129, 255, 256, 257, EDGE_N - 1, EDGE_N]
LAYOUTS = [(torch.float16, False), (torch.bfloat16, False), (torch.float16, True)]


def _edge_inputs(D, dtype, v_dn, seed):
    B, H, N = len(EDGE_LENS), 2, EDGE_N
    q, k, v = [_rand((B, H, N, D), dtype, seed + i) for i in range(3)]
    return q, k, (v.transpose(-2, -1).contiguous() if v_dn else v)


@pytest.mark.parametrize("causal", [False, True], ids=["full", "causal"])
@pytest.mark.parametrize("dtype,v_dn", LAYOUTS, ids=["f16", "bf16", "f16-vdn"])
@pytest.mark.parametrize("D", FA2_D)
def test_seqlens_tile_edges_vs_f64(D, dtype, v_dn, causal, request):
    """Lengths 1, BC/2 - 1 .. 2 BC + 1, N - 1 and N in one call, one per batch (BC = 128 keys per KV tile, 64 for D = 96)."""
    q, k, v = _edge_inputs(D, dtype, v_dn, 600 + D)
    o = fa2(q, k, v, None, causal, EDGE_LENS, v_dn)
    _record(request, check_f64(o, q, k, v, c_default_scale(D), causal, EDGE_LENS, v_dn))


@pytest.mark.parametrize("poison", [float("nan"), float("inf"), float("-inf")], ids=["nan", "+inf", "-inf"])
@pytest.mark.parametrize("causal", [False, True], ids=["full", "causal"])
@pytest.mark.parametrize("dtype,v_dn", LAYOUTS, ids=["f16", "bf16", "f16-vdn"])
@pytest.mark.parametrize("D", FA2_D)
def test_seqlens_poisoned_padding_is_never_used(D, dtype, v_dn, causal, poison):
    """Keys and values at or past seqlens_k[b] are never used, so they may hold anything, e.g. uninitialised memory: the
    output stays finite and bit-identical to the call with clean padding.  The last KV tile is loaded whole, so its rows
    past the length reach the kernel as real memory (unlike rows past N, which TMA fills with zeros)."""
    q, k, v = _edge_inputs(D, dtype, v_dn, 700 + D)
    o = fa2(q, k, v, None, causal, EDGE_LENS, v_dn)
    k2, v2 = k.clone(), v.clone()
    for b, n in enumerate(EDGE_LENS):
        k2[b, :, n:] = poison
        if v_dn:
            v2[b, :, :, n:] = poison
        else:
            v2[b, :, n:] = poison
    o2 = fa2(q, k2, v2, None, causal, EDGE_LENS, v_dn)
    bad = [n for b, n in enumerate(EDGE_LENS) if not torch.equal(o2[b], o[b])]
    assert torch.isfinite(o2).all() and not bad, "lengths whose output changed: %s" % bad


# ------------------------------------------------------------------------------------------------ 5. row independence
ROWS_X30 = [3, 70, 130, 300]


def _rows_scaled(q, rows, f=30.0):
    q2 = q.clone()
    q2[:, :, rows] *= f
    return q2


def _others(N, rows):
    keep = torch.ones(N, dtype=torch.bool)
    keep[rows] = False
    return keep.nonzero().flatten().cuda()


@pytest.mark.parametrize("causal", [False, True], ids=["full", "causal"])
@pytest.mark.parametrize("D", FA2_D)
def test_fa2_row_independence_under_rescale(D, causal, request):
    """A few query rows scaled by 30 move their running max many times (lazy O rescales).  The rescale is decided per
    warp, so the other rows of those warps are multiplied by alpha = 1: every other output row stays bit-identical.
    Causal: rows < m never see keys >= m, so replacing K / V there with other finite values changes no bit of them."""
    N = 777
    q, k, v = [_rand((1, 2, N, D), torch.float16, 800 + D + i) for i in range(3)]
    o = fa2(q, k, v, None, causal)
    q2 = _rows_scaled(q, ROWS_X30)
    o2 = fa2(q2, k, v, None, causal)
    keep = _others(N, ROWS_X30)
    assert torch.equal(o2[:, :, keep], o[:, :, keep])
    _record(request, check_f64(o2, q2, k, v, c_default_scale(D), causal))
    if causal:
        m = 333
        k3, v3 = k.clone(), v.clone()
        k3[:, :, m:] = _rand((1, 2, N - m, D), torch.float16, 1)
        v3[:, :, m:] = _rand((1, 2, N - m, D), torch.float16, 2)
        assert torch.equal(fa2(q, k3, v3, None, True)[:, :, :m], o[:, :, :m])


@pytest.mark.parametrize("D,variant", [(256, 0x200), (512, 0)])
def test_ffpa_otrans_row_independence_across_the_pair(D, variant, request):
    """In the O^T kernel the two CTAs of a pair share one rescale verdict per KV tile (O^T's columns are the rows of
    both).  Rows 3 and 130 live in the first CTA of their pair, 70 in the second: the rows that did not move are
    multiplied by alpha = 1 in either CTA and stay bit-identical."""
    N = 640
    q, k, v = [_rand((1, 2, N, D), torch.float16, 900 + D + i) for i in range(3)]
    o = ffpa(q, k, v, None, variant)
    q2 = _rows_scaled(q, ROWS_X30)
    o2 = ffpa(q2, k, v, None, variant)
    keep = _others(N, ROWS_X30)
    assert torch.equal(o2[:, :, keep], o[:, :, keep])
    _record(request, check_f64(o2, q2, k, v, c_default_scale(D)))


# ------------------------------------------------------------------------------------------------ 6. grid limit
GRID_CASES = [("fa2", 64, torch.float16, False), ("fa2", 64, torch.bfloat16, True), ("ffpa", 256, torch.float16, False),
              ("ffpa", 512, torch.float16, False), ("ffpa", 1024, torch.float16, False)]


@pytest.mark.parametrize("kind,D,dtype,causal", GRID_CASES, ids=["fa2-f16", "fa2-bf16-causal", "ffpa256", "ffpa512",
                                                                 "ffpa1024"])
def test_grid_limit_65535_heads(kind, D, dtype, causal, request):
    """B*H = 65535 is the largest grid the kernels accept (one grid dimension per (batch, head)): every head is
    written, and the first and last heads match fp64."""
    B, H, N = 3, 21845, 9
    q, k, v = [_rand((B, H, N, D), dtype, 1000 + D + i) for i in range(3)]
    o = fa2(q, k, v, None, causal) if kind == "fa2" else ffpa(q, k, v)
    assert torch.isfinite(o).all()
    worst = 0.0
    for b, h in ((0, 0), (1, 7), (B - 1, H - 1)):
        sel = (slice(b, b + 1), slice(h, h + 1))
        worst = max(worst, check_f64(o[sel], q[sel], k[sel], v[sel], c_default_scale(D), causal, what="head %d,%d" % (b, h)))
    _record(request, worst)


@pytest.mark.parametrize("D", [64, 256, 512, 1024])
def test_grid_limit_65536_heads_rejected(D):
    """B*H = 65536 does not fit the grid: ESHAPE, returned before any launch (O untouched)."""
    L = _lib()
    B, H, N = 2, 32768, 1
    q, k, v = [torch.zeros(B, H, N, D, dtype=torch.half, device="cuda") for _ in range(3)]
    o = torch.full_like(q, 7.0)
    if D == 64:
        assert _fa2_rc(q, k, v, o, 0, L.F16, B, H, N, D) == L.ESHAPE
        assert _fa2_rc(q, k, v, o, 0, L.F16, B, H, N, D, causal=1) == L.ESHAPE
    rc = L.lib.b200k_ffpa_fwd_f16(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), B, H, N, D, 0.0, 0, None)
    assert rc == L.ESHAPE
    torch.cuda.synchronize()
    assert bool((o == 7.0).all())


# ------------------------------------------------------------------------------------------------ 7. 64-bit offsets in FFPA
@pytest.mark.parametrize("H,D", [(16400, 256), (8200, 512), (4100, 1024), (7296, 576)],
                         ids=["d-sliced", "otrans", "pair", "streaming-q"])
def test_ffpa_more_than_2pow31_elements(H, D):
    """(1, H, 512, D) holds more than 2^31 elements per tensor, so neither a 32-bit byte offset nor a 32-bit element
    index would do.  Heads whose byte offsets lie around 0, 2^31 and 2^32 equal the same head run alone, bit for bit,
    and match fp64."""
    free, _ = torch.cuda.mem_get_info()
    if free < 24 * 2 ** 30:
        pytest.skip("needs 24 GiB of free device memory")
    N = 512
    assert H * N * D > 2 ** 31
    q, k, v = [_rand((1, H, N, D), torch.float16, 1100 + D + i) for i in range(3)]
    o = ffpa(q, k, v)
    head_bytes = N * D * 2
    heads = {0, H - 1}
    for off in (2 ** 31, 2 ** 32):
        heads |= {off // head_bytes - 1, off // head_bytes, off // head_bytes + 1}
    for h in sorted(x for x in heads if x < H):
        sel = (slice(0, 1), slice(h, h + 1))
        assert torch.equal(ffpa(q[sel], k[sel], v[sel]), o[sel]), "head %d" % h
        check_f64(o[sel], q[sel], k[sel], v[sel], c_default_scale(D), what="head %d" % h)
    assert torch.isfinite(o[0, ::97]).all()
