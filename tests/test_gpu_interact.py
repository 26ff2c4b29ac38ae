"""evs_interact against a float64 reference: every launch configuration of k_interact_mma (8 and 4 warps per CTA, one and
several resident waves, 16-byte and scalar staging, padded widths) and of the fp32 FMA kernel, the output's layout and
guard region, non-finite inputs, refused shapes and interact_features' argument checks.

The error bound.  For a sample T = [x; ly] (fp32, n_f + 1 rows of d) the reference is Z = T Tᵀ in float64 and
S = |T| |T|ᵀ.  Every packed pair must satisfy

    |got − Z| <= (SPLIT + Dp · 2⁻²³) · S + 1e-38,      Dp = d rounded up to a multiple of 8.

* SPLIT, the split residue of one product.  k_interact_mma splits v = hi + lo: hi is v rounded to TF32 (11 significant
  bits, |lo| <= 2⁻¹¹ |v|, |hi| <= (1 + 2⁻¹¹) |v|), lo = v − hi is exact in fp32 and the tensor core reads only its top 19
  bits, a truncation to TF32 that loses δ with |δ| < 2⁻¹⁰ |lo| <= 2⁻²¹ |v|.  The product is hi·hi + hi·lo' + lo'·hi with
  lo' = lo − δ; against v_i v_j it misses hi_i δ_j + δ_i hi_j + lo_i lo_j, at most 2 (1 + 2⁻¹¹) 2⁻²¹ + 2⁻²² (about 5 · 2⁻²²)
  of |v_i v_j|.  TF32 × TF32 products are exact in fp32.  (Rounding lo to TF32 instead would give 3 · 2⁻²², but the
  rounding's carry turns a NaN into ±0: see test_split_keeps_nan_bit_patterns.)
* Dp · 2⁻²³, the fp32 accumulation.  The kernel adds the products of Dp contraction indices (the padding contributes
  zeros) into fp32 accumulators.  Every partial sum is bounded by S (to 2⁻⁹ relative), and a truncating add (round toward
  zero, as the tensor core's adds may be) errs by less than 2⁻²³ of it; Dp such adds give the term.  The fp32 FMA kernel
  (d adds at 2⁻²⁴, no split) lies well inside the same bound.
* 1e-38 covers results in fp32's subnormal range.

The bound is tight enough to catch a kernel that drops one of the three products (2⁻¹¹ relative error per term) or runs
plain TF32: test_bound_accepts_only_the_full_split emulates all of them on the CPU at every d used here.
"""
import numpy as np
import pytest

from helpers import SMALL_ROWS, pkg

gpu = pytest.mark.gpu

SPLIT = 2 * (1 + 2.0 ** -11) * 2.0 ** -21 + 2.0 ** -22
TINY = 1e-38


def coeff(d):
    return SPLIT + ((d + 7) // 8 * 8) * 2.0 ** -23


# (n_f, d) per launch configuration of launch_interact
MMA_8_WARPS = [(26, 16), (27, 16), (26, 8), (26, 12), (26, 20), (26, 24), (1, 4), (3, 8)]
MMA_4_WARPS = [(28, 16), (31, 16), (26, 32), (26, 36), (26, 64), (26, 96), (26, 128), (31, 128), (31, 20)]
FMA = [(32, 16), (26, 129), (26, 160), (63, 128), (127, 128)]
# B = 16 389: several resident waves of k_interact_mma (3 552 samples at 8 warps, 1 776 at 4, 592 at d = 128) plus a tail
BATCHES = [1, 37, 16389]
MMA_WIDTHS = sorted({d for _, d in MMA_8_WARPS + MMA_4_WARPS} | {18, 30})

SENTINEL = 0x7FBADBAD          # a NaN no arithmetic produces: marks output words the kernel did not write
GUARD = 1024


# ---- CPU: the split and the bound's power --------------------------------------------------------------------------

def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def _f32(u):
    return np.asarray(u, dtype=np.uint32).view(np.float32)


def _hi(v):
    """The kernel's hi: round to TF32 by adding half an ulp and masking (uint32 wrap-around, as on the GPU)."""
    return _f32((_bits(v).astype(np.uint64) + 0x1000 & 0xFFFFE000).astype(np.uint32))


def _gpu_sub(a, b):
    """fp32 a − b with the GPU's NaN result (the canonical 0x7FFFFFFF, whatever the operands' payloads)."""
    with np.errstate(invalid="ignore", over="ignore"):
        r = (np.asarray(a, np.float32) - np.asarray(b, np.float32)).astype(np.float32)
    return np.where(np.isnan(r), _f32(np.uint32(0x7FFFFFFF)), r).astype(np.float32)


def _tf32_operand(v):
    """What the tensor core reads of an fp32 register: its top 19 bits."""
    return _f32(_bits(v) & np.uint32(0xFFFFE000))


def _trunc_f32(s):
    """float64 -> float32 rounded toward zero."""
    r = s.astype(np.float32)
    over = np.abs(r.astype(np.float64)) > np.abs(s)
    r[over] = np.nextafter(r[over], np.float32(0))
    return r


def emulate(T, scheme):
    """Z = T Tᵀ for T float32 [n, nt, d] as k_interact_mma forms it under `scheme`: products of TF32 operands, each mma.sync
    of 8 contraction indices summed exactly and added to the fp32 accumulator with one truncation."""
    n, nt, d = T.shape
    Dp = (d + 7) // 8 * 8
    Tp = np.zeros((n, nt, Dp), np.float32)
    Tp[:, :, :d] = T
    hi = _hi(Tp)
    lo_exact = _gpu_sub(Tp, hi)
    lo = _hi(lo_exact) if scheme == "3xtf32-lo-rounded" else _tf32_operand(lo_exact)
    terms = {"3xtf32": [(hi, hi), (hi, lo), (lo, hi)], "3xtf32-lo-rounded": [(hi, hi), (hi, lo), (lo, hi)],
             "drop-hi.hi": [(hi, lo), (lo, hi)], "drop-hi.lo": [(hi, hi), (lo, hi)], "drop-lo.hi": [(hi, hi), (hi, lo)],
             "1xtf32": [(hi, hi)]}[scheme]
    acc = np.zeros((n, nt, nt), np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        for k0 in range(0, Dp, 8):
            for a, b in terms:
                s = np.einsum("nik,njk->nij", a[:, :, k0:k0 + 8].astype(np.float64), b[:, :, k0:k0 + 8].astype(np.float64))
                acc = _trunc_f32(acc.astype(np.float64) + s)
    return acc


def _worst_ratio(T, Z):
    T64 = T.astype(np.float64)
    ref = np.einsum("nik,njk->nij", T64, T64)
    S = np.einsum("nik,njk->nij", np.abs(T64), np.abs(T64))
    li, lj = np.tril_indices(T.shape[1], -1)
    err = np.abs(Z.astype(np.float64) - ref)[:, li, lj]
    return float((err / (coeff(T.shape[2]) * S[:, li, lj] + TINY)).max())


def _cpu_inputs(rng, n, nt, d, scale):
    if scale == "randn":
        return rng.standard_normal((n, nt, d)).astype(np.float32)
    rows = np.array(SMALL_ROWS * 2)[:nt] * 1000
    bound = np.minimum(1.0 / np.sqrt(rows), 0.6499).astype(np.float32)
    return ((rng.random((n, nt, d), dtype=np.float32) * 2 - 1) * bound[None, :, None]).astype(np.float32)


@pytest.mark.parametrize("scale", ["randn", "tables"])
@pytest.mark.parametrize("d", MMA_WIDTHS)
def test_bound_accepts_only_the_full_split(d, scale):
    """At every width the GPU tests use, the shipped 3xTF32 split (and the rounded-lo variant) lies within the bound, and
    each scheme that drops one of the three products, or plain TF32, breaks it."""
    rng = np.random.default_rng(d)
    T = _cpu_inputs(rng, 48, 27, d, scale)
    for scheme in ("3xtf32", "3xtf32-lo-rounded"):
        r = _worst_ratio(T, emulate(T, scheme))
        assert r <= 1.0, (scheme, d, r)
    for scheme in ("drop-hi.hi", "drop-hi.lo", "drop-lo.hi", "1xtf32"):
        r = _worst_ratio(T, emulate(T, scheme))
        assert r > 1.5, (scheme, d, r)


def test_split_keeps_nan_bit_patterns():
    """The rounding add carries a NaN's mantissa into the sign bit: hi of 0x7FFFFFFF is −0.0 and of 0xFFFFFFFF +0.0, and
    the NaN that v − hi gives is squashed the same way if lo is rounded.  lo goes to the tensor core unrounded, so it stays
    NaN for every NaN, and for ±Inf (hi = ±Inf, lo = Inf − Inf)."""
    pats = np.array([0x7FFFFFFF, 0xFFFFFFFF, 0x7FC00000, 0xFFC00000, 0x7F800001, 0x7F800000, 0xFF800000], np.uint32)
    v = _f32(pats)
    assert _bits(_hi(v)).tolist() == [0x80000000, 0x00000000, 0x7FC00000, 0xFFC00000, 0x7F800000, 0x7F800000, 0xFF800000]
    lo = _gpu_sub(v, _hi(v))
    assert np.isnan(_tf32_operand(lo)).all()
    assert not np.isnan(_hi(lo)[:2]).any()        # the rounded lo of the first two NaNs is ±0: the NaN would be lost
    # through the whole emulated product: every pair touching the non-finite row is NaN, the others are finite
    T = np.ones((len(pats), 3, 8), np.float32)
    T[np.arange(len(pats)), 1, np.arange(len(pats)) % 8] = v
    Z = emulate(T, "3xtf32")
    assert np.isnan(Z[:, 1, 0]).all() and np.isnan(Z[:, 2, 1]).all()
    assert (Z[:, 2, 0] == 8.0).all()
    Zr = emulate(T, "3xtf32-lo-rounded")
    assert np.isfinite(Zr[:2, 1, 0]).all()        # what the rounded split did with the first two NaNs


# ---- GPU ----------------------------------------------------------------------------------------------------------

def _lib():
    return pkg().load_library()


def _make_T(B, nt, d, scale, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    if scale == "randn":
        return torch.randn((B, nt, d), device="cuda", generator=g)
    rows = torch.tensor((SMALL_ROWS * 5)[:nt], dtype=torch.float64) * 1000
    bound = torch.clamp(rows.rsqrt(), max=0.6499).float().cuda()
    return (torch.rand((B, nt, d), device="cuda", generator=g) * 2 - 1) * bound[None, :, None]


def _placed(t, offset):
    """t's values in a fresh contiguous tensor whose data starts `offset` floats into its storage."""
    import torch
    buf = torch.empty(t.numel() + offset + 4, device=t.device, dtype=t.dtype)
    v = buf[offset:offset + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def _guarded_out(B, W):
    """[B, W] in the middle of a buffer filled with the sentinel: (buffer, out)."""
    import torch
    buf = torch.full((B * W + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    return buf, buf[GUARD:GUARD + B * W].view(B, W)


def _run(x, ly, out, B, n_f, d, stream=None):
    import torch
    torch.cuda.synchronize()
    rc = _lib().evs_interact(x.data_ptr(), ly.data_ptr(), out.data_ptr(), B, n_f, d, stream)
    assert rc == 0, (rc, _lib().evs_last_error())
    torch.cuda.synchronize()


def _check(buf, out, x, ly, d, nonfinite=False):
    """The guard region is untouched, every output word is written, the head is x bit for bit, and every pair is within
    the bound of the float64 reference (non-finite inputs: NaN where the reference is NaN, non-finite where it is ±Inf)."""
    import torch
    ib = buf.view(torch.int32)
    assert (ib[:GUARD] == SENTINEL).all() and (ib[-GUARD:] == SENTINEL).all(), "write outside [B, d + pairs]"
    assert not (out.view(torch.int32) == SENTINEL).any(), "output words left unwritten"
    assert torch.equal(out[:, :d].contiguous().view(torch.int32), x.contiguous().view(torch.int32)), "x head differs"
    T = torch.cat([x.unsqueeze(1), ly], dim=1).double()
    nt = T.shape[1]
    li, lj = torch.tril_indices(nt, nt, -1, device=T.device)
    Z = torch.bmm(T, T.transpose(1, 2))[:, li, lj]
    A = T.abs()
    S = torch.bmm(A, A.transpose(1, 2))[:, li, lj]
    got = out[:, d:].double()
    del T, A
    plain = torch.isfinite(Z)
    if nonfinite:
        assert torch.isnan(got[torch.isnan(Z)]).all(), "a pair that is NaN in the reference is not NaN"
        assert (~torch.isfinite(got[torch.isinf(Z)])).all(), "a pair that is ±Inf in the reference is finite"
        assert (~plain).any()
    else:
        assert plain.all()
    err = (got - Z).abs()
    lim = coeff(x.shape[1]) * S + TINY
    ok = (err <= lim) | ~plain
    if not bool(ok.all()):
        ratio = torch.where(plain, err / lim, torch.zeros_like(err))
        ratio[~(err <= lim) & plain] = float("inf")
        k = int(ratio.argmax())
        b, p = divmod(k, Z.shape[1])
        raise AssertionError(f"sample {b} pair ({int(li[p])}, {int(lj[p])}): got {float(got[b, p])!r}, float64 "
                             f"{float(Z[b, p])!r}, bound {float(lim[b, p]):.3e}; {int((~ok).sum())} pairs outside")


def _case(B, n_f, d, scale, seed, x_off=0, ly_off=0, stream=None):
    import torch
    T = _make_T(B, n_f + 1, d, scale, seed)
    x = _placed(T[:, 0], x_off)
    ly = _placed(T[:, 1:], ly_off)
    del T
    buf, out = _guarded_out(B, d + (n_f + 1) * n_f // 2)
    _run(x, ly, out, B, n_f, d, stream)
    _check(buf, out, x, ly, d)
    torch.cuda.synchronize()


@gpu
@pytest.mark.parametrize("scale", ["randn", "tables"])
@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("n_f,d", MMA_8_WARPS + MMA_4_WARPS + FMA)
def test_interaction_within_float64_bound(n_f, d, B, scale):
    """Tensor-core path with 8 and 4 warps per CTA (one sample, one partial wave, several waves of the double buffer) and
    the fp32 FMA kernel (n_f + 1 > 32 or d > 128; n_f = 127 at d = 128 fits 3 warps per CTA, 63 at 128 fits 4)."""
    _case(B, n_f, d, scale, seed=B * 1000 + n_f * 7 + d)


@gpu
@pytest.mark.parametrize("x_off,ly_off", [(1, 0), (0, 1), (1, 1)])
@pytest.mark.parametrize("n_f,d", [(26, 16), (26, 64), (31, 128)])
def test_operands_off_16_byte_alignment(n_f, d, x_off, ly_off):
    """x or ly starting 4 bytes past a 16-byte boundary: scalar staging at d % 4 = 0, across several waves."""
    _case(16389, n_f, d, "randn", seed=d + 10 * x_off + 20 * ly_off, x_off=x_off, ly_off=ly_off)


@gpu
@pytest.mark.parametrize("B", [16, 16389])
@pytest.mark.parametrize("d", [18, 30])
def test_width_not_a_multiple_of_four(d, B):
    """d % 4 != 0: scalar staging and zeroed padding columns up to Dp, across several waves."""
    _case(B, 26, d, "tables", seed=d + B)


@gpu
def test_interaction_mixed_shapes_within_float64_bound():
    """Both kernels at the shapes and batch sizes of an everyday mix, through EvStore.interact as well as the C-ABI: the
    tensor-core path for n_f + 1 <= 32 and d <= 128, the fp32 FMA kernel for (32, 16) and (26, 160)."""
    import torch
    p = pkg()
    store = p.EvStore(p.workload.make_tables(SMALL_ROWS, 16), p.CacheConfig(total_size=300, max_batch=32))
    try:
        for B, n_f, d in [(1, 26, 16), (37, 26, 36), (256, 26, 64), (5, 3, 8), (300, 31, 20), (9, 1, 4), (16, 26, 18),
                          (5, 26, 128), (4, 32, 16), (3, 26, 160)]:
            _case(B, n_f, d, "randn", seed=B)
            T = _make_T(B, n_f + 1, d, "randn", seed=B + 1)
            x, ly = T[:, 0].contiguous(), T[:, 1:].contiguous()
            buf, out = _guarded_out(B, d + (n_f + 1) * n_f // 2)
            assert store.interact(x, ly, out=out).data_ptr() == out.data_ptr()
            torch.cuda.synchronize()
            _check(buf, out, x, ly, d)
    finally:
        store.close()


@gpu
def test_interaction_b2048_d64_within_float64_bound():
    """B = 2048, n_f = 26, d = 64: a little over one resident wave of the 4-warp configuration."""
    _case(2048, 26, 64, "randn", seed=3)


@gpu
def test_caller_supplied_stream():
    import torch
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    _case(16389, 26, 16, "randn", seed=5, stream=s.cuda_stream)


NONFINITE = [0x7FFFFFFF, 0xFFFFFFFF, 0x7FC00000, 0x7F800000, 0xFF800000]


@gpu
@pytest.mark.parametrize("n_f,d", [(26, 16), (31, 16), (26, 64)])
def test_nonfinite_inputs(n_f, d):
    """NaN (the GPU's own 0x7FFFFFFF, its negative, the quiet 0x7FC00000) and ±Inf in x or in one ly row of samples spread
    over the waves.  Pairs of those rows must be NaN / non-finite; every other pair -- including those of the finite
    samples that a warp stages into the same buffers after a non-finite one -- must be finite and within the bound."""
    import torch
    B = 16389
    T = _make_T(B, n_f + 1, d, "randn", seed=n_f + d)
    Ti = T.view(torch.int32)
    samples = [0, 1, 31, 777, 3551, 3552, 3553, 5000, 8191, 9999, 12000, 16387, 16388]
    pats = np.array(NONFINITE, np.uint32).view(np.int32).tolist()
    for k, s in enumerate(samples):
        row = 0 if k % 3 == 0 else 1 + (s * 7) % n_f
        Ti[s, row, (s * 5) % d] = pats[k % len(pats)]
        if k % 4 == 1:
            Ti[s, row, d - 1] = pats[(k + 2) % len(pats)]
    x, ly = T[:, 0].contiguous(), T[:, 1:].contiguous()
    buf, out = _guarded_out(B, d + (n_f + 1) * n_f // 2)
    _run(x, ly, out, B, n_f, d)
    _check(buf, out, x, ly, d, nonfinite=True)


def _optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


@gpu
def test_fma_shape_over_the_shared_memory_limit_is_refused():
    """(n_f + 1)(d + 1) floats of one warp over the device's opt-in shared memory: EVS_ERR_INVALID naming the limit, no
    launch, and no CUDA error left behind for the next call.  The widest d that fits runs with one warp per CTA."""
    import torch
    optin = _optin()
    n_f = 26
    d_max = optin // (4 * (n_f + 1)) - 1
    d = d_max + 2
    assert 4 * (n_f + 1) * (d + 1) > optin >= 4 * (n_f + 1) * (d_max + 1)
    x = torch.zeros((2, d), device="cuda")
    ly = torch.zeros((2, n_f, d), device="cuda")
    buf, out = _guarded_out(2, d + (n_f + 1) * n_f // 2)
    torch.cuda.synchronize()
    rc = _lib().evs_interact(x.data_ptr(), ly.data_ptr(), out.data_ptr(), 2, n_f, d, None)
    msg = _lib().evs_last_error().decode()
    assert rc == -1, (rc, msg)
    assert str(optin) in msg, msg
    torch.cuda.synchronize()
    assert (buf.view(torch.int32) == SENTINEL).all()
    _case(37, 26, 16, "randn", seed=1)                 # a valid call straight after succeeds
    _case(37, n_f, d_max, "randn", seed=2)             # one warp per CTA


@gpu
def test_interact_features_views_narrower_than_their_base():
    """ly = views buf[:, k, :d] of a wider [B, n_f, D] buffer: not the base's layout, so they must be packed first."""
    import torch
    p = pkg()
    B, n_f, d, D = 300, 26, 16, 24
    T = _make_T(B, n_f + 1, D, "randn", seed=9)
    x = T[:, 0, :d].contiguous()
    base = T[:, 1:].contiguous()
    views = [base[:, k, :d] for k in range(n_f)]
    got = p.dlrm_ops.interact_features(x, views)
    buf, out = _guarded_out(B, got.shape[1])
    out.copy_(got)
    _check(buf, out, x, base[:, :, :d], d)
    # full-width views of the base are read in place and give the same
    views = [base[:, k, :] for k in range(n_f)]
    xw = T[:, 0].contiguous()
    got = p.dlrm_ops.interact_features(xw, views)
    buf, out = _guarded_out(B, got.shape[1])
    out.copy_(got)
    _check(buf, out, xw, base, D)


@gpu
def test_interact_features_rejects_bad_arguments_before_launch():
    """Wrong dtypes, batch sizes or output shapes raise ValueError and launch nothing (the sentinel `out` stays as it
    was).  Every operand lies in storage at least as large as a launch with x's shape would touch."""
    import torch
    p = pkg()
    B, n_f, d = 64, 26, 16
    W = d + (n_f + 1) * n_f // 2
    ly = torch.randn((B, n_f, d), device="cuda")
    x = torch.randn((B, d), device="cuda")
    big = torch.full((B * (W + 1),), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)

    def untouched():
        torch.cuda.synchronize()
        return bool((big.view(torch.int32) == SENTINEL).all())

    out = big[:B * W].view(B, W)
    x64 = torch.randn((B, d), device="cuda", dtype=torch.float64)
    x16 = torch.zeros((2 * B * d,), device="cuda", dtype=torch.bfloat16)[:B * d].view(B, d)
    bad = [
        dict(x=x64, ly=ly, out=out),
        dict(x=x16, ly=ly, out=out),
        dict(x=x, ly=torch.randn((B + 1, n_f, d), device="cuda"), out=out),
        dict(x=x, ly=[ly[:, k] for k in range(n_f - 1)] + [torch.randn((B + 1, d), device="cuda")], out=out),
        dict(x=x, ly=[ly[:, k] for k in range(n_f - 1)] + [ly[:, -1].double()], out=out),
        dict(x=x, ly=ly, out=big[:B * (W + 1)].view(B, W + 1)),
        dict(x=x, ly=ly, out=big[:B * (W - 1)].view(B, W - 1)),
        dict(x=x, ly=ly, out=big[:B * W].view(B // 2, 2 * W)[:, :W]),
        dict(x=x, ly=ly, out=big[:B * W].view(torch.int32).view(B, W)),
    ]
    for k, kw in enumerate(bad):
        with pytest.raises(ValueError):
            p.dlrm_ops.interact_features(**kw)
        assert untouched(), f"case {k} launched"
    # and the same arguments, well formed, work
    got = p.dlrm_ops.interact_features(x, ly, out=out)
    assert got.data_ptr() == out.data_ptr()
    buf, o2 = _guarded_out(B, W)
    o2.copy_(got)
    _check(buf, o2, x, ly, d)


@gpu
def test_evstore_interact_is_interact_features():
    import torch
    p = pkg()
    store = p.EvStore(p.workload.make_tables(SMALL_ROWS, 16), p.CacheConfig(total_size=300, max_batch=32))
    try:
        T = _make_T(37, 27, 16, "tables", seed=3)
        x, ly = T[:, 0].contiguous(), T[:, 1:].contiguous()
        got = store.interact(x, ly)
        torch.cuda.synchronize()
        assert torch.equal(got.view(torch.int32), p.dlrm_ops.interact_features(x, ly).view(torch.int32))
        with pytest.raises(ValueError):
            store.interact(x.double(), ly)
    finally:
        store.close()
