"""evs_knn (csrc/evs_knn.cuh) against float64: every launch configuration of k_knn / k_knn_merge, exact ties, special
values, the C-ABI's output contract and refusals, and the alt keys of generate_alt_keys.

The kernel ranks database row x for query q by the expanded form v = fl(|x|²) − 2·fl₃(q·x), as cuML's brute-force kNN
does, and reports dist = fl(v + fl(|q|²)).  The reference is float64: v* = Σ x² − 2 Σ q x over the D columns, and
dist* = Σ (q − x)² of the row returned.

The error bound.  With X2 = Σ x², Q2 = Σ q² and QX = Σ |q| |x| (elementwise absolute values, so that the bound holds for
data far from the origin, where |v| is much larger than the distance), every candidate satisfies

    |v − v*| <= E(q, x) = 1.001 · [ (D + 1) · 2⁻²⁴ · X2 + 2 · (SPLIT + Dp · 2⁻²³ + 2⁻²⁴) · QX ] + 1e-38

* SPLIT = 2 (1 + 2⁻¹¹) 2⁻²¹ + 2⁻²², the split residue of one product, derived in tests/test_gpu_interact.py: hi is v
  rounded to TF32 by an integer add, lo = v − hi is exact and the tensor core truncates it to TF32.
* Dp · 2⁻²³, the fp32 accumulation of fl₃(q·x): Dp = D rounded up to a multiple of 8, 3 Dp / 8 mma.sync adds of 8
  products each, every partial sum bounded by QX and every add truncating (less than 2⁻²³ of it).
* (D + 1) · 2⁻²⁴ · X2: the norm.  Either order the kernel uses -- the butterfly (four fmaf per lane, then log2(Dp / 4)
  shuffle adds) or the serial fmaf chain over the row in shared memory -- rounds at most D times on the way from a
  square to the sum, each time by at most 2⁻²⁴ of a partial sum bounded by X2; one more 2⁻²⁴ for the final fmaf.
* 2 · 2⁻²⁴ · QX, the rest of the final fmaf(−2, acc, |x|²): |v| <= X2 + 2 QX.  The factor 1.001 covers the products of
  these terms; 1e-38 the subnormal range.

dist adds fl(|q|²) (a D-term fmaf chain) in fp32, so |dist − dist*| <= E + 1.001 · 2⁻²⁴ · ((D + 1) · Q2 + X2 + 2 QX).

What is checked against that bound (check_knn), for every query checked: the ids are distinct, in range and rows with a
finite ranking value; −1 only at the tail and only when fewer than k + 1 rows qualify; the list is ordered up to E; every
row left out, other than the one dropped entry [0], ranks no better than the k-th returned row up to E of both; at most
one row can be the dropped entry, and it ranks no worse than the first returned row up to E; dist[p] is within its bound
of the float64 distance of the id returned at p.  test_bound_accepts_only_the_full_split emulates the kernel's arithmetic
on the CPU and shows that the neighbour checks and the dist check each reject plain TF32 and every scheme that drops one
of hi·hi, hi·lo, lo·hi.

Exact ties.  On small-integer data (hi = v, lo = 0, every product and sum exact in fp32) the kernel must equal
oracle/altkeys.py exactly, ids and dist, every tie broken by row index.

Non-finite values.  A row with a NaN or ±Inf element, or a finite element whose fp32 square overflows the norm, is never
returned and never becomes an alt key.  A query with a NaN or ±Inf element (or FLT_MAX, whose hi is Inf) gets −1 at every
position, a non-finite dist and alt key 0.
"""
import numpy as np
import pytest

from helpers import pkg
from oracle import altkeys

gpu = pytest.mark.gpu

SPLIT = 2 * (1 + 2.0 ** -11) * 2.0 ** -21 + 2.0 ** -22
U = 2.0 ** -24
TINY = 1e-38
FLT_MAX = float(np.finfo(np.float32).max)
BIG = 2.0 ** 127                 # a row whose float64 |x|² reaches this cannot have a finite fp32 norm in these tests

KQ, KT, MAXSPLITS = 128, 64, 64     # kKnnQ, kKnnT of evs_knn.cuh, the split cap of evs_knn

SENTINEL = 0x7FBADBAD            # a NaN no arithmetic produces: marks output words the kernel did not write
SENTINEL64 = 0x7FBADBAD7FBADBAD
GUARD = 512


def dpad(d):
    return (d + 7) // 8 * 8


def knn_config(n, nq, d, sms, x_aligned=True):
    """Which launch of launch_knn a call reaches (evs_api.cu: evs_knn, evs_knn.cuh: launch_knn, k_knn)."""
    Dp = dpad(d)
    qblocks = -(-nq // KQ)
    tiles = -(-n // KT)
    splits = max(1, min(tiles, MAXSPLITS, -(-2 * sms // qblocks)))
    rows_per_split = -(-tiles // splits) * KT
    return {"kernel": "k_knn<2>" if Dp <= 16 else "k_knn<0>",
            "norm": "butterfly" if 32 % (Dp // 4) == 0 else "serial",
            "staging": "vector" if d % 4 == 0 and x_aligned else "scalar",
            "splits": splits, "tiles": tiles,
            "empty_splits": sum(1 for s in range(splits) if s * rows_per_split >= n)}


# ---- the bound and the checks (CPU) --------------------------------------------------------------------------------

def _eligible_rows(x):
    x64 = x.astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.isfinite(x).all(axis=1) & ((x64 * x64).sum(axis=1) < BIG)


def _rankable_queries(q):
    """Queries that get neighbours: every element finite, and none whose hi (tf32_rn) overflows to Inf (FLT_MAX)."""
    with np.errstate(invalid="ignore", over="ignore"):
        return np.isfinite(q).all(axis=1) & np.isfinite(_hi(q)).all(axis=1)


def _bounds(xb, qb):
    """E [nq, n] and the float64 ranking values v* [nq, n] (+inf for rows that may not be returned)."""
    d = xb.shape[1]
    x64, q64 = xb.astype(np.float64), qb.astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        X2 = (x64 * x64).sum(axis=1)
        QX = np.abs(q64) @ np.abs(x64).T
        E = 1.001 * ((d + 1) * U * X2[None, :] + 2 * (SPLIT + dpad(d) * 2.0 ** -23 + U) * QX) + TINY
        v = X2[None, :] - 2.0 * (q64 @ x64.T)
    bad = ~_eligible_rows(xb)
    v[:, bad] = np.inf
    E[:, bad] = 0.0
    return v, E


def check_knn(x, q, nbr, dist, k, rows=None, parts=("nbr", "dist")):
    """Holds nbr [nq, k] / dist [nq, k] (numpy; dist may be None) for queries `rows` (default all) to the float64 bound.
    `parts` selects the neighbour-list checks and / or the dist check.  Raises AssertionError naming the first failure."""
    nq = q.shape[0]
    rows = np.arange(nq) if rows is None else np.asarray(rows)
    elig_x = _eligible_rows(x)
    n_ok = int(elig_x.sum())
    finite_q = _rankable_queries(q)
    x64 = x.astype(np.float64)
    for b0 in range(0, len(rows), 256):
        blk = rows[b0:b0 + 256]
        v, E = _bounds(x, q[blk])
        q64 = q[blk].astype(np.float64)
        for j, i in enumerate(blk):
            got = nbr[i]
            where = f"query {i}"
            if not finite_q[i]:
                assert (got == -1).all(), f"{where} (non-finite) returned {got.tolist()}"
                if dist is not None and "dist" in parts:
                    assert not np.isfinite(dist[i]).any(), f"{where} (non-finite): finite dist {dist[i].tolist()}"
                continue
            m = int((got >= 0).sum())
            assert (got[:m] >= 0).all() and (got[m:] == -1).all(), f"{where}: -1 before the tail: {got.tolist()}"
            want_m = max(0, min(k, n_ok - 1))
            assert m == want_m, f"{where}: {m} neighbours, {n_ok} rows qualify (k = {k}): {got.tolist()}"
            ids = got[:m]
            assert (ids < x.shape[0]).all() and len(set(ids.tolist())) == m, f"{where}: ids {ids.tolist()}"
            assert elig_x[ids].all(), f"{where}: returned a non-finite row: {ids.tolist()}"
            vi, Ei = v[j], E[j]
            if "nbr" in parts and m > 0:
                vr, Er = vi[ids], Ei[ids]
                bad = np.nonzero(vr[:-1] - Er[:-1] > vr[1:] + Er[1:])[0]
                assert len(bad) == 0, (f"{where}: positions {bad[0]}, {bad[0] + 1} (ids {ids[bad[0]]}, {ids[bad[0] + 1]}) out "
                                       f"of order: v* {vr[bad[0]]!r} > {vr[bad[0] + 1]!r} beyond the bound")
                left = elig_x.copy()
                left[ids] = False
                # rows left out that rank better than the k-th beyond the bound: only the dropped entry [0] may
                better = left & (vi + Ei < vr[-1] - Er[-1]) if m == k else np.zeros_like(left)
                nb = int(better.sum())
                assert nb <= 1, (f"{where}: {nb} rows left out rank better than the k-th ({ids[-1]}, v* {vr[-1]!r}), e.g. "
                                 f"{np.nonzero(better)[0][:4].tolist()}")
                first = left & (vi - Ei <= vr[0] + Er[0])
                if nb == 1:
                    r = int(np.nonzero(better)[0][0])
                    assert first[r], f"{where}: row {r} left out ranks between the returned rows (v* {vi[r]!r})"
                else:
                    assert first.any(), f"{where}: no row left out can be the dropped entry [0]"
            if dist is not None and "dist" in parts:
                if m > 0:
                    diff = x64[ids] - q64[j][None, :]
                    ref = (diff * diff).sum(axis=1)
                    Q2 = (q64[j] * q64[j]).sum()
                    X2 = (x64[ids] * x64[ids]).sum(axis=1)
                    QX = np.abs(x64[ids]) @ np.abs(q64[j])
                    lim = Ei[ids] + 1.001 * U * ((x.shape[1] + 1) * Q2 + X2 + 2 * QX) + TINY
                    err = np.abs(dist[i, :m].astype(np.float64) - ref)
                    p = int(np.argmax(err / lim))
                    assert (err <= lim).all(), (f"{where} position {p} (id {ids[p]}): dist {float(dist[i, p])!r}, float64 "
                                                f"{ref[p]!r}, bound {lim[p]:.3e}")
                assert not np.isfinite(dist[i, m:]).any(), f"{where}: finite dist past the neighbours {dist[i].tolist()}"


def exact_oracle(x, q, k):
    """oracle.altkeys.knn_bruteforce, distances as fp32 (exact on small-integer data)."""
    nbr, d = altkeys.knn_bruteforce(x, q, k=k)
    return nbr, d.astype(np.float32)


# ---- CPU: an emulation of k_knn's arithmetic, and the bound's power -----------------------------------------------

def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def _f32(u):
    return np.asarray(u, dtype=np.uint32).view(np.float32)


def _hi(v):
    """tf32_rn: round to TF32 by adding half an ulp and masking (uint32 wrap-around, as on the GPU)."""
    return _f32((_bits(v).astype(np.uint64) + 0x1000 & 0xFFFFE000).astype(np.uint32))


def _tf32_operand(v):
    """What the tensor core reads of an fp32 register: its top 19 bits."""
    return _f32(_bits(v) & np.uint32(0xFFFFE000))


def _trunc_f32(s):
    """float64 -> float32 rounded toward zero."""
    r = s.astype(np.float32)
    over = np.abs(r.astype(np.float64)) > np.abs(s)
    r[over] = np.nextafter(r[over], np.float32(0))
    return r


TERMS = {"3xtf32": ("hh", "hl", "lh"), "drop-hi.hi": ("hl", "lh"), "drop-hi.lo": ("hh", "lh"),
         "drop-lo.hi": ("hh", "hl"), "1xtf32": ("hh",)}


def emulate(x, q, k, scheme):
    """(nbr, dist) as k_knn + k_knn_merge form them for finite x [n, d], q [nq, d] under `scheme`: the split, mma.sync
    k-steps of 8 products summed exactly and added with one truncation each (hi·hi, hi·lo, lo·hi per k-step), the norm in
    the kernel's order (butterfly or serial), fmaf(−2, acc, norm), selection by (v, index)."""
    n, d = x.shape
    Dp = dpad(d)
    xp = np.zeros((n, Dp), np.float32)
    qp = np.zeros((q.shape[0], Dp), np.float32)
    xp[:, :d], qp[:, :d] = x, q
    op = {}
    for name, a in (("x", xp), ("q", qp)):
        h = _hi(a)
        op[name + "h"], op[name + "l"] = h, _tf32_operand((a - h).astype(np.float32))
    acc = np.zeros((q.shape[0], n), np.float32)
    for k0 in range(0, Dp, 8):
        for t in TERMS[scheme]:
            a, b = op["q" + t[0]][:, k0:k0 + 8], op["x" + t[1]][:, k0:k0 + 8]
            acc = _trunc_f32(acc.astype(np.float64) + a.astype(np.float64) @ b.T.astype(np.float64))
    sq = xp.astype(np.float64) ** 2                       # exact; each fmaf rounds once
    if 32 % (Dp // 4) == 0:                               # butterfly: fmaf over a lane's 4 values, then pairwise adds
        part = np.zeros((n, Dp // 4), np.float32)
        lanes = sq.reshape(n, Dp // 4, 4)
        for c in range(4):
            part = (part.astype(np.float64) + lanes[:, :, c]).astype(np.float32)
        while part.shape[1] > 1:
            part = (part[:, 0::2].astype(np.float64) + part[:, 1::2]).astype(np.float32)
        norm = part[:, 0]
    else:
        norm = np.zeros(n, np.float32)
        for c in range(Dp):
            norm = (norm.astype(np.float64) + sq[:, c]).astype(np.float32)
    v = (norm[None, :].astype(np.float64) - 2.0 * acc.astype(np.float64)).astype(np.float32)
    qn = np.zeros(q.shape[0], np.float32)
    for c in range(d):
        qn = (qn.astype(np.float64) + q[:, c].astype(np.float64) ** 2).astype(np.float32)
    order = np.argsort(v, axis=1, kind="stable")[:, :k + 1]
    nbr = order[:, 1:].astype(np.int64)
    dist = (np.take_along_axis(v, nbr, axis=1).astype(np.float64) + qn[:, None]).astype(np.float32)
    return nbr, dist


def _lo_heavy(a):
    """Each value moved to 0.45 TF32 ulp past its hi (same sign): every dropped hi·lo or lo·hi product errs the same way."""
    h = _hi(np.asarray(a, np.float32)).astype(np.float64)
    e = np.floor(np.log2(np.abs(h) + 1e-30))
    return (h + np.sign(h) * 0.45 * 2.0 ** (e - 10)).astype(np.float32)


def _teeth_inputs(d, seed):
    """Off-centre clusters with queries among them, and 'shells': for 32 more queries, 12 rows each at radius 2 ± 1 %
    along +q and −q.  A shell's rows are a few bound-widths apart in v, and a dropped product shifts the + and − rows by
    2⁻¹¹ q·x in opposite directions, far more than the bound: a wrong scheme reorders them."""
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((6, d)) + 1.5
    xc = c[rng.integers(0, 6, 200)] + rng.standard_normal((200, d)) * 2e-2
    qc = c[rng.integers(0, 6, 32)] + rng.standard_normal((32, d)) * 2e-2
    qs = _lo_heavy(rng.standard_normal((32, d)) + 1.5).astype(np.float64)
    qh = qs / np.linalg.norm(qs, axis=1, keepdims=True)
    sgn = np.where(np.arange(12) % 2 == 0, 1.0, -1.0)[None, :, None]
    xs = qs[:, None, :] + 2.0 * sgn * qh[:, None, :] * (1 + 1e-2 * rng.random((32, 12, 1)))
    x = np.concatenate([xc, _lo_heavy(xs.reshape(-1, d))]).astype(np.float32)
    return x, np.concatenate([qc, qs]).astype(np.float32)


TEETH_WIDTHS = [3, 8, 12, 16, 18, 20, 24, 28, 32, 36, 40, 44, 48, 50, 56, 60, 64]


@pytest.mark.parametrize("d", TEETH_WIDTHS)
def test_bound_accepts_only_the_full_split(d):
    """At every width the GPU tests use, the kernel's 3xTF32 arithmetic passes check_knn, and the neighbour checks and
    the dist check each reject plain TF32 and each scheme that drops one of the three products."""
    x, q = _teeth_inputs(d, seed=d)
    nbr, dist = emulate(x, q, 10, "3xtf32")
    check_knn(x, q, nbr, dist, 10)
    for scheme in ("drop-hi.hi", "drop-hi.lo", "drop-lo.hi", "1xtf32"):
        nbr, dist = emulate(x, q, 10, scheme)
        for part in ("nbr", "dist"):
            with pytest.raises(AssertionError):
                check_knn(x, q, nbr, dist, 10, parts=(part,))


def test_emulation_is_exact_on_small_integers():
    """On small-integer data every scheme but the one without hi·hi computes v exactly, and emulate() equals the oracle
    bit for bit: the exact-tie tests on the GPU need no bound."""
    rng = np.random.default_rng(3)
    for d in (3, 4, 16, 64):
        x = rng.integers(-4, 5, (300, d)).astype(np.float32)
        x[200:220] = x[5]
        nbr, dist = emulate(x, x, 10, "3xtf32")
        want, want_d = exact_oracle(x, None, 10)
        assert np.array_equal(nbr, want) and np.array_equal(dist, want_d), d


def test_split_squashes_nan_only_when_lo_is_rounded():
    """The rounding add carries a NaN's mantissa into the sign bit: hi of 0x7FFFFFFF is −0.0 and of 0xFFFFFFFF +0.0,
    and v − hi is the GPU's NaN 0x7FFFFFFF, which rounding would squash the same way.  Passed unrounded, lo stays NaN, so
    every product with the element is NaN; for ±Inf hi is ±Inf and lo = Inf − Inf is NaN."""
    v = _f32(np.array([0x7FFFFFFF, 0xFFFFFFFF, 0x7FC00000, 0x7F800000, 0xFF800000, 0x7F7FFFFF], np.uint32))
    assert _bits(_hi(v)).tolist() == [0x80000000, 0x00000000, 0x7FC00000, 0x7F800000, 0xFF800000, 0x7F800000]
    gpu_nan = _f32(np.uint32(0x7FFFFFFF))
    with np.errstate(invalid="ignore"):
        lo = np.where(np.isnan(v - _hi(v)), gpu_nan, v - _hi(v)).astype(np.float32)
    assert np.isnan(_tf32_operand(lo[:5])).all() and _bits(lo[5]) == 0xFF800000      # FLT_MAX: hi = Inf, lo = −Inf
    assert _bits(_hi(lo[:2])).tolist() == [0x80000000, 0x80000000]                   # what the rounded lo did


def test_launch_configurations_of_the_cases():
    """The cases below reach what they claim on a B200 (148 SMs); the GPU tests assert it again with the device's count."""
    sms = 148
    reached = set()
    for n, nq, d, k, qm, off, _, what in CASES:
        c = knn_config(n, _nq(n, qm, nq, sms), d, sms, off == 0)
        _assert_claims(what, c)
        reached.add((c["kernel"], c["norm"], c["staging"]))
    for kern in ("k_knn<2>", "k_knn<0>"):
        for norm in ("butterfly", "serial"):
            if kern == "k_knn<2>" and norm == "serial":
                continue                                   # Dp <= 16 is always a butterfly width
            for st in ("vector", "scalar"):
                assert (kern, norm, st) in reached, (kern, norm, st)
    assert knn_config(4100, 512, 24, sms)["empty_splits"] > 0
    assert knn_config(3000, 2 * sms * KQ + 1, 16, sms)["splits"] == 1


# ---- GPU ----------------------------------------------------------------------------------------------------------

def _lib():
    return pkg().load_library()


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _placed(t, offset):
    """t's values in a fresh contiguous tensor whose data starts `offset` floats into its storage."""
    import torch
    buf = torch.empty(t.numel() + offset + 4, device=t.device, dtype=t.dtype)
    v = buf[offset:offset + t.numel()].view(t.shape)
    v.copy_(t)
    return v


class Outs:
    """nbr int64 [nq, k], dist fp32 [nq, k] and alt uint32 [nq], each in the middle of a sentinel-filled buffer."""

    def __init__(self, nq, k, nbr=True, dist=True, alt=False):
        import torch
        self.nq, self.k = nq, k
        self.nbr_buf = torch.full((nq * k + 2 * GUARD,), SENTINEL64, dtype=torch.int64, device="cuda") if nbr else None
        self.dist_buf = torch.full((nq * k + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda") if dist else None
        self.alt_buf = torch.full((nq + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda") if alt else None

    def ptr(self, buf):
        return None if buf is None else buf[GUARD:].data_ptr()

    def check(self, written=True):
        """The guard regions are untouched; every output word is written (or, with written=False, none)."""
        for buf, s, w in ((self.nbr_buf, SENTINEL64, self.k), (self.dist_buf, SENTINEL, self.k), (self.alt_buf, SENTINEL, 1)):
            if buf is None:
                continue
            h = buf.cpu().numpy()
            assert (h[:GUARD] == s).all() and (h[-GUARD:] == s).all(), "write outside the output"
            body = h[GUARD:GUARD + self.nq * w]
            if written:
                assert not (body == s).any(), f"{int((body == s).sum())} output words left unwritten"
            else:
                assert (body == s).all(), "output written"

    def nbr(self):
        return self.nbr_buf[GUARD:GUARD + self.nq * self.k].view(self.nq, self.k).cpu().numpy()

    def dist(self):
        return self.dist_buf[GUARD:GUARD + self.nq * self.k].view(torch_f32()).view(self.nq, self.k).cpu().numpy()

    def alt(self):
        return self.alt_buf[GUARD:GUARD + self.nq].cpu().numpy().view(np.uint32)


def torch_f32():
    import torch
    return torch.float32


def _call(x, n, q_ptr, nq, d, k, outs, freq=None, off=None, n_tables=0, stream=None):
    import torch
    torch.cuda.synchronize()
    rc = _lib().evs_knn(x.data_ptr(), n, q_ptr, nq, d, k, outs.ptr(outs.nbr_buf), outs.ptr(outs.dist_buf),
                        None if freq is None else freq.data_ptr(), None if off is None else off.data_ptr(), n_tables,
                        outs.ptr(outs.alt_buf), stream)
    torch.cuda.synchronize()
    return rc


def _data(n, d, scale, seed):
    rng = np.random.default_rng(seed)
    if scale == "randn":
        return rng.standard_normal((n, d)).astype(np.float32)
    if scale == "offset":                                  # far from the origin: |x|² >> the distances
        return (rng.standard_normal((n, d)) * 0.25 + 4.0).astype(np.float32)
    return (rng.random((n, d)) * 0.02 - 0.01).astype(np.float32)     # embedding-table magnitudes


def _nq(n, qmode, nq, sms):
    """nq of a case: n when q is x, 2 SMs x 128 + 1 (one query block past splits = 1) for -1."""
    return n if qmode == "self" else 2 * sms * KQ + 1 if nq == -1 else nq


def _assert_claims(what, cfg):
    """The launch a case's description names is the one knn_config says it reaches."""
    assert ("k_knn<2>" in what) <= (cfg["kernel"] == "k_knn<2>") and ("k_knn<0>" in what) <= (cfg["kernel"] == "k_knn<0>")
    assert ("serial" in what) <= (cfg["norm"] == "serial") and ("butterfly" in what) <= (cfg["norm"] == "butterfly")
    assert ("scalar" in what) <= (cfg["staging"] == "scalar")
    assert ("splits = 1" in what) <= (cfg["splits"] == 1)
    assert ("splits = tiles" in what) <= (cfg["splits"] == cfg["tiles"] < MAXSPLITS)
    assert ("64 splits" in what) <= (cfg["splits"] == MAXSPLITS)
    assert ("empty ones" in what) <= (cfg["empty_splits"] > 0)
    assert ("between 1 and tiles" in what) <= (1 < cfg["splits"] < cfg["tiles"])


def _sample(nq, seed):
    """Every query of the first and the last query block, and a seeded sample of the others."""
    last = (nq - 1) // KQ * KQ
    s = set(range(min(KQ, nq))) | set(range(last, nq))
    if nq > 4 * KQ:
        s |= set(np.random.default_rng(seed).choice(nq, 512, replace=False).tolist())
    else:
        s = set(range(nq))
    return np.array(sorted(s))


# (n, nq, d, k, q mode, x offset in floats, scale, what the case is for); q mode: "self" = q is x (aliased), "slice" =
# q = x[n // 3 : n // 3 + nq], "sep" = a separate array
CASES = [
    (1000, 0, 16, 10, "self", 0, "randn", "splits = tiles, k_knn<2>, butterfly (Dp 16)"),
    (777, 0, 36, 10, "self", 0, "offset", "splits = tiles, k_knn<0>, serial (Dp 40)"),
    (300, 0, 64, 10, "self", 0, "randn", "splits = tiles, butterfly (Dp 64)"),
    (2500, 0, 8, 10, "self", 0, "tables", "splits between 1 and tiles, butterfly (Dp 8)"),
    (130, 0, 20, 10, "self", 0, "randn", "serial (Dp 24)"),
    (4100, 512, 24, 10, "sep", 0, "randn", "64 splits, empty ones, serial (Dp 24)"),
    (4100, 300, 48, 4, "sep", 0, "offset", "64 splits, empty ones, serial (Dp 48), k = 4"),
    (4100, 129, 16, 10, "sep", 0, "tables", "64 splits, empty ones, butterfly"),
    (3000, -1, 16, 10, "sep", 0, "randn", "splits = 1 (nq >= 2 SMs x 128), k_knn<2>"),
    (2000, -1, 56, 10, "sep", 0, "offset", "splits = 1, serial (Dp 56)"),
    (1000, 200, 40, 10, "slice", 0, "randn", "q a row slice of x, serial (Dp 40)"),
    (70, 0, 18, 10, "self", 0, "randn", "scalar staging (d % 4), serial (Dp 24), n not a multiple of 64"),
    (500, 0, 3, 10, "self", 0, "offset", "scalar staging (d % 4), Dp 8"),
    (640, 77, 16, 10, "sep", 1, "randn", "scalar staging (x 4 bytes off 16-byte alignment), k_knn<2>"),
    (640, 77, 64, 10, "sep", 1, "offset", "scalar staging (x off alignment), k_knn<0>, butterfly"),
    (640, 77, 24, 10, "slice", 1, "randn", "scalar staging (x off alignment), serial, q a slice"),
    (333, 0, 32, 1, "self", 0, "randn", "k = 1, butterfly (Dp 32)"),
    (1, 1, 16, 10, "sep", 0, "randn", "n = 1: no neighbours"),
    (6, 0, 16, 10, "self", 0, "randn", "n <= k"),
    (11, 0, 40, 10, "self", 0, "randn", "n = k + 1"),
    (12000, 1, 64, 10, "sep", 0, "randn", "nq = 1, 64 splits"),
    (5000, 1, 12, 4, "sep", 0, "offset", "nq = 1, k = 4, k_knn<2> (Dp 16)"),
    (901, 130, 28, 10, "sep", 0, "randn", "nq not a multiple of 128, butterfly (Dp 32)"),
    (2048, 0, 44, 10, "self", 0, "tables", "serial (Dp 48)"),
    (1500, 1000, 50, 4, "sep", 0, "randn", "scalar staging (d % 4), serial (Dp 56)"),
    (800, 0, 60, 10, "self", 0, "offset", "butterfly (Dp 64), d % 8"),
]


def _case_id(c):
    return f"n{c[0]}-nq{c[1]}-d{c[2]}-k{c[3]}-{c[4]}-off{c[5]}-{c[6]}"


def _run_case(n, nq, d, k, qmode, x_off, scale, stream=None):
    import torch
    sms = _sms()
    nq = _nq(n, qmode, nq, sms)
    seed = n * 131 + d * 7 + nq
    x = _data(n, d, scale, seed)
    xd = _placed(torch.from_numpy(x).cuda(), x_off)
    if qmode == "self":
        q, q_ptr = x, xd.data_ptr()
    elif qmode == "slice":
        a = n // 3
        q, q_ptr = x[a:a + nq], xd[a:a + nq].data_ptr()
    else:
        q = _data(nq, d, scale, seed + 1)
        if scale != "tables":                              # queries near database rows: close neighbours and near-ties
            src = np.random.default_rng(seed + 2).integers(0, n, nq)
            q[: nq // 2] = x[src[: nq // 2]] + q[: nq // 2] * 1e-3
        qd = torch.from_numpy(q).cuda()
        q_ptr = qd.data_ptr()
    cfg = knn_config(n, nq, d, sms, x_off == 0)
    outs = Outs(nq, k)
    rc = _call(xd, n, q_ptr, nq, d, k, outs, stream=stream)
    assert rc == 0, (rc, _lib().evs_last_error())
    outs.check()
    check_knn(x, q, outs.nbr(), outs.dist(), k, rows=_sample(nq, seed))
    return cfg


@gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_knn_within_float64_bound(case):
    n, nq, d, k, qmode, x_off, scale, what = case
    cfg = _run_case(n, nq, d, k, qmode, x_off, scale)
    _assert_claims(what, cfg)                          # the launch the case is for was reached on this device


@gpu
def test_caller_supplied_stream():
    import torch
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    _run_case(4100, 300, 16, 10, "sep", 0, "randn", stream=s.cuda_stream)
    _run_case(2000, 1000, 40, 10, "slice", 0, "offset", stream=s.cuda_stream)


@gpu
def test_no_queries_launches_nothing():
    import torch
    x = torch.randn((100, 16), device="cuda")
    outs = Outs(4, 10, alt=True)
    off = torch.zeros(2, dtype=torch.int64, device="cuda")
    assert _call(x, 100, x.data_ptr(), 0, 16, 10, outs, off=off, n_tables=1) == 0
    outs.check(written=False)


# ---- exact arithmetic: ties broken by index, bit for bit --------------------------------------------------------------

def _int_data(n, d, lo, hi, seed, copies=True):
    """Integers in [lo, hi]; with `copies`, blocks of identical rows spread over quads, tiles and splits."""
    rng = np.random.default_rng(seed)
    x = rng.integers(lo, hi + 1, (n, d)).astype(np.float32)
    if copies and n > 200:
        for src in (3, 70, n // 2):
            for j in range(1, 7):
                x[(src + j * 61 + j * j * 67) % n] = x[src]
    return x


EXACT = [(1000, 0, 3, -4, 4), (1000, 0, 4, -4, 4), (1000, 0, 16, -4, 4), (1000, 0, 64, -4, 4),
         (4100, 512, 3, -4, 4), (4100, 300, 16, -1, 1), (4100, 400, 64, -4, 4), (4100, 129, 20, -2, 2),
         (650, 0, 36, -1, 1), (300, 77, 4, -4, 4)]


@gpu
@pytest.mark.parametrize("k", [1, 4, 10])
@pytest.mark.parametrize("n,nq,d,lo,hi", EXACT)
def test_exact_ties_equal_the_oracle(n, nq, d, lo, hi, k):
    """Small-integer data: the kernel equals oracle.altkeys.knn_bruteforce exactly, ids and dist, every tie broken by
    row index.  Blocks of identical rows: entry [0] is the lowest-indexed copy, not the query itself.  nq = 0: q is x."""
    import torch
    x = _int_data(n, d, lo, hi, seed=n + d + hi)
    xd = torch.from_numpy(x).cuda()
    if nq:
        rng = np.random.default_rng(d)
        q = rng.integers(lo, hi + 1, (nq, d)).astype(np.float32)
        q[::3] = x[rng.integers(0, n, len(q[::3]))]            # queries that are database rows, copies included
        q[1] = x[70]
        qd = torch.from_numpy(q).cuda()
        q_ptr = qd.data_ptr()
    else:
        q, q_ptr = x, xd.data_ptr()
    outs = Outs(q.shape[0], k)
    assert _call(xd, n, q_ptr, q.shape[0], d, k, outs) == 0
    outs.check()
    want, want_d = exact_oracle(x, None if not nq else q, k)
    got, got_d = outs.nbr(), outs.dist()
    bad = np.argwhere((got != want) | (got_d != want_d))
    assert len(bad) == 0, (f"{len(bad)} entries differ, first query {bad[0][0]}: {got[bad[0][0]].tolist()} / "
                           f"{got_d[bad[0][0]].tolist()} vs {want[bad[0][0]].tolist()} / {want_d[bad[0][0]].tolist()}")
    if not nq:
        # the copies of row 3 tie at the minimum: the lowest-indexed one is dropped, the others open the list in index order
        dup = np.nonzero((x == x[3]).all(axis=1))[0]
        assert len(dup) >= 7
        m = min(k, len(dup) - 1)
        for r in dup:
            assert got[r, :m].tolist() == dup[1:1 + m].tolist(), (r, got[r].tolist(), dup.tolist())


# ---- special values ------------------------------------------------------------------------------------------------

PATTERNS = [0x7FFFFFFF, 0xFFFFFFFF, 0x7FC00000, 0x7F800000, 0xFF800000, 0x7F7FFFFF]   # NaNs, ±Inf, FLT_MAX


def _poisoned(n, d, seed):
    """randn rows; every pattern once as a whole row and once as one element of a row (the last column for some)."""
    import torch
    x = np.random.default_rng(seed).standard_normal((n, d)).astype(np.float32)
    xi = x.view(np.int32)
    rows = []
    for j, p in enumerate(PATTERNS):
        pv = np.array([p], np.uint32).view(np.int32)[0]
        r = 5 + 97 * j
        xi[r, :] = pv
        r2 = r + 40
        xi[r2, (j * 5) % d if j % 2 else d - 1] = pv
        rows += [r, r2]
    return x, rows


@gpu
@pytest.mark.parametrize("mode", ["self", "database", "query"])
@pytest.mark.parametrize("d", [16, 20, 36, 64])
def test_nonfinite_rows_are_never_neighbours(d, mode):
    """NaN (the GPU's own 0x7FFFFFFF and its negative, the quiet 0x7FC00000), ±Inf and FLT_MAX as a whole row and as one
    element, at butterfly (16, 64) and serial (20, 36) norm widths, in the database, in the queries, or both (q is x).
    Such rows are never returned; such queries get −1 and a non-finite dist everywhere; every other list is held to the
    bound."""
    import torch
    n = 700
    xp, rows = _poisoned(n, d, seed=d)
    clean = np.random.default_rng(d + 1).standard_normal((n, d)).astype(np.float32)
    if mode == "self":
        x, q = xp, xp
    elif mode == "database":
        x, q = xp, clean[:300]
    else:
        x, q = clean, xp
    xd, qd = torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda()
    outs = Outs(q.shape[0], 10)
    assert _call(xd, n, xd.data_ptr() if mode == "self" else qd.data_ptr(), q.shape[0], d, 10, outs) == 0
    outs.check()
    nbr = outs.nbr()
    if mode != "query":
        assert not np.isin(nbr, rows).any(), "a non-finite row was returned"
    if mode != "database":
        assert (nbr[rows] == -1).all(), f"non-finite queries got neighbours: {nbr[rows].tolist()}"
        assert not np.isfinite(outs.dist()[rows]).any(), f"non-finite queries got finite distances: {outs.dist()[rows].tolist()}"
    check_knn(x, q, nbr, outs.dist(), 10)


@gpu
@pytest.mark.parametrize("d", [16, 20, 36, 64])
def test_nonfinite_rows_get_and_give_no_alt_key(d):
    """Through generate_alt_keys: a non-finite row gets alt key 0 and is nobody's alt key; the other rows' keys equal the
    oracle's wherever the bound leaves the choice unambiguous."""
    p = pkg()
    x, rows = _poisoned(700, d, seed=d + 7)
    tables = [x[:300], x[300:301], x[301:]]
    freq = [np.random.default_rng(d).permutation(t.shape[0]).astype(np.uint32) for t in tables]
    got = np.concatenate(p.altkeys.generate_alt_keys(tables, freq))
    assert (got[rows] == 0).all(), f"non-finite rows {rows} got alt keys {got[rows].tolist()}"
    off = np.array([0, 300, 301, 700])
    gl = np.where(got > 0, off[np.maximum(got % 100, 1) - 1] + got // 100, -1)
    assert not np.isin(gl, rows).any(), "a non-finite row became an alt key"
    _check_alt_unambiguous(x, np.concatenate(freq), got, off)


# ---- the C-ABI -----------------------------------------------------------------------------------------------------

@gpu
def test_alt_only_and_guard_regions():
    """nbr = dist = NULL with only alt, and all three inside sentinel-filled guards: nothing outside them is written, and
    alt equals the popularity pick of the neighbours the same call returns with nbr (exact-integer data: the oracle's)."""
    import torch
    x = _int_data(3000, 16, -3, 3, seed=5)
    n = x.shape[0]
    off = np.array([0, 1, 1000, 1064, 3000], np.int64)
    freq = np.random.default_rng(5).integers(0, 4, n).astype(np.uint32)
    xd = torch.from_numpy(x).cuda()
    offd = torch.from_numpy(off).cuda()
    fd = torch.from_numpy(freq.view(np.int32)).cuda()
    a = Outs(n, 10, nbr=False, dist=False, alt=True)
    assert _call(xd, n, xd.data_ptr(), n, 16, 10, a, freq=fd, off=offd, n_tables=4) == 0
    a.check()
    b = Outs(n, 10, alt=True)
    assert _call(xd, n, xd.data_ptr(), n, 16, 10, b, freq=fd, off=offd, n_tables=4) == 0
    b.check()
    assert np.array_equal(a.alt(), b.alt())
    want = np.concatenate(altkeys.alt_keys([x[off[t]:off[t + 1]] for t in range(4)],
                                           [freq[off[t]:off[t + 1]] for t in range(4)]))
    assert np.array_equal(a.alt(), want)
    want_n, want_d = exact_oracle(x, None, 10)
    assert np.array_equal(b.nbr(), want_n) and np.array_equal(b.dist(), want_d)


@gpu
def test_bad_arguments_are_refused():
    """d = 0 and 65, k = 0 and 11, n = 0, alt without table_off: EVS_ERR_INVALID, nothing written, no CUDA error left for
    the next call."""
    import torch
    x = torch.randn((200, 64), device="cuda").contiguous()
    xs = x[:, :16].contiguous()
    off = torch.tensor([0, 200], dtype=torch.int64, device="cuda")
    bad = [dict(d=0), dict(d=65), dict(k=0), dict(k=11), dict(n=0), dict(alt=True, off=None)]
    for kw in bad:
        d, k, n = kw.get("d", 16), kw.get("k", 10), kw.get("n", 200)
        outs = Outs(50, 11, alt=kw.get("alt", False))
        xx = x if d > 16 else xs
        rc = _call(xx, n, xx.data_ptr(), 50, d, k, outs, off=kw.get("off", None), n_tables=1 if "off" in kw else 0)
        assert rc == -1, (kw, rc)
        outs.check(written=False)
        ok = Outs(50, 10, alt=True)
        assert _call(xs, 200, xs.data_ptr(), 50, 16, 10, ok, off=off, n_tables=1) == 0, (kw, _lib().evs_last_error())
        ok.check()


# ---- alt keys ------------------------------------------------------------------------------------------------------

def _check_alt_unambiguous(x, freq, got, off, min_share=0.8):
    """got (uint32 keys of every row of x, tables at `off`) equals the oracle's pick for every row whose neighbour set
    and popularity pick the bound cannot change; at least min_share of the finite rows qualify."""
    n = x.shape[0]
    elig = _eligible_rows(x)
    with np.errstate(invalid="ignore", over="ignore"):              # NaN / Inf rows rank last in the oracle
        want = np.concatenate(altkeys.alt_keys([x[off[t]:off[t + 1]] for t in range(len(off) - 1)],
                                               [freq[off[t]:off[t + 1]] for t in range(len(off) - 1)]))
    checked = 0
    for b0 in range(0, n, 256):
        blk = np.arange(b0, min(n, b0 + 256))
        v, E = _bounds(x, x[blk])
        for j, i in enumerate(blk):
            if not elig[i]:
                continue
            o = np.argsort(v[j], kind="stable")[:13]
            vo, Eo = v[j][o], E[j][o]
            finite = np.isfinite(vo)
            if finite.sum() < 12:
                continue
            # entry [0] and the set of the next 10 are fixed when the gaps around them exceed the bound
            if vo[0] + Eo[0] >= vo[1] - Eo[1] or vo[10] + Eo[10] >= vo[11] - Eo[11]:
                continue
            f = freq[o[1:11]].astype(np.int64)
            if (f == f.max()).sum() > 1:                   # a popularity tie is decided by the order: not checked here
                continue
            checked += 1
            assert got[i] == want[i], f"row {i}: alt key {got[i]} vs {want[i]}"
    assert checked >= min_share * elig.sum(), (checked, int(elig.sum()))


@gpu
def test_alt_keys_on_exact_data_in_small_query_chunks():
    """generate_alt_keys in query chunks of 100 rows (not a multiple of 128), tables of 1, 63, 64, 65 and more rows,
    frequencies >= 2^31 (through the int32 conversion) with ties, and freq=None: the oracle's keys, exactly."""
    p = pkg()
    rng = np.random.default_rng(13)
    sizes = [1, 63, 64, 65, 1, 700, 2, 190]
    x = _int_data(sum(sizes), 12, -2, 2, seed=13)
    off = np.concatenate([[0], np.cumsum(sizes)])
    tables = [x[off[t]:off[t + 1]] for t in range(len(sizes))]
    big = (np.uint32(2 ** 31) + rng.integers(0, 3, x.shape[0]).astype(np.uint32)).astype(np.uint32)
    big[::7] = np.uint32(2 ** 32 - 1)
    small = rng.integers(0, 3, x.shape[0]).astype(np.uint32)
    for f in (None, small, big):
        fl = None if f is None else [f[off[t]:off[t + 1]] for t in range(len(sizes))]
        got = p.altkeys.generate_alt_keys(tables, fl, query_chunk=100)
        want = altkeys.alt_keys(tables, fl)
        for t in range(len(sizes)):
            assert got[t].dtype == np.uint32 and np.array_equal(got[t], want[t]), (t, None if f is None else f.max())


@gpu
def test_alt_keys_on_random_data_where_unambiguous():
    """Random tables (the former test's shapes, randn and embedding-table magnitudes), distinct frequencies: the oracle's
    keys wherever the bound leaves the neighbour set fixed."""
    p = pkg()
    rng = np.random.default_rng(11)
    for scale, d in (("randn", 16), ("tables", 36)):
        sizes = (400, 30, 7, 900, 3)
        x = _data(sum(sizes), d, scale, seed=d)
        off = np.concatenate([[0], np.cumsum(sizes)])
        freq = rng.permutation(x.shape[0]).astype(np.uint32)
        tables = [x[off[t]:off[t + 1]] for t in range(len(sizes))]
        got = np.concatenate(p.altkeys.generate_alt_keys(tables, [freq[off[t]:off[t + 1]] for t in range(len(sizes))]))
        _check_alt_unambiguous(x, freq, got, off)
