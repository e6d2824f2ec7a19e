"""The dct packer's kernels against an extended-precision DCT.

The reference (signal_packer_dct.cpp) defines the coefficients as a truncated O(n^2) sum.  Here that sum is
evaluated exactly enough to decide the truncation: direct sums in np.longdouble (64-bit mantissa on x86-64)
over a 4n-entry cosine table, with the scale constants the kernels use.  With e the exact value and
delta = 2^-44 * scale * sum|input| (about 40x the error of an FP64 FFT), a kernel's value must be
trunc(e) wherever trunc(e - delta) == trunc(e + delta), one of the two elsewhere, and 0x80000000 where
|e| >= 2^31 (the reference's x86-64 conversion).  Every power-of-two length from 2 to 8192 runs, so both
fast-path kernel families (n < 16 and the half-length FFT with each radix-8 / radix-4 / radix-2 tail) and
both word kernels (four-channel groups and the generic one) are covered, over 1- to 4-byte samples and
inputs at the edges of the sample range and of the Makhoul reordering.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import has_ref

LD = np.longdouble
CS0 = LD(float(np.float32(1 / np.sqrt(2.0))))       # the k = 0 factor, float32(1/sqrt 2) as the kernels use it
DELTA_REL = LD(2.0) ** -44
UNDECIDED_MAX = 0.001                                 # share of values in the band, per case
INT32_MIN = -(1 << 31)

needs_longdouble = pytest.mark.skipif(np.finfo(LD).nmant < 63, reason="np.longdouble has no 64-bit mantissa here")


# ---- exact transforms (CPU) ---------------------------------------------------------------------------
def _cos_table(n):
    """cos(pi j / 2n) for j < 4n."""
    pi = np.arctan(LD(1)) * 4
    return np.cos(pi * np.arange(4 * n).astype(LD) / LD(2 * n))


def _cos_block(table, n, i, k):
    """cos(pi (2i+1) k / 2n) for the sample indices i (rows) and the frequencies k (columns); the integer
    argument is reduced mod 4n before the table look-up."""
    return table[np.outer(2 * np.asarray(i, np.int64) + 1, np.asarray(k, np.int64)) % (4 * n)]


def _sums(rows, n, block):
    """rows (R, n) longdouble -> (R, n): column j of the result is rows @ block(cols) for column chunks."""
    out = np.zeros(rows.shape, LD)
    live = np.flatnonzero(np.any(rows != 0, axis=1))  # all-zero rows transform to zero
    if live.size == 0:
        return out
    r = rows[live]
    step = max(1, (1 << 20) // n)
    chunks = [np.arange(c, min(n, c + step)) for c in range(0, n, step)]
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        parts = list(ex.map(lambda cols: r @ block(cols), chunks))
    out[live] = np.concatenate(parts, axis=1)
    return out


def dct2_exact(x):
    """Forward DCT of int rows (R, n) as the kernels scale it: X[k] = cs_k sqrt(2/n)/128 sum_i x_i
    cos(pi (2i+1) k / 2n), cs_0 = float32(1/sqrt 2), else 1.  Returns (X, delta), both longdouble."""
    x = np.atleast_2d(np.asarray(x, np.int64))
    n = x.shape[1]
    tab, idx = _cos_table(n), np.arange(n)
    s = _sums(x.astype(LD), n, lambda k: _cos_block(tab, n, idx, k))
    scale = np.full(n, np.sqrt(LD(2) / LD(n)) / 128)
    scale[0] *= CS0
    return s * scale, DELTA_REL * scale * np.abs(x).sum(axis=1, keepdims=True).astype(LD)


def dct3_exact(c):
    """Inverse DCT of int coefficient rows (R, n) as the kernels scale it: x[i] = 128 sqrt(2/n) (T_0 +
    sum_{k>0} T_k cos(pi (2i+1) k / 2n)), T_0 = float32(1/sqrt 2) c_0 (an exact product), T_k = c_k.
    Returns (x, delta), both longdouble."""
    t = np.atleast_2d(np.asarray(c, np.int64)).astype(LD)
    n = t.shape[1]
    t[:, 0] *= CS0
    tab, idx = _cos_table(n), np.arange(n)
    s = _sums(t, n, lambda i: _cos_block(tab, n, i, idx).T)
    scale = 128 * np.sqrt(LD(2) / LD(n))
    return s * scale, DELTA_REL * scale * np.abs(t).sum(axis=1, keepdims=True)


def x86_trunc(v):
    """double -> int32 as the reference's x86-64 build converts (cvttsd2si): toward zero, 0x80000000 out of range."""
    out = np.trunc(np.clip(v, LD(-(2 ** 32)), LD(2 ** 32))).astype(np.int64)
    out[np.abs(v) >= LD(2 ** 31)] = INT32_MIN
    return out


def truncation_band(e, delta):
    """(lo, hi): the converted value at e - delta and at e + delta.  Where they agree the result is decided."""
    return x86_trunc(e - delta), x86_trunc(e + delta)


# ---- the packer's integer steps, restated ------------------------------------------------------------
def wrap32(v):
    return ((np.asarray(v, np.int64) + (1 << 31)) % (1 << 32)) - (1 << 31)


def average_32(row):
    """utils.cpp:30-40: the int64 sum divided as UNSIGNED 64-bit by the length, narrowed to int32."""
    s = int(np.asarray(row, np.int64).sum())
    return int(wrap32(((s % (1 << 64)) // len(row)) % (1 << 32)))


def samples_of(raw, bps, ch, ns):
    """interleaved [ns][ch][bps] little-endian bytes -> int64 [ch][ns], sign-extended."""
    b = np.asarray(raw, np.uint8).reshape(ns, ch, bps).astype(np.int64)
    v = sum(b[:, :, k] << (8 * k) for k in range(bps))
    return (((v + (1 << (8 * bps - 1))) % (1 << (8 * bps))) - (1 << (8 * bps - 1))).T


def sext16(words):
    return ((np.asarray(words, np.int64) + 0x8000) & 0xFFFF) - 0x8000


def decoded_coefficients(post_stencil_words):
    """Coefficient words the decoder reconstructs from the dct packer's two byte planes: the low 16 bits
    sign-extended, then the prefix XOR and the prefix sum of +128 (signal_packer_dct.cpp:137-146), mod 2^32."""
    d = np.bitwise_xor.accumulate(sext16(post_stencil_words).astype(np.uint32))
    return wrap32(np.cumsum(d.astype(np.uint64) + 128, dtype=np.uint64) % (1 << 32))


def stencil(coefs):
    """delta - 128, then XOR with the previous delta (signal_packer_dct.cpp:117-119), over the flat array."""
    x = np.asarray(coefs, np.int64) % (1 << 32)
    d = (x - np.concatenate([[0], x[:-1]]) - 128) % (1 << 32)
    return wrap32(d ^ np.concatenate([[0], d[:-1]]))


def mean24(hdr, c):
    v = int(hdr[3 * c]) | (int(hdr[3 * c + 1]) << 8) | (int(hdr[3 * c + 2]) << 16)
    return v - (1 << 24) if v & 0x800000 else v


# ---- frames -----------------------------------------------------------------------------------------
FRAME_KINDS = ("ecg", "noise", "cosines", "impulses", "alternating", "const_min", "const_max", "zeros")


def make_frame(oracle, kind, bps, ch, ns, seed):
    lo, hi = -(1 << (8 * bps - 1)), (1 << (8 * bps - 1)) - 1
    rng = np.random.default_rng(seed)
    i = np.arange(ns)
    lg = ns.bit_length() - 1
    if kind == "ecg":
        amp = 20000 if bps >= 3 else (3000 if bps == 2 else 100)
        return oracle.synth_ecg(seed, 1, bps, ch, ns, amplitude=amp).reshape(-1)
    if kind == "noise":
        x = rng.integers(lo, hi + 1, (ns, ch), dtype=np.int64)
    elif kind == "cosines":
        # the Makhoul butterfly pairs k with M - k and n - k (M = n/2): its special indices.  A dither of a
        # few LSB keeps most of these spectra from being one exact spike: the inverse of c at k = M alone
        # is +-128 c / sqrt(n), an exact integer for n a power of 4, which no truncation rule decides.
        m = ns // 2
        ks = (0, 1, m - 1, m, m + 1, ns - 1)
        a = hi - 2
        x = np.stack([np.rint(a * np.cos(np.pi * (2 * i + 1) * ks[(c + lg) % 6] / (2 * ns))) for c in range(ch)], axis=1)
        x = x.astype(np.int64) + rng.integers(-2, 3, (ns, ch))
    elif kind == "impulses":
        # the ends of the even / odd reordering
        x = np.zeros((ns, ch), np.int64)
        for c in range(ch):
            x[(0, 1, ns - 2, ns - 1)[(c + lg) % 4], c] = hi if c % 2 == 0 else -hi
    elif kind == "alternating":
        x = np.stack([np.where((i + c) % 2 == 0, hi, -hi) for c in range(ch)], axis=1)
    elif kind == "const_min":
        x = np.full((ns, ch), lo, np.int64)
    elif kind == "const_max":
        x = np.full((ns, ch), hi, np.int64)
    else:
        x = np.zeros((ns, ch), np.int64)
    return np.asarray(x, np.int64).astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].reshape(-1)


# (ns, bps, ch, frame kinds): every power of two from 2 to 8192; bps 1-4; ch 1, 3, 4, 12, so that the
# four-channel-group word kernels (ch % 4 == 0, ns % 1024 == 0) and the generic ones both run.  From 4096
# up the O(n^2) sums dominate: two frames with content, plus the constant frames (free, they transform to 0).
# Short frames get more noise and ECG frames, up to MIN_VALUES values per case, so that one value whose
# exact transform happens to be an integer stays within the undecided share.
CHEAP = ("const_min", "const_max", "zeros")
MIN_VALUES = 4096


def with_filler(ns, ch, kinds):
    extra = max(0, -(-MIN_VALUES // (ns * ch)) - len(kinds))
    return tuple(kinds) + ("noise", "ecg") * (extra // 2) + ("noise",) * (extra % 2)


DCT_EXACT_CASES = [(ns, bps, ch, with_filler(ns, ch, kinds)) for ns, bps, ch, kinds in [
    (2, 1, 1, FRAME_KINDS), (2, 4, 12, FRAME_KINDS),
    (4, 2, 3, FRAME_KINDS), (4, 4, 4, FRAME_KINDS),
    (8, 3, 12, FRAME_KINDS), (8, 4, 1, FRAME_KINDS),
    (16, 1, 4, FRAME_KINDS), (16, 4, 3, FRAME_KINDS),
    (32, 2, 12, FRAME_KINDS), (64, 3, 1, FRAME_KINDS),
    (128, 4, 4, FRAME_KINDS), (256, 1, 3, FRAME_KINDS),
    (512, 2, 4, FRAME_KINDS), (1024, 4, 12, FRAME_KINDS), (1024, 1, 3, FRAME_KINDS),
    (2048, 3, 4, FRAME_KINDS), (2048, 2, 1, FRAME_KINDS),
    (4096, 4, 3, ("ecg", "noise") + CHEAP), (4096, 1, 4, ("cosines", "impulses") + CHEAP),
    (8192, 4, 3, ("noise", "alternating") + CHEAP), (8192, 2, 4, ("ecg", "cosines") + CHEAP),
]]


def case_id(c):
    return f"n{c[0]}-bps{c[1]}-ch{c[2]}"


def case_frames(oracle, ns, bps, ch, kinds):
    return np.stack([make_frame(oracle, k, bps, ch, ns, 1000 * ns + 10 * bps + j) for j, k in enumerate(kinds)])


def check_against_band(got, e, delta, mod, what, offset=0):
    """got == x86_trunc(e) + offset (mod `mod`) where the band decides the value, either candidate elsewhere.

    A value with band delta falls in it with a chance of about 2 delta, so two kinds of undecided value are
    excused from the undecided share, which must stay at UNDECIDED_MAX: values whose band is wider than
    2^-12 (full-range 4-byte inputs, whose sums cancel from near 2^40 down to the int32 range), and exact
    integers (a spectrum that is one coefficient at k = M for n a power of 4, or the DC alone for n = 2 4^j),
    which no truncating implementation decides.  At least half of a case's values must be decided."""
    lo, hi = truncation_band(e, delta)
    lo_m, hi_m, got_m = wrap32(lo + offset) % mod, wrap32(hi + offset) % mod, np.asarray(got, np.int64) % mod
    undecided = lo != hi
    bad = np.where(undecided, (got_m != lo_m) & (got_m != hi_m), got_m != lo_m)
    if bad.any():
        where = np.argwhere(bad)[:8]
        detail = [(tuple(int(v) for v in w), int(got_m[tuple(w)]), int(lo_m[tuple(w)]), int(hi_m[tuple(w)]), float(e[tuple(w)]))
                  for w in where]
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} values off the exact transform "
                             f"(index, got, want, want if undecided, exact): {detail}")
    delta = np.broadcast_to(delta, e.shape)
    excused = undecided & ((delta >= LD(2) ** -12) | (np.abs(e - np.rint(e)) <= delta / 256))
    share = float((undecided & ~excused).mean())
    print(f"{what}: {int(undecided.sum())} of {undecided.size} values undecided, {int(excused.sum())} of them excused "
          f"(wide band or exact integer); the others are {100 * share:.4f} %")
    assert undecided.mean() <= 0.5, (what, float(undecided.mean()))
    assert share <= UNDECIDED_MAX, (what, share)


# ---- CPU tests -------------------------------------------------------------------------------------------
@needs_longdouble
@pytest.mark.parametrize("n", [2, 3, 16, 64])
def test_exact_transforms_agree_with_mpmath(n):
    """The longdouble helpers against 40-digit sums: their own error is far inside the acceptance band."""
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 40
    rng = np.random.default_rng(n)
    x = np.concatenate([rng.integers(-(1 << 31), 1 << 31, (2, n)), np.full((1, n), (1 << 31) - 1)])
    cs0 = mp.mpf(float(np.float32(1 / np.sqrt(2.0))))
    for fwd in (True, False):
        e, delta = dct2_exact(x) if fwd else dct3_exact(x)
        worst = 0.0
        for r in range(x.shape[0]):
            for k in range(n):
                if fwd:
                    s = mp.fsum(int(x[r, i]) * mp.cos(mp.pi * (2 * i + 1) * k / (2 * n)) for i in range(n))
                    want = s * mp.sqrt(mp.mpf(2) / n) / 128 * (cs0 if k == 0 else 1)
                else:
                    s = cs0 * int(x[r, 0]) + mp.fsum(int(x[r, j]) * mp.cos(mp.pi * (2 * k + 1) * j / (2 * n)) for j in range(1, n))
                    want = s * 128 * mp.sqrt(mp.mpf(2) / n)
                top = float(e[r, k])   # the longdouble value is exactly top + the double that remains
                err = abs(mp.mpf(top) + mp.mpf(float(e[r, k] - LD(top))) - want)
                worst = max(worst, float(err / mp.mpf(float(delta[r, 0]))))
        print(f"n={n} {'forward' if fwd else 'inverse'}: largest error {worst:.3g} of the band")
        assert worst < 2 ** -10, (n, fwd, worst)


FULL_RANGE_NOISE = dict(bps=4, ch=12, ns=4096)


def full_range_noise_frame():
    """One 4-byte 12-channel frame of full-range noise: about 0.15 % of its decoded samples have an inverse
    sum outside int32."""
    x = np.random.default_rng(1).integers(-(1 << 31), 1 << 31, (4096, 12))
    return x.astype("<i4").view(np.uint8).reshape(-1)


@needs_longdouble
def test_out_of_range_inverse_sums_decode_to_integer_indefinite(oracle):
    """Where the exact inverse sum leaves the int32 range, the reference's x86-64 conversion gives
    0x80000000, so the decoded sample is 0x80000000 + the channel mean.  Pins the oracle (and, where it
    is built, the reference) to that, on the frame the GPU tests decode as well."""
    bps, ch, ns = FULL_RANGE_NOISE["bps"], FULL_RANGE_NOISE["ch"], FULL_RANGE_NOISE["ns"]
    raw = full_range_noise_frame()
    o = oracle.OraclePacker("dct", bps, ch, ns)
    stream = o.compress(raw)
    dec = samples_of(np.frombuffer(o.decompress(stream)[0], np.uint8), bps, ch, ns)
    ww, hdr = o.transform(raw)
    e, delta = dct3_exact(decoded_coefficients(ww).reshape(ch, ns))
    out = np.abs(e) - delta >= LD(2 ** 31)
    assert not ((np.abs(e) + delta >= LD(2 ** 31)) & ~out).any(), "a sum within the band of the int32 limit"
    n_out, n_pos = int(out.sum()), int((out & (e > 0)).sum())
    print(f"{n_out} of {out.size} inverse sums out of range, {n_pos} of them positive")
    assert n_out > 0 and n_pos > 0
    means = np.array([mean24(hdr, c) for c in range(ch)])[:, None]
    want = wrap32(INT32_MIN + np.broadcast_to(means, dec.shape))
    assert np.array_equal(dec[out], want[out])
    if has_ref():
        ref = oracle.RefPacker("dct", bps, ch, ns)
        assert ref.compress(raw) == stream
        rdec = samples_of(np.frombuffer(ref.decompress(stream)[0], np.uint8), bps, ch, ns)
        assert np.array_equal(rdec[out], want[out])


@needs_longdouble
def test_decoded_coefficient_derivation(oracle):
    """decoded_coefficients is what the oracle's decoder computes: re-stenciled it gives the sign-extended
    plane words back, and the oracle's inverse of those words is its decode of the stream."""
    for bps, ch, ns in ((4, 3, 64), (2, 4, 16)):
        o = oracle.OraclePacker("dct", bps, ch, ns)
        for kind in ("noise", "ecg", "alternating"):
            raw = make_frame(oracle, kind, bps, ch, ns, 7)
            ww, hdr = o.transform(raw)
            c = decoded_coefficients(ww)
            assert np.array_equal(stencil(c), sext16(ww))
            assert o.inverse(sext16(ww).astype(np.int32), hdr).tobytes() == o.decompress(o.compress(raw))[0]


# ---- GPU tests ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def R():
    torch = pytest.importorskip("torch")
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


def to_dev(a):
    import torch
    return torch.from_numpy(np.array(a, dtype=np.uint8, copy=True).reshape(-1)).cuda()


@needs_longdouble
@pytest.mark.gpu
@pytest.mark.timeout(300)
@pytest.mark.parametrize("ns,bps,ch,kinds", DCT_EXACT_CASES, ids=[case_id(c) for c in DCT_EXACT_CASES])
def test_dct_fast_forward_matches_exact_transform(R, oracle, ns, bps, ch, kinds):
    """Coefficients mod 2^16 (the two byte planes the packer keeps, stencil undone) equal the truncated
    exact transform of wrap32(sample - mean) outside the band; the means header equals the oracle's."""
    from test_gpu_parity import unstencil16
    raws = case_frames(oracle, ns, bps, ch, kinds)
    nfr = len(kinds)
    p = R.SignalPacker.new_dct(bps, ch, ns, max_batch_frames=nfr)
    planes, gh = p.debug_planes(to_dev(raws))
    p.close()
    o = oracle.OraclePacker("dct", bps, ch, ns)
    xs, got = [], []
    for f in range(nfr):
        hdr = o.transform(raws[f])[1]
        assert np.array_equal(gh[f], hdr), (kinds[f], "means header")
        smp = samples_of(raws[f], bps, ch, ns)
        means = [average_32(smp[c]) for c in range(ch)]
        assert [m & 0xFFFFFF for m in means] == [mean24(hdr, c) & 0xFFFFFF for c in range(ch)]
        xs.append(wrap32(smp - np.array(means)[:, None]))
        got.append(unstencil16(planes[f][0].astype(np.uint32) | (planes[f][1].astype(np.uint32) << 8)).reshape(ch, ns))
    e, delta = dct2_exact(np.concatenate(xs))
    assert np.abs(e).max() < LD(2 ** 31)
    check_against_band(np.concatenate(got), e, delta, 1 << 16, f"forward {case_id((ns, bps, ch))}")


@needs_longdouble
@pytest.mark.gpu
@pytest.mark.timeout(300)
@pytest.mark.parametrize("ns,bps,ch,kinds", DCT_EXACT_CASES, ids=[case_id(c) for c in DCT_EXACT_CASES])
def test_dct_fast_inverse_matches_exact_transform(R, oracle, ns, bps, ch, kinds):
    """The GPU's decode of the oracle's streams: every sample is wrap32(x86_trunc(e) + mean), cut to bps
    bytes, with e the exact inverse transform of the coefficient words the decoder reconstructs."""
    raws = case_frames(oracle, ns, bps, ch, kinds)
    nfr = len(kinds)
    o = oracle.OraclePacker("dct", bps, ch, ns)
    streams = [o.compress(r) for r in raws]
    p = R.SignalPacker.new_dct(bps, ch, ns, max_batch_frames=nfr)
    dec, status = p.decompress_stream(b"".join(streams), np.concatenate([[0], np.cumsum([len(s) for s in streams])]))
    p.close()
    assert not status.any(), status
    coefs, means, got = [], [], []
    for f in range(nfr):
        ww, hdr = o.transform(raws[f])
        assert o.inverse(sext16(ww).astype(np.int32), hdr).tobytes() == o.decompress(streams[f])[0]
        coefs.append(decoded_coefficients(ww).reshape(ch, ns))
        means.append([mean24(hdr, c) for c in range(ch)])
        got.append(samples_of(dec[f], bps, ch, ns))
    e, delta = dct3_exact(np.concatenate(coefs))
    check_against_band(np.concatenate(got), e, delta, 1 << (8 * bps), f"inverse {case_id((ns, bps, ch))}",
                       offset=np.array(means).reshape(-1, 1))
