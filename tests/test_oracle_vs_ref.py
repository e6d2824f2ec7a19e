"""Differential pinning of the oracle port to the UNMODIFIED reference on generated inputs: hzr streams,
CRC-32C, all four packers on random shapes, the plane-escalation rule and the pre-filters.  The answers
are stored as digests in tests/golden/ref_vectors.json (written by tests/golden/make_ref_vectors.py from
the input generators below; its "source" names the implementation that computed them), so the comparison
runs without the reference; where oracle/_ref/libref.so has been built the reference is held to the same
answers.  CPU only."""
import hashlib
import json
import os
import zlib

import numpy as np
import pytest

from conftest import GOLDEN_DIR, has_ref

VECTORS_PATH = os.path.join(GOLDEN_DIR, "ref_vectors.json")


@pytest.fixture(scope="module")
def vectors():
    with open(VECTORS_PATH) as f:
        return json.load(f)


def impls():
    return ["port", "reference"] if has_ref() else ["port"]


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


# ---- input generators and the answers recorded for them ----------------------------------------
def hzr_buffers():
    """hzr inputs across all three block modes, zero-run classes and block boundaries."""
    rng = np.random.default_rng(7)
    out = []
    for n in (1, 2, 3, 7, 22, 23, 278, 279, 1000, 16662, 16663, 33324, 65535, 65536, 65537, 140000):
        out.append(np.zeros(n, np.uint8))
        out.append(rng.integers(0, 256, n, dtype=np.uint8))
        out.append(rng.integers(0, 4, n, dtype=np.uint8))
        sparse = np.zeros(n, np.uint8)
        k = max(1, n // 50)
        sparse[rng.integers(0, n, k)] = rng.integers(1, 256, k, dtype=np.uint8)
        out.append(sparse)
        lap = np.clip(np.rint(rng.laplace(0, 6, n)), -120, 120).astype(np.int8).view(np.uint8)
        out.append(lap)
        out.append(np.full(n, 255, np.uint8))
    # near the COPY/HUFF boundary: skewed two-symbol data and nearly uniform data
    for p in (0.5, 0.9, 0.99):
        out.append((rng.random(65536) < p).astype(np.uint8) * 3 + 1)
    out.append(rng.integers(0, 200, 65536, dtype=np.uint8))
    out.append(rng.integers(1, 256, 300, dtype=np.uint8))
    return out


def hzr_answers(oracle, impl):
    out = []
    for buf in hzr_buffers():
        enc = oracle.hzr_encode(buf, impl)
        out.append({"n": int(buf.size), "len": len(enc), "sha256": sha(enc)})
    return out


CRC_SIZES = (0, 1, 2, 3, 4, 5, 63, 64, 65, 1000, 65536)


def crc32c_answers(oracle, impl):
    rng = np.random.default_rng(3)
    return [oracle.crc32c(rng.integers(0, 256, n, dtype=np.uint8), impl) for n in CRC_SIZES]


PACKER_KINDS = ("xdelta_hzr", "hzr", "hadamard", "dct")


def packer_shapes(kind):
    """14 random shapes and random-walk frames of one packer kind."""
    rng = np.random.default_rng(zlib.crc32(kind.encode()) & 0xFFFF)
    for _ in range(14):
        bps = int(rng.integers(1, 5))
        ch = int(rng.integers(1, 5))
        if kind in ("hadamard", "dct"):
            ns = 1 << int(rng.integers(3, 10 if kind == "dct" else 13))
        else:
            ns = int(rng.integers(1, 30000))
        nb = int(rng.integers(1, 5))
        amp = 1 << int(rng.integers(2, 8 * bps))
        walk = np.cumsum(rng.integers(-amp // 16 - 1, amp // 16 + 2, (ns, ch)), axis=0)
        x = np.clip(walk, -(1 << (8 * bps - 1)), (1 << (8 * bps - 1)) - 1).astype(np.int32)
        raw = x.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].copy().reshape(-1)
        yield bps, ch, ns, nb, raw


def packer_answers(oracle, impl, kind):
    out = []
    for bps, ch, ns, nb, raw in packer_shapes(kind):
        p = oracle.make_packer(kind, bps, ch, ns, nb, impl)
        reps = []
        for _ in range(2):  # twice: the xdelta plane-count state carries over
            comp = p.compress(raw)
            dec, used = p.decompress(comp)
            reps.append({"len": len(comp), "sha256": sha(comp), "dec_sha256": sha(dec), "used": int(used)})
        out.append({"bps": bps, "ch": ch, "ns": ns, "nb": nb, "reps": reps})
    return out


def escalation_frames():
    rng = np.random.default_rng(11)
    for _ in range(40):
        bps = int(rng.integers(2, 5))
        ch = int(rng.integers(1, 4))
        ns = int(rng.integers(16, 400))
        nb0 = int(rng.integers(1, bps + 1))
        amp = 1 << int(rng.integers(2, 8 * bps - 1))
        x = rng.integers(-amp, amp, (ns, ch)).astype(np.int32)
        raw = x.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].copy().reshape(-1)
        yield bps, ch, ns, nb0, raw


def escalation_answers(oracle, impl):
    out = []
    for bps, ch, ns, nb0, raw in escalation_frames():
        comp = oracle.make_packer("xdelta_hzr", bps, ch, ns, nb0, impl).compress(raw)
        out.append({"len": len(comp), "sha256": sha(comp)})
    return out


# the band-pass the reference's own pipeline uses (rspt_test.cpp:123-125) and two shorter filters
IIR5_N = [1.00000000000, -3.14332095199, 3.70064088865, -1.97083923944, 0.41351972908]
IIR5_D = [0.06722876941, 0.00000000000, -0.13445753881, 0.00000000000, 0.06722876941]


def prefilter_answers(oracle, impl):
    """oracle_prefilter_iir / _fir, or the compiled i_filter (lib_filter/*.cpp) driven the way
    rspt_test.cpp:116-136 drives it: the filtered frame bytes, including the state that leaks from one
    channel into the next through the single filter object."""
    rng = np.random.default_rng(3)
    out = []
    for bps, ch, ns in ((3, 12, 8192), (4, 3, 1000), (2, 2, 500), (1, 1, 64)):
        raws = oracle.synth_ecg(5, 2, bps, ch, ns, amplitude=20000 if bps >= 3 else (3000 if bps == 2 else 50))
        for f in raws:
            for nc, init in ((5, 2000), (3, 100), (2, 0), (4, 7)):
                y = oracle.prefilter_iir(f, bps, ch, ns, IIR5_N[:nc], IIR5_D[:nc], init, impl)
                out.append({"filter": f"iir{nc}", "bps": bps, "ch": ch, "ns": ns, "sha256": sha(y)})
            for K in (1, 5, 31):
                k = rng.normal(size=K)
                k /= np.abs(k).sum()
                y = oracle.prefilter_fir(f, bps, ch, ns, k, impl)
                out.append({"filter": f"fir{K}", "bps": bps, "ch": ch, "ns": ns, "sha256": sha(y)})
    return out


def all_answers(oracle, impl):
    """Everything ref_vectors.json records, computed by `impl`."""
    return {"hzr": hzr_answers(oracle, impl), "crc32c": crc32c_answers(oracle, impl),
            "packers": {k: packer_answers(oracle, impl, k) for k in PACKER_KINDS},
            "escalation": escalation_answers(oracle, impl), "prefilter": prefilter_answers(oracle, impl)}


# ---- tests -----------------------------------------------------------------------------------
def test_hzr_stream_bit_exact(oracle, vectors):
    for impl in impls():
        assert hzr_answers(oracle, impl) == vectors["hzr"], impl
    for buf in hzr_buffers():
        enc = oracle.hzr_encode(buf, "port")
        for impl in impls():
            dec, ok = oracle.hzr_decode(enc, buf.size, impl)
            assert ok and dec == buf.tobytes(), (buf.size, impl)


def test_crc32c_matches(oracle, vectors):
    for impl in impls():
        assert crc32c_answers(oracle, impl) == vectors["crc32c"], impl


@pytest.mark.parametrize("kind", PACKER_KINDS)
def test_packers_random_shapes(oracle, vectors, kind):
    for impl in impls():
        assert packer_answers(oracle, impl, kind) == vectors["packers"][kind], impl


def test_xdelta_escalation_matches_bit_range_rule(oracle, vectors):
    """SURVEY.md a-3: the plane count ends at max(nb0, planes needed by the post-xor words)."""
    for impl in impls():
        assert escalation_answers(oracle, impl) == vectors["escalation"], impl
    for bps, ch, ns, nb0, raw in escalation_frames():
        o = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, nb0)
        o.compress(raw)
        words, _ = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 4).transform(raw)
        need = nb0
        for nb in range(nb0, bps):
            top = words.astype(np.int64) >> (8 * nb - 1)
            lim = (1 << (8 * (bps - nb) + 1)) - 1
            ok = np.all(((top & lim) == 0) | ((top & lim) == lim))
            if ok:
                break
            need = nb + 1
        assert o.nb == need, (bps, ch, ns, nb0, o.nb, need)


def test_prefilter_restatement_equals_reference(oracle, vectors):
    for impl in impls():
        assert prefilter_answers(oracle, impl) == vectors["prefilter"], impl
