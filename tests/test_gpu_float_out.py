"""decompress_tensor / decompress_frames_tensor with dtype float32 / bfloat16 (rspt_gpu_decompress_batch_float /
rspt_gpu_decompress_frames_float): the int32 samples, dequantized per channel inside the inverse kernels.  Every
result is compared bit for bit with the conversion of the int32 output: numpy
((v.astype(int64) - zp).astype(float32) * scale), torch eager on the device for the full-scale batches, and bf16
as that float32 rounded to nearest even.  Needs a B200."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E_ARG, E_CAPACITY = -1, -3
OUT_F32, OUT_BF16 = 0, 1


@pytest.fixture(scope="module")
def R():
    import rspt_b200  # noqa: F401
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


def make_frames(oracle, rng, bps, ch, ns, nfr):
    """ECG-like (or a random walk for tiny shapes), full-range noise, then ECG again: native uint8 [nfr, fb]."""
    frames = []
    for i in range(nfr):
        if i % 3 == 1:
            lo, hi = -(1 << (8 * bps - 1)), 1 << (8 * bps - 1)
            x = rng.integers(lo, hi, (ns, ch)).astype(np.int32)
            frames.append(x.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].reshape(-1))
        elif bps >= 2 and ns >= 64:
            frames.append(oracle.synth_ecg(5 + i, 1, bps, ch, ns, amplitude=20000 if bps >= 3 else 3000)[0])
        else:
            amp = 1 << min(8 * bps - 2, 14)
            x = np.cumsum(rng.integers(-amp // 16 - 1, amp // 16 + 2, (ns, ch)), axis=0)
            x = np.clip(x, -(1 << (8 * bps - 1)), (1 << (8 * bps - 1)) - 1).astype(np.int32)
            frames.append(x.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].reshape(-1))
    return np.stack(frames)


def dev_u8(a):
    return torch.from_numpy(np.array(a, dtype=np.uint8, copy=True).reshape(-1)).cuda()


# (kind, bps, ch, ns, nb, frames, dct_exact): the shapes of test_gpu_i32_io.py
CASES = [
    ("xdelta_hzr", 3, 12, 8192, 3, 3, False), ("xdelta_hzr", 4, 12, 4096, 3, 3, False),
    ("xdelta_hzr", 2, 5, 1000, 2, 3, False), ("xdelta_hzr", 1, 3, 700, 1, 3, False),
    ("xdelta_hzr", 3, 7, 33, 3, 4, False), ("xdelta_hzr", 3, 2, 1, 3, 4, False), ("xdelta_hzr", 4, 3, 2, 3, 3, False),
    ("xdelta_hzr", 4, 2, 70001, 4, 2, False), ("xdelta_hzr", 2, 4, 1000, 2, 3, False), ("xdelta_hzr", 4, 1, 8192, 3, 3, False),
    ("xdelta_hzr", 3, 4, 6, 2, 3, False),
    ("hzr", 3, 12, 8192, 0, 3, False), ("hzr", 1, 2, 999, 0, 3, False), ("hzr", 2, 1, 140000, 0, 2, False),
    ("hzr", 4, 3, 5000, 0, 3, False), ("hzr", 2, 7, 33, 0, 3, False), ("hzr", 1, 4, 1024, 0, 3, False),
    ("hadamard", 4, 12, 4096, 0, 3, False), ("hadamard", 3, 12, 8192, 0, 3, False), ("hadamard", 3, 3, 16384, 0, 2, False),
    ("hadamard", 2, 2, 8, 0, 3, False), ("hadamard", 2, 3, 4096, 0, 3, False), ("hadamard", 1, 4, 4096, 0, 3, False),
    ("hadamard", 4, 1, 8192, 0, 2, False), ("hadamard", 2, 7, 64, 0, 3, False), ("hadamard", 1, 12, 1024, 0, 3, False),
    ("dct", 3, 12, 4096, 0, 3, False), ("dct", 2, 3, 256, 0, 3, False), ("dct", 4, 1, 8192, 0, 2, False),
    ("dct", 1, 4, 64, 0, 3, False), ("dct", 3, 2, 8, 0, 3, False), ("dct", 2, 7, 1024, 0, 3, False),
    ("dct", 3, 3, 1000, 0, 3, True), ("dct", 2, 4, 256, 0, 3, True), ("dct", 4, 2, 77, 0, 3, True),
]


def ref_f32(v, zp=None, scale=None):
    """numpy reference: float32 [n, ch, ns] of int32 v [n, ch, ns]."""
    v = np.asarray(v, np.int32).astype(np.int64)
    ch = v.shape[1]
    zp = np.zeros(ch, np.int64) if zp is None else np.asarray(zp, np.int32).astype(np.int64)
    sc = np.ones(ch, np.float32) if scale is None else np.asarray(scale, np.float32)
    with np.errstate(over="ignore"):
        return ((v - zp[None, :, None]).astype(np.float32) * sc[None, :, None]).astype(np.float32)


def bf16_bits(f32):
    """Bit pattern (int16) of float32 values rounded to nearest even to bfloat16 (torch's conversion)."""
    return torch.from_numpy(np.ascontiguousarray(f32)).to(torch.bfloat16).view(torch.int16).numpy()


def bits(t):
    """int32 view of a float32 tensor, int16 view of a bfloat16 tensor, on the host."""
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16).cpu().numpy()


def want_bits(ref, dtype):
    return ref.view(np.int32) if dtype == torch.float32 else bf16_bits(ref)


def offset_out(n, ch, ns, dtype):
    """An output tensor that starts one element (4 or 2 bytes) past a 16-byte boundary, and the sentinel before it."""
    buf = torch.full((n * ch * ns + 1,), 7.0, dtype=dtype, device="cuda")
    out = buf[1:].view(n, ch, ns)
    assert out.data_ptr() % 16 == buf.element_size()
    return buf, out


@pytest.mark.parametrize("kind,bps,ch,ns,nb,nfr,exact", CASES)
def test_float_out_every_kernel_row(R, oracle, kind, bps, ch, ns, nb, nfr, exact):
    rng = np.random.default_rng(ns * 31 + ch * 7 + bps)
    raws = make_frames(oracle, rng, bps, ch, ns, nfr)
    p = R.SignalPacker(kind, bps, ch, ns, nb or 3, max_batch_frames=nfr)
    if exact:
        p.set_dct_exact(True)
    b = p.compress_batch(dev_u8(raws))
    v = p.decompress_tensor(b)
    torch.cuda.synchronize()
    v = v.cpu().numpy()
    lim = 1 << (8 * bps - 1)
    zp = rng.integers(-lim, lim, ch).astype(np.int32)
    scale = (rng.standard_normal(ch) * 10.0 ** rng.integers(-6, 3, ch)).astype(np.float32)
    scale[0] = -abs(scale[0]) - 0.25
    for params in ({}, {"zero_point": zp.tolist(), "scale": scale.tolist()},
                   {"zero_point": torch.from_numpy(zp).cuda(), "scale": torch.from_numpy(scale).cuda()}):
        ref = ref_f32(v, zp, scale) if params else ref_f32(v)
        for dtype in (torch.float32, torch.bfloat16):
            want = want_bits(ref, dtype)
            for use_sc in (True, False):
                status = torch.full((nfr,), 7, dtype=torch.int32, device="cuda")
                got = p.decompress_tensor(b, status=status, use_sidecar=use_sc, dtype=dtype, **params)
                torch.cuda.synchronize()
                assert not status.cpu().numpy().any()
                assert got.dtype == dtype and tuple(got.shape) == (nfr, ch, ns)
                assert np.array_equal(bits(got), want), (kind, dtype, use_sc, bool(params))
            buf, out = offset_out(nfr, ch, ns, dtype)
            p.decompress_tensor(b, out=out, dtype=dtype, **params)
            torch.cuda.synchronize()
            assert np.array_equal(bits(out), want), (kind, dtype, "offset output")
            assert float(buf[0].item()) == 7.0


def test_float_out_ieee_edges(R):
    """One frame of full-range 4-byte samples: int -> float rounding above 2^24, v - zp beyond int32, subnormal
    results, overflow to inf in f32 and in bf16 only."""
    bps, ch, ns = 4, 8, 1024
    rng = np.random.default_rng(5)
    x = rng.integers(-(1 << 31), 1 << 31, (ns, ch), dtype=np.int64).astype(np.int32)
    x[:5, :] = [[2**31 - 1], [-2**31], [2**24 + 1], [-(2**24 + 3)], [1000]]
    p = R.SignalPacker.new_hzr(bps, ch, ns, max_batch_frames=1)
    b = p.compress_batch(dev_u8(x.astype("<i4").view(np.uint8)))
    v = p.decompress_tensor(b)
    torch.cuda.synchronize()
    v = v.cpu().numpy()
    assert np.array_equal(v[0], x.T)
    # channel: 0 exact, 1 zp = -2^31 (d up to 2^32 - 1), 2 subnormal, 3 f32 overflow, 4 bf16-only overflow,
    # 5 negative, 6 zp = 2^31 - 1, 7 plain
    zp = np.array([0, -2**31, 0, 0, 0, 12345, 2**31 - 1, -7], np.int32)
    scale = np.array([1.0, 1.0, 1e-42, 1e30, 1.584e29, -3.25e-3, 0.5, 2.0 ** -20], np.float32)
    ref = ref_f32(v, zp, scale)
    assert np.isinf(ref[0, 3]).any() and (np.abs(ref[0, 2]) < np.finfo(np.float32).tiny).any()
    assert not np.isinf(ref[0, 4]).any() and ((bf16_bits(ref[0, 4]).view(np.uint16) & 0x7FFF) == 0x7F80).any()
    for dtype in (torch.float32, torch.bfloat16):
        got = p.decompress_tensor(b, dtype=dtype, zero_point=zp.tolist(), scale=scale.tolist())
        torch.cuda.synchronize()
        assert np.array_equal(bits(got), want_bits(ref, dtype)), dtype
        # torch eager on the device gives the same bits
        vt = torch.from_numpy(v).cuda()
        te = (vt.long() - torch.from_numpy(zp).cuda()[None, :, None]).float() * torch.from_numpy(scale).cuda()[None, :, None]
        assert torch.equal(got.view(torch.int32 if dtype == torch.float32 else torch.int16),
                           te.to(dtype).view(torch.int32 if dtype == torch.float32 else torch.int16))


@pytest.mark.parametrize("use_sidecar", [True, False])
def test_float_out_gather(R, oracle, use_sidecar):
    """A store appended past max_batch_frames; ids shuffled, repeated and out of range; status equals that of the
    int32 gather and every ok slot is the conversion of its int32 output."""
    bps, ch, ns, mb = 3, 12, 1024, 4
    rng = np.random.default_rng(17)
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=mb)
    store = p.new_store(2)
    for k in range(3):
        p.append_batch(store, dev_u8(make_frames(oracle, rng, bps, ch, ns, mb)))
    assert store.n_frames == 3 * mb > p.max_batch
    zp = rng.integers(-1000, 1000, ch).astype(np.int32)
    scale = rng.uniform(-2, 2, ch).astype(np.float32)
    for ids in ([7, 0, 11, 7], [3, -1, 12, 3], [11, 10, 2, 2]):
        st_i = torch.full((mb,), 7, dtype=torch.int32, device="cuda")
        v = p.decompress_frames_tensor(store, ids, status=st_i, use_sidecar=use_sidecar)
        torch.cuda.synchronize()
        v, st_i = v.cpu().numpy(), st_i.cpu().numpy()
        ok = st_i == 0
        ref = ref_f32(v, zp, scale)
        for dtype in (torch.float32, torch.bfloat16):
            st_f = torch.full((mb,), 7, dtype=torch.int32, device="cuda")
            got = p.decompress_frames_tensor(store, torch.tensor(ids, dtype=torch.int64, device="cuda"), status=st_f,
                                             use_sidecar=use_sidecar, dtype=dtype, zero_point=zp.tolist(),
                                             scale=torch.from_numpy(scale).cuda())
            torch.cuda.synchronize()
            assert np.array_equal(st_f.cpu().numpy(), st_i), (ids, dtype)
            assert np.array_equal(bits(got)[ok], want_bits(ref, dtype)[ok]), (ids, dtype)
        assert ok.sum() == sum(0 <= i < store.n_frames for i in ids)


def test_float_out_refusals(R):
    bps, ch, ns, n = 3, 4, 256, 2
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    x = torch.zeros((n, ch, ns), dtype=torch.int32, device="cuda")
    b = p.compress_tensor(x)
    L, h = p.L, p.h
    dst = torch.zeros((n + 1, ch, ns), dtype=torch.float32, device="cuda")
    a = (b.stream.data_ptr(), b.offsets.data_ptr())
    assert L.rspt_gpu_decompress_batch_float(h, *a, n, None, None, OUT_F32, None, None, dst.data_ptr(), None) == 0
    assert L.rspt_gpu_decompress_batch_float(h, *a, n, None, None, 2, None, None, dst.data_ptr(), None) == E_ARG
    assert L.rspt_gpu_decompress_batch_float(h, *a, n, None, None, -1, None, None, dst.data_ptr(), None) == E_ARG
    assert L.rspt_gpu_decompress_batch_float(h, *a, n, None, None, OUT_F32, None, None, None, None) == E_ARG
    assert L.rspt_gpu_decompress_batch_float(h, *a, n, None, None, OUT_F32, None, None, dst.data_ptr() + 2, None) == E_ARG
    assert L.rspt_gpu_decompress_batch_float(h, *a, n, None, None, OUT_BF16, None, None, dst.data_ptr() + 1, None) == E_ARG
    assert L.rspt_gpu_decompress_batch_float(h, *a, n, None, None, OUT_BF16, None, None, dst.data_ptr() + 2, None) == 0
    assert L.rspt_gpu_decompress_batch_float(h, *a, n + 1, None, None, OUT_F32, None, None, dst.data_ptr(), None) == E_CAPACITY
    ids = torch.tensor([0, 1, 1], dtype=torch.int64, device="cuda")
    fa = (b.stream.data_ptr(), b.offsets.data_ptr(), n, None, None, ids.data_ptr())
    assert L.rspt_gpu_decompress_frames_float(h, *fa, n, OUT_BF16, None, None, dst.data_ptr(), None) == 0
    assert L.rspt_gpu_decompress_frames_float(h, *fa, n, 5, None, None, dst.data_ptr(), None) == E_ARG
    assert L.rspt_gpu_decompress_frames_float(h, *fa, n, OUT_F32, None, None, None, None) == E_ARG
    assert L.rspt_gpu_decompress_frames_float(h, *fa, n, OUT_F32, None, None, dst.data_ptr() + 2, None) == E_ARG
    assert L.rspt_gpu_decompress_frames_float(h, *fa, n + 1, OUT_F32, None, None, dst.data_ptr(), None) == E_CAPACITY
    torch.cuda.synchronize()
    for kw in ({"zero_point": [0] * ch}, {"scale": [1.0] * ch}):
        with pytest.raises(ValueError):
            p.decompress_tensor(b, **kw)
        with pytest.raises(ValueError):
            p.decompress_frames_tensor(b, [0, 1], **kw)
    for bad in (torch.empty((n, ch, ns), dtype=torch.bfloat16, device="cuda"), torch.empty((n, ch, ns), dtype=torch.int32, device="cuda"),
                torch.empty((n + 1, ch, ns), dtype=torch.float32, device="cuda"), torch.empty((n, ns, ch), dtype=torch.float32, device="cuda"),
                torch.empty((n, ns, ch), dtype=torch.float32, device="cuda").transpose(1, 2), torch.empty((n, ch, ns), dtype=torch.float32)):
        with pytest.raises(ValueError):
            p.decompress_tensor(b, out=bad, dtype=torch.float32)
    for kw in ({"dtype": torch.float16}, {"dtype": torch.float32, "zero_point": [0] * (ch + 1)},
               {"dtype": torch.float32, "scale": torch.ones(ch, dtype=torch.float64, device="cuda")},
               {"dtype": torch.bfloat16, "zero_point": torch.zeros(ch, dtype=torch.int64, device="cuda")}):
        with pytest.raises(ValueError):
            p.decompress_tensor(b, **kw)


def test_float_out_state(R, oracle):
    """Counters and the INVERSE timer count float calls; an xdelta_hzr handle's plane count and a following int32
    decode are unchanged by float calls in between."""
    bps, ch, ns, n = 4, 4, 1024, 3
    rng = np.random.default_rng(23)
    raws = make_frames(oracle, rng, bps, ch, ns, n)
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 1, max_batch_frames=n)
    b = p.compress_batch(dev_u8(raws))
    v0 = p.decompress_tensor(b)
    torch.cuda.synchronize()
    nb0, c0 = p.nb, p.counters()["frames_decompressed"]
    p.set_stage_timing(True)
    p.stage_times(reset=True)
    p.decompress_tensor(b, dtype=torch.float32, scale=[0.5] * ch)
    p.decompress_frames_tensor(b, [2, 0], dtype=torch.bfloat16, zero_point=[1] * ch)
    torch.cuda.synchronize()
    st = p.stage_times(reset=True)
    p.set_stage_timing(False)
    assert st["inverse"][1] == 2 and st["inverse"][0] > 0
    assert p.counters()["frames_decompressed"] == c0 + n + 2
    assert p.nb == nb0
    v1 = p.decompress_tensor(b)
    torch.cuda.synchronize()
    assert torch.equal(v0, v1)


@pytest.mark.parametrize("kind", ["xdelta_hzr", "hadamard", "dct"])
def test_float_out_full_scale(R, kind):
    """4096 frames of synth_ecg (shape A for xdelta_hzr, B for hadamard and dct): the fused outputs equal torch eager
    on the device applied to decompress_tensor."""
    bps, ch, ns = (3, 12, 8192) if kind == "xdelta_hzr" else (4, 12, 4096)
    n = 4096
    p = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=n)
    b = p.compress_batch(R.synth_ecg(0, n, bps, ch, ns), sidecar=True)
    gen = torch.Generator().manual_seed(3)
    zp = torch.randint(-20000, 20000, (ch,), dtype=torch.int32, generator=gen).cuda()
    scale = (torch.randn(ch, generator=gen) * 1e-3).cuda()
    v = p.decompress_tensor(b)
    want = (v.long() - zp[None, :, None]).float() * scale[None, :, None]
    del v
    got = p.decompress_tensor(b, dtype=torch.float32, zero_point=zp, scale=scale)
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    del got
    got = p.decompress_tensor(b, dtype=torch.bfloat16, zero_point=zp, scale=scale)
    assert torch.equal(got.view(torch.int16), want.to(torch.bfloat16).view(torch.int16))


# ---- which kernel a float call launches ------------------------------------------------------------------------
# Bit-exact output does not show which kernel produced it: a 16-byte aligned xdelta_hzr call that fell back to the
# generic sample kernel would still pass every test above.  Each row: (entry, kind, bps, ch, ns, dtype, dct_exact,
# element offset of the output, the sample-stage kernels the call must launch in order).
KERNEL_ROWS = [
    ("batch", "xdelta_hzr", 3, 12, 8192, "float32", False, 0, ["k_dq_planes_to_samples_fast<3,true,float>"]),
    ("batch", "hzr", 3, 12, 8192, "bfloat16", False, 0, ["k_dq_planes_to_samples_fast<3,false,__nv_bfloat16>"]),
    ("batch", "xdelta_hzr", 3, 12, 8192, "float32", False, 1, ["k_dq_planes_to_samples<3,true,float>"]),
    ("batch", "hzr", 3, 12, 8192, "bfloat16", False, 1, ["k_dq_planes_to_samples<3,false,__nv_bfloat16>"]),
    ("batch", "hzr", 2, 5, 1000, "bfloat16", False, 0, ["k_dq_planes_to_samples<2,false,__nv_bfloat16>"]),
    ("batch", "hadamard", 4, 12, 4096, "float32", False, 0, ["k_dq_fwht_fast_inv<12,float>"]),
    ("batch", "hadamard", 3, 12, 8192, "bfloat16", False, 1, ["k_dq_fwht_fast_inv<13,__nv_bfloat16>"]),
    ("batch", "hadamard", 3, 3, 16384, "float32", False, 0, ["k_dq_fwht_inv<float>"]),
    ("batch", "dct", 3, 12, 4096, "bfloat16", False, 0,
     ["k_planes_to_samples_fast<4,true,true>", "k_words_to_float<3,__nv_bfloat16>"]),
    ("batch", "dct", 2, 3, 256, "float32", True, 1, ["k_planes_to_samples<4,true,false>", "k_words_to_float<2,float>"]),
    ("frames", "xdelta_hzr", 3, 12, 8192, "bfloat16", False, 0, ["k_dq_planes_to_samples_fast<3,true,__nv_bfloat16>"]),
]
SAMPLE_KERNEL = re.compile(r"^k_(dq_|words_to_float|planes_to_samples|fwht_|words_sext|words_to_raw)")


def kernel_name(demangled):
    """'void rspt::k_dq_fwht_inv<float>(...)' or '... k_x<(int)3, (bool)1, float>(...)' -> 'k_x<3,true,float>'."""
    s = demangled.replace("(bool)0", "false").replace("(bool)1", "true")
    s = re.sub(r"\((?:unsigned )?int\)", "", s)
    m = re.search(r"\bk_\w+(?:<[^>]*>)?", s)
    return m.group(0).replace(" ", "") if m else None


def trace_kernel_rows(out_path):
    """Child process: each row's call under torch.profiler between two marker kernels; writes the sample-stage
    kernels of every call window, in launch order."""
    sys.path.insert(0, ROOT)
    from rspt_b200 import packer as R
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.set_device(0)
    marker = torch.zeros(1, dtype=torch.int64, device="cuda")
    rng = np.random.default_rng(13)
    nfr = 2
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        marker.bitwise_not_()
        marker.neg_()
        torch.cuda.synchronize()
        for entry, kind, bps, ch, ns, dt, exact, off, _ in KERNEL_ROWS:
            dtype = getattr(torch, dt)
            p = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=nfr)
            if exact:
                p.set_dct_exact(True)
            b = p.compress_batch(dev_u8(rng.integers(0, 256, nfr * bps * ch * ns, dtype=np.uint8)))
            buf = torch.empty(nfr * ch * ns + off, dtype=dtype, device="cuda")
            out = buf[off:].view(nfr, ch, ns)
            kw = dict(out=out, dtype=dtype, zero_point=[1] * ch, scale=[0.5] * ch)
            torch.cuda.synchronize()
            marker.bitwise_not_()
            if entry == "batch":
                p.decompress_tensor(b, **kw)
            else:
                p.decompress_frames_tensor(b, [1, 0], **kw)
            torch.cuda.synchronize()
            marker.neg_()
            p.close()
        torch.cuda.synchronize()
    path = out_path + ".trace.json"
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    os.remove(path)
    kernels = [e["name"] for e in sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])]
    opening, closing = kernels[:2]
    windows, cur = [], None
    for name in kernels[2:]:
        if name == opening:
            cur = []
        elif name == closing:
            windows.append(cur)
            cur = None
        elif cur is not None:
            k = kernel_name(name)
            if k and SAMPLE_KERNEL.match(k):
                cur.append(k)
    with open(out_path, "w") as f:
        json.dump(windows, f)


@pytest.mark.timeout(600)
def test_float_out_launches_its_kernels(tmp_path):
    out = str(tmp_path / "kernels.json")
    p = subprocess.run([sys.executable, os.path.abspath(__file__), out], capture_output=True, text=True, timeout=500)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    with open(out) as f:
        got = json.load(f)
    assert len(got) == len(KERNEL_ROWS), f"{len(got)} call windows in the trace for {len(KERNEL_ROWS)} rows"
    bad = [f"{r[:8]}: launched {g}, expected {r[8]}" for r, g in zip(KERNEL_ROWS, got) if g != r[8]]
    assert not bad, "\n".join(bad)


if __name__ == "__main__":
    trace_kernel_rows(sys.argv[1])
