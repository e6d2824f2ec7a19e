"""Every path of the hzr entropy decoder (k_hzr_decode, k_hzr_build_index) held to the oracle by a table of crafted
blocks.  The decoder picks per block a decode class by payload length (1: <= 4096 B, 2: <= 16384 B, 0: longer), a
token loop (12-bit single-symbol table with up to four chained literals; 11-bit pair table with one chained look-up
for xdelta_hzr / hzr; the pair table without chaining for hadamard / dct) and, per thread, a start from the decode
index (the encoder's, the one k_hzr_build_index rebuilds, or a gather call's own).  The rows reach the long-code
chains, every run class at both ends of its extra bits, the class and pair-table edges, the smallest and the largest
trees, and payloads at every address mod 16 up to the last byte of the decoder's shared-memory staging.

Two packers give exact control over the block: `hzr` 1 B x 1 ch x n, whose low byte plane is the input; and
`hadamard` 4 B x 1 ch x n (n a power of two) fed x = FWHT(c) for coefficients 0 <= c[i] < 256 with c[0] = 0, whose
transform gives back c: plane 0 is then c and planes 1-2 are FILL blocks.

test_table_covers_every_decode_path classifies every HUFF block of the table on the host and needs no GPU: it keeps a
row from drifting off its path after a change to the encoder or the table.  The other tests need a B200."""
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")

# k_hzr_decode / k_hzr_build_index (hzr_decode.cuh, common.cuh) and the host's launch (rspt_gpu.cu)
LUT_BITS, PAIR_BITS, PAIR_MAX_BITS = 12, 11, 4
SMALL, MEDIUM, BLOCK = 4096, 16384, 65536
IDX_MIN_BITS, MAX_SEGS, POS_SHIFT = 512, 512, 12
EXTRA = {256: 0, 257: 2, 258: 4, 259: 8, 260: 14}
RUN_BASE = {256: 2, 257: 3, 258: 7, 259: 23, 260: 279}
# both ends of every run class's extra bits; 16663 is a full 260 token and a zero byte
RUN_LENGTHS = (2, 3, 6, 7, 22, 23, 278, 279, 16662, 16663)
LOOPS = ("single", "pairs_chain", "pairs")
GUARD = 64
NB = {"hzr": 4, "hadamard": 3}


def idx_geom(plen):
    """(interval bits, intervals) of a HUFF payload of plen bytes (common.cuh idx_geom)"""
    total = 8 * plen
    bits = max(IDX_MIN_BITS, (total + MAX_SEGS - 1) // MAX_SEGS)
    return bits, (total + bits - 1) // bits


def decode_class(plen):
    return 1 if plen <= SMALL else 2 if plen <= MEDIUM else 0


def loop_of(kind, plen, n):
    """the token loop k_hzr_decode runs for a HUFF block (use_pairs, chain_pairs)"""
    if not (plen * 16 >= n and plen * 8 <= PAIR_MAX_BITS * n):
        return "single"
    return "pairs_chain" if kind == "hzr" else "pairs"


# ---- block content ------------------------------------------------------------------------------------------
def compose(rng, n, runs, lits=None, vals=None, p=None, first_zero=False):
    """n bytes: zero runs of the lengths in `runs` (each maximal: nonzero literals on both sides, or the block start
    for the first one when first_zero), the other bytes nonzero literals -- the array `lits` shuffled, or drawn from
    `vals` with probabilities `p`.  A run of 1 is the symbol-0 token."""
    runs = list(runs)
    nl = n - sum(runs)
    assert nl >= len(runs) + 1, "not enough literals to separate the runs"
    if lits is None:
        lits = rng.choice(np.asarray(vals, np.uint8), nl, p=p)
    lits = np.asarray(lits, np.uint8).copy()
    assert lits.size == nl and lits.all()
    rng.shuffle(lits)
    rng.shuffle(runs)
    inner = list(runs[1:]) if first_zero else runs
    gaps = np.sort(rng.choice(np.arange(1, nl), len(inner), replace=False))
    parts, prev = ([np.zeros(runs[0], np.uint8)] if first_zero else []), 0
    for g, z in zip(gaps, inner):
        parts += [lits[prev:g], np.zeros(z, np.uint8)]
        prev = g
    parts.append(lits[prev:])
    out = np.concatenate(parts)
    assert out.size == n
    return out


def geo(k, r, lo=1):
    """literal values lo .. lo + k - 1 with geometric probabilities (ratio r)"""
    w = r ** np.arange(k)
    return np.arange(lo, lo + k), w / w.sum()


def deep_lits(heavy, tail, n_lits, rng):
    """literal multiset: `heavy` {value: count} (the first one takes up the rest of n_lits) and a Fibonacci tail of
    rare values (the deepest codes of the tree)"""
    out = [np.full(c, v, np.uint8) for v, c in list(heavy.items())[1:]]
    out += [np.full(c, v, np.uint8) for v, c in tail.items()]
    rest = n_lits - sum(x.size for x in out)
    assert rest > 0
    out.append(np.full(rest, list(heavy)[0], np.uint8))
    return np.concatenate(out)


def fib(k):
    f = [1, 1]
    while len(f) < k:
        f.append(f[-1] + f[-2])
    return f[:k]


def mixed_runs(rng, count, hi=40):
    return list(rng.integers(1, hi, count))


# ---- the oracle's plan and exact payload lengths --------------------------------------------------------------
def plan_len(O, block):
    mode, plen = O.hzr_block_plan(block)
    return plen if mode == 1 else (10 ** 9 if mode == 0 else -1)


def tune(O, make, lo, hi, target):
    """make(m) for m in [lo, hi] gives blocks whose HUFF payload grows with m: the block whose payload is exactly
    `target` bytes (a byte next to the edge is varied when one step of m jumps over it)"""
    while lo < hi:
        mid = (lo + hi) // 2
        if plan_len(O, make(mid)) >= target:
            hi = mid
        else:
            lo = mid + 1
    for m in range(max(0, lo - 2), lo + 3):
        b = make(m)
        if plan_len(O, b) == target:
            return b
        for i in range(max(0, m - 2), min(b.size, m + 3)):
            if b[i] == 0:
                continue
            for v in range(1, 256):
                c = b.copy()
                c[i] = v
                if plan_len(O, c) == target:
                    return c
    raise AssertionError(f"no block with a {target}-byte payload")


def blend(a, b):
    """make(m): a with its first m nonzero bytes taken from b (the zero runs stay where they are)"""
    nz = np.flatnonzero(a)

    def make(m):
        c = a.copy()
        c[nz[:m]] = b[nz[:m]]
        return c
    return make, nz.size


# ---- the rows --------------------------------------------------------------------------------------------------
class Row:
    """kind, plane length n, the intended plane-0 block, and whether the batch repeats it at every address mod 16"""

    def __init__(self, name, kind, block, sweep=False, stage=None, ch=1):
        self.name, self.kind, self.block, self.sweep, self.stage = name, kind, np.asarray(block, np.uint8), sweep, stage
        self.n, self.ch = self.block.size, ch
        self.ns = self.n // ch

    def oracle(self):
        from oracle import oracle as O
        return O.OraclePacker(self.kind, 1 if self.kind == "hzr" else 4, self.ch, self.ns, NB[self.kind])

    def frame(self, c=None):
        """the packer input whose plane 0 is `c` (default: the row's block)"""
        c = self.block if c is None else c
        if self.kind == "hzr":
            return c.copy()
        # plane 0 holds the channels one after the other; the samples are interleaved
        from oracle import oracle as O
        x = np.empty((self.ch, self.ns), np.int32)
        for i in range(self.ch):
            cc = np.ascontiguousarray(c[i * self.ns:(i + 1) * self.ns], np.int32)
            O.oracle_lib().oracle_fwht(self.ns, cc.ctypes.data, x[i].ctypes.data)
        return np.ascontiguousarray(x.T).astype("<i4").view(np.uint8).reshape(-1).copy()


ROW_NAMES = []
_BUILDERS = {}


def row(name):
    def deco(fn):
        ROW_NAMES.append(name)
        _BUILDERS[name] = fn
        return fn
    return deco


def _rng(name):
    return np.random.default_rng(sum(map(ord, name)) * 7919)


# single-symbol table + chain (hzr, more than 4 payload bits per byte)
@row("hzr_single_c1_261_leaves")
def _(O, rng):
    # every one of the 261 symbols: 2870 tree bits over six 512-bit intervals of a class-1 payload
    runs = [1] * 3 + [2] * 3 + [3, 6, 5] + [7, 22, 9] + [23, 278, 40] + [279, 300, 400]
    lits = np.repeat(np.arange(1, 256), 4).astype(np.uint8)
    return Row("hzr_single_c1_261_leaves", "hzr", compose(rng, lits.size + sum(runs), runs, lits=lits))


@row("hzr_single_c2")
def _(O, rng):
    v, p = geo(200, 0.995)
    return Row("hzr_single_c2", "hzr", compose(rng, 17000, [2, 3, 6, 7, 22, 23, 278, 279] + mixed_runs(rng, 300), vals=v, p=p))


@row("hzr_single_c0_long_runs")
def _(O, rng):
    # two blocks: a run of 16662 in the first, of 16663 in the second, the short run lengths in both
    v, p = geo(255, 0.999)
    short = [2, 3, 6, 7, 22, 23, 278, 279]
    b0 = compose(rng, BLOCK, [16662] + short + mixed_runs(rng, 400), vals=v, p=p)
    b1 = compose(rng, BLOCK, [16663] + short + mixed_runs(rng, 400), vals=v, p=p)
    return Row("hzr_single_c0_long_runs", "hzr", np.concatenate([b0, b1]))


@row("hzr_single_deep")
def _(O, rng):
    # 150 equal literals and a Fibonacci tail whose rarest members are the run symbols: codes of up to ~17 bits,
    # the long ones on one spine (one 12-bit prefix), every run class among them
    tail_runs = {260: [300], 259: [24], 258: [8], 257: [3], 256: [2]}
    tail_lits = dict(zip(range(200, 206), fib(11)[5:]))
    heavy = {v: 200 for v in range(1, 151)}
    runs = [z for zs in tail_runs.values() for z in zs] + [1] * 8
    n_lits = sum(heavy.values()) + sum(tail_lits.values())
    lits = deep_lits(heavy, tail_lits, n_lits, rng)
    return Row("hzr_single_deep", "hzr", compose(rng, n_lits + sum(runs), runs, lits=lits))


@row("hzr_fibonacci_22")
def _(O, rng):
    # Fibonacci counts on 22 literals: the deepest tree a block allows, codes of up to 21 bits
    lits = np.repeat(np.arange(1, 23), fib(22)).astype(np.uint8)
    return Row("hzr_fibonacci_22", "hzr", compose(rng, lits.size, [], lits=lits))


# pair table + chain (hzr, 1/2 .. 4 payload bits per byte)
@row("hzr_pairs_c1")
def _(O, rng):
    v, p = geo(12, 0.6)
    return Row("hzr_pairs_c1", "hzr", compose(rng, 16384, mixed_runs(rng, 1500, 12), vals=v, p=p))


@row("hzr_pairs_c2_all_runs")
def _(O, rng):
    v, p = geo(16, 0.75)
    return Row("hzr_pairs_c2_all_runs", "hzr", compose(rng, BLOCK, list(RUN_LENGTHS) + mixed_runs(rng, 1500, 12), vals=v, p=p))


@row("hzr_pairs_c0")
def _(O, rng):
    v, p = geo(40, 0.88)
    return Row("hzr_pairs_c0", "hzr", compose(rng, BLOCK, mixed_runs(rng, 3000, 24), vals=v, p=p))


@row("hzr_pairs_deep")
def _(O, rng):
    tail_runs = {260: [280], 259: [30], 258: [10], 257: [4], 256: [2]}
    tail_lits = dict(zip(range(200, 208), fib(13)[5:]))
    heavy = {1: 0, 2: 9000, **{v: 300 for v in range(3, 21)}}
    runs = [z for zs in tail_runs.values() for z in zs] + [1] * 8
    n = 40000
    lits = deep_lits(heavy, tail_lits, n - sum(runs), rng)
    return Row("hzr_pairs_deep", "hzr", compose(rng, n, runs, lits=lits))


# pair table without chaining (hadamard coefficient planes)
@row("had_pairs_c1")
def _(O, rng):
    v, p = geo(12, 0.6)
    return Row("had_pairs_c1", "hadamard", compose(rng, 16384, [3] + mixed_runs(rng, 1500, 12), vals=v, p=p, first_zero=True))


# (2 channels of 32768 samples: one 65536-byte block, each channel's coefficients from c[0] = 0)
@row("had_pairs_c2_all_runs")
def _(O, rng):
    v, p = geo(16, 0.75)
    h0 = compose(rng, BLOCK // 2, [16662, 2, 3, 6, 7, 22] + mixed_runs(rng, 700, 12), vals=v, p=p, first_zero=True)
    h1 = compose(rng, BLOCK // 2, [16663, 23, 278, 279] + mixed_runs(rng, 700, 12), vals=v, p=p, first_zero=True)
    return Row("had_pairs_c2_all_runs", "hadamard", np.concatenate([h0, h1]), ch=2)


@row("had_pairs_c0")
def _(O, rng):
    v, p = geo(40, 0.88, lo=100)
    h = [compose(rng, BLOCK // 2, [1] + mixed_runs(rng, 1500, 24), vals=v, p=p, first_zero=True) for _ in range(2)]
    return Row("had_pairs_c0", "hadamard", np.concatenate(h), ch=2)


@row("had_pairs_deep")
def _(O, rng):
    tail_runs = {260: [280], 259: [30], 258: [10], 257: [4], 256: [2]}
    tail_lits = dict(zip(range(200, 208), fib(13)[5:]))
    heavy = {1: 0, 2: 6000, **{v: 150 for v in range(3, 21)}}
    runs = [1] + [z for zs in tail_runs.values() for z in zs] + [1] * 8
    n = BLOCK // 2
    lits = deep_lits(heavy, tail_lits, n - sum(runs), rng)
    return Row("had_pairs_deep", "hadamard", compose(rng, n, runs, lits=lits, first_zero=True))


# class and pair-table edges: exact payload lengths, the class maxima at every address mod 16
def _edge(O, rng, name, n, target, sweep=False, lo_geo=(6, 0.5), runs=200, run_hi=12):
    v, p = geo(*lo_geo)
    a = compose(rng, n, mixed_runs(rng, runs, run_hi), vals=v, p=p)
    b = a.copy()
    nz = a != 0
    b[nz] = rng.integers(1, 256, int(nz.sum()))
    make, m = blend(a, b)
    return Row(name, "hzr", tune(O, make, 0, m, target), sweep=sweep)


@row("hzr_c1_max_pair_edge")          # plen 4096 = n / 2: the largest class-1 payload, last pair-table length
def _(O, rng):
    return _edge(O, rng, "hzr_c1_max_pair_edge", 8192, 4096, sweep=True)


@row("hzr_c2_min_single")             # plen 4097 = n / 2 + 1: class 2, the single-symbol table
def _(O, rng):
    return _edge(O, rng, "hzr_c2_min_single", 8192, 4097)


@row("hzr_c2_max")                    # plen 16384: the largest class-2 payload
def _(O, rng):
    return _edge(O, rng, "hzr_c2_max", 40000, 16384, sweep=True)


@row("hzr_c0_min")                    # plen 16385
def _(O, rng):
    return _edge(O, rng, "hzr_c0_min", 40000, 16385)


@row("hzr_pairs_min_edge")            # plen * 16 == n: the pair table
def _(O, rng):
    return _edge(O, rng, "hzr_pairs_min_edge", 16384, 1024, lo_geo=(3, 0.1), runs=250, run_hi=110)


@row("hzr_pairs_min_below")           # plen * 16 == n - 1: the single-symbol table
def _(O, rng):
    return _edge(O, rng, "hzr_pairs_min_below", 16385, 1024, lo_geo=(3, 0.1), runs=250, run_hi=110)


@row("hzr_c0_max_65535")              # the largest HUFF payload of a 65536-byte block: staging full at lead 15
def _(O, rng):
    return _edge(O, rng, "hzr_c0_max_65535", BLOCK, BLOCK - 1, sweep=True, lo_geo=(255, 0.99), runs=50)


@row("hzr_c0_max_n")                  # plen == n == the shape's largest block
def _(O, rng):
    return _edge(O, rng, "hzr_c0_max_n", 30001, 30001, sweep=True, lo_geo=(255, 0.99), runs=50)


@row("hzr_c1_max_n")                  # a class-1 shape whose block is its whole payload
def _(O, rng):
    return _edge(O, rng, "hzr_c1_max_n", 3001, 3001, sweep=True, lo_geo=(255, 0.97), runs=10)


@row("hzr_c2_max_n")                  # a class-2 shape (no block over 16384 bytes) whose block is its whole payload
def _(O, rng):
    return _edge(O, rng, "hzr_c2_max_n", 10001, 10001, sweep=True, lo_geo=(255, 0.97), runs=30)


# trees, ragged and tiny planes, sparse blocks
@row("hzr_tiny_two_leaves")           # 3 bytes, a two-leaf tree (1-bit codes), payload == n
def _(O, rng):
    # the smallest tree a HUFF block has: a block of one token class is a FILL block, so the encoder never writes
    # the lone-leaf tree (1-bit code) that the decoder also accepts
    return Row("hzr_tiny_two_leaves", "hzr", np.array([5, 0, 5], np.uint8), sweep=True)


@row("hzr_ragged_13")
def _(O, rng):
    return Row("hzr_ragged_13", "hzr", np.array([0, 0, 0, 9, 9, 9, 9, 1, 9, 9, 0, 0, 9], np.uint8))


@row("hzr_ragged_70001")              # blocks of 65536 and 4465 bytes
def _(O, rng):
    v, p = geo(30, 0.85)
    return Row("hzr_ragged_70001", "hzr", compose(rng, 70001, mixed_runs(rng, 6000, 20), vals=v, p=p))


@row("hzr_sparse")
def _(O, rng):
    b = np.zeros(BLOCK, np.uint8)
    at = rng.choice(BLOCK, 700, replace=False)
    b[at] = rng.integers(1, 256, at.size)
    return Row("hzr_sparse", "hzr", b)


@row("hzr_sparse_handed_back")        # the sparse encoder hands its list to the dense encoder past 300 payload bytes
def _(O, rng):
    b = np.zeros(BLOCK, np.uint8)
    at = rng.choice(BLOCK, 700, replace=False)
    b[at] = rng.integers(1, 256, at.size)
    return Row("hzr_sparse_handed_back", "hzr", b, stage=300)


@functools.lru_cache(maxsize=None)
def build_row(name):
    from oracle import oracle as O
    r = _BUILDERS[name](O, _rng(name))
    assert r.name == name
    return r


# ---- host-side stream walk -----------------------------------------------------------------------------------
def le16(b, i):
    return int(b[i]) | int(b[i + 1]) << 8


def le32(b, i):
    return int.from_bytes(bytes(b[i:i + 4]), "little")


def parse_frame(fr, kind, n, ch=1):
    """the blocks of one frame: (plane, block, payload offset in the frame, payload length, mode)"""
    nblk = (n + BLOCK - 1) // BLOCK
    pos = 1 + (3 * ch if kind == "hadamard" else 0)
    out = []
    for k in range(NB[kind]):
        clen = le32(fr, pos)
        assert le32(fr, pos + 4) == n
        q = pos + 8
        for b in range(nblk):
            plen, mode = le16(fr, q) + 1, int(fr[q + 6])
            out.append((k, b, q + 7, plen, mode))
            q += 7 + plen
        assert q == pos + 4 + clen
        pos += 4 + clen
    assert pos == len(fr)
    return out


class Walk:
    """The tokens of one HUFF block, walked on the host from its payload: the tree (pre-order, 0 = branch,
    1 + 9-bit symbol = leaf, LSB-first code words), then tokens up to n output bytes.  starts / opos / syms / lens /
    ends per token; `pseudo`: the boundaries of what the zero padding behind the last token decodes to, up to the
    payload's last bit (k_hzr_build_index walks through them)."""

    def __init__(self, pay, n):
        self.plen, self.n = len(pay), n
        self.buf = bytes(pay) + bytes(16)
        self.codes = {}
        self.p = 0
        self._tree(0, 0)
        self.tree_nbits = self.p
        lut = [None] * (1 << LUT_BITS)
        longs = {}
        for s, (c, l) in self.codes.items():
            if l <= LUT_BITS:
                for i in range(1 << (LUT_BITS - l)):
                    lut[(i << l) | c] = (s, l)
            else:
                longs.setdefault(l, {})[c] = s
        self.lut, self.longs = lut, sorted(longs.items())
        starts, opos, syms, lens, ends = [], [], [], [], []
        p, o = self.tree_nbits, 0
        while o < n:
            s, l, z, e = self._token(p)
            assert e <= 8 * self.plen, "token past the payload"
            starts.append(p); opos.append(o); syms.append(s); lens.append(l); ends.append(e)
            o += z
            p = e
        assert o == n
        self.end_bits = p
        self.pseudo = []
        while p < 8 * self.plen:
            self.pseudo.append(p)
            p = self._token(p)[3]
        self.starts, self.opos, self.syms, self.lens, self.ends = map(np.array, (starts, opos, syms, lens, ends))

    def bits(self, p, k):
        return (int.from_bytes(self.buf[p >> 3:(p >> 3) + 8], "little") >> (p & 7)) & ((1 << k) - 1)

    def _tree(self, depth, code):
        leaf = self.bits(self.p, 1)
        self.p += 1
        if leaf:
            self.codes[self.bits(self.p, 9)] = (code, max(depth, 1))
            self.p += 9
            return
        self._tree(depth + 1, code)
        self._tree(depth + 1, code | 1 << depth)

    def _token(self, p):
        """(symbol, code length, output bytes, end bit) of the token at bit p"""
        w = self.bits(p, 56)
        e = self.lut[w & ((1 << LUT_BITS) - 1)]
        if e is None:
            e = next((s, l) for l, t in self.longs for c, s in t.items() if (w & ((1 << l) - 1)) == c)
        s, l = e
        if s < 256:
            return s, l, 1, p + l
        eb = EXTRA[s]
        return s, l, RUN_BASE[s] + ((w >> l) & ((1 << eb) - 1)), p + l + eb

    def content(self):
        out = np.zeros(self.n, np.uint8)
        lit = self.syms < 256
        out[self.opos[lit]] = self.syms[lit]
        return out


_COMP = {}


def oracle_frame(r, fr):
    key = (r.name, fr.tobytes())
    if key not in _COMP:
        _COMP[key] = r.oracle().compress(fr)
    return _COMP[key]


_WALKS = {}


def walk_of(pay, n):
    key = (bytes(pay), n)
    if key not in _WALKS:
        _WALKS[key] = Walk(pay, n)
    return _WALKS[key]


def batch_frames(r):
    """the frames of the row's batch: its frame once, or (sweep) once at every payload address mod 16 of plane 0's
    first block, with fillers of other compressed lengths in front"""
    main = r.frame()
    if not r.sweep:
        return [main]
    fillers = [r.frame(np.zeros(r.n, np.uint8))]
    for v in range(1, 40):
        c = np.zeros(r.n, np.uint8)
        c[min(1, r.n - 1)] = v
        c[r.n // 2] = v ^ 0x55
        fillers.append(r.frame(c))
    flen = [len(oracle_frame(r, f)) for f in fillers]
    comp = oracle_frame(r, main)
    p0 = parse_frame(np.frombuffer(comp, np.uint8), r.kind, r.n, r.ch)[0][2]
    frames, cur, want = [], 0, set(range(16))
    while want:
        # the shortest run of fillers that brings plane 0's payload to a residue not yet seen
        paths = {cur % 16: []}
        frontier = [cur % 16]
        while not any((c + p0) % 16 in want for c in paths):
            nxt = []
            for c in frontier:
                for i, L in enumerate(flen):
                    d = (c + L) % 16
                    if d not in paths:
                        paths[d] = paths[c] + [i]
                        nxt.append(d)
            frontier = nxt
        c = next(c for c in sorted(paths, key=lambda c: len(paths[c])) if (c + p0) % 16 in want)
        for i in paths[c]:
            frames.append(fillers[i])
            cur += flen[i]
        want.discard((cur + p0) % 16)
        frames.append(main)
        cur += len(comp)
    return frames


def huff_blocks(r, frames):
    """every HUFF block of the batch: (frame, plane, block, payload offset in the batch stream, payload bytes, Walk)"""
    out, base = [], 0
    for f, fr in enumerate(frames):
        comp = oracle_frame(r, fr)
        a = np.frombuffer(comp, np.uint8)
        for k, b, off, plen, mode in parse_frame(a, r.kind, r.n, r.ch):
            if mode == 1:
                out.append((f, k, b, base + off, plen, walk_of(a[off:off + plen], min(BLOCK, r.n - b * BLOCK))))
        base += len(comp)
    return out


# ---- classification of a HUFF block (the coverage test) ------------------------------------------------------
def classify(kind, plen, off, w):
    n = w.n
    loop = loop_of(kind, plen, n)
    width = LUT_BITS if loop == "single" else PAIR_BITS
    bits, nint = idx_geom(plen)
    lens = {s: l for s, (c, l) in w.codes.items()}
    long_syms = [s for s, l in lens.items() if l > width]
    prefixes = {}
    for s in long_syms:
        pre = w.codes[s][0] & ((1 << width) - 1)
        prefixes[pre] = prefixes.get(pre, 0) + 1
    cells = {("class", decode_class(plen), loop), ("off16", decode_class(plen), off % 16)}
    if long_syms:
        cells.add(("long", loop))
    if prefixes and max(prefixes.values()) >= 3:
        cells.add(("shared_prefix3", loop))
    for s in long_syms:
        if s >= 256:
            cells.add(("long_run", loop, s))
    # maximal zero runs
    z = np.concatenate([[0], (w.content() == 0).astype(np.int8), [0]])
    d = np.diff(z)
    for L in np.flatnonzero(d == -1) - np.flatnonzero(d == 1):
        if int(L) in RUN_LENGTHS:
            cells.add(("run_len", loop, int(L)))
    # tokens whose bits straddle an index interval boundary, by output position mod 4
    s, e, o, sy, ln = w.starts, w.ends, w.opos, w.syms, w.lens
    cross = (s // bits) != ((e - 1) // bits)
    for i in np.flatnonzero(cross & (sy >= 256)):
        cells.add(("run_straddle", loop, int(o[i]) & 3))
    lit = sy < 256
    pair_ok = lit[:-1] & lit[1:] & ((s[:-1] // bits) != ((e[1:] - 1) // bits))
    if loop != "single":
        pair_ok &= (ln[:-1] + ln[1:]) <= PAIR_BITS
    for i in np.flatnonzero(pair_ok):
        cells.add(("pair_straddle", loop, int(o[i]) & 3))
    # a pair / chain that the padding behind the last literal would complete past n
    zero_sym = next((s_ for s_, (c, l) in w.codes.items() if c == 0), None)
    if lit[-1] and zero_sym is not None and zero_sym < 256:
        lz = lens[zero_sym]
        if (loop == "single" and lz <= LUT_BITS) or (loop != "single" and ln[-1] + lz <= PAIR_BITS):
            cells.add(("past_n", loop))
    if len(w.codes) == 261 and decode_class(plen) == 1 and w.tree_nbits // bits >= 5:
        cells.add(("tree261_class1",))
    if len(w.codes) == 2:
        cells.add(("tree2",))
    cells.add(("maxlen", max(lens.values())))
    if plen in (SMALL, SMALL + 1, MEDIUM, MEDIUM + 1):
        cells.add(("plen", plen))
    if plen * 16 == n and loop != "single":
        cells.add(("pair_lo_edge",))
    if plen * 16 == n - 1:
        cells.add(("pair_lo_below",))
    if plen * 8 == PAIR_MAX_BITS * n and loop != "single":
        cells.add(("pair_hi_edge",))
    if plen * 8 == PAIR_MAX_BITS * n + 8:
        cells.add(("pair_hi_above",))
    if plen == min(n, BLOCK - 1) and off % 16 == 15:
        cells.add(("max_payload_lead15", decode_class(plen), n == BLOCK))
    if plen in (SMALL, MEDIUM) and off % 16 == 15:
        cells.add(("class_max_lead15", plen))
    if plen * 8 < n // 2:
        cells.add(("sparse",))
    return cells


def required_cells():
    req = {("class", c, lp) for c in (1, 2, 0) for lp in LOOPS}
    req |= {("off16", c, a) for c in (1, 2, 0) for a in range(16)}
    for lp in LOOPS:
        req |= {("long", lp), ("shared_prefix3", lp), ("past_n", lp)}
        req |= {("long_run", lp, s) for s in range(256, 261)}
        req |= {("run_len", lp, L) for L in RUN_LENGTHS}
        req |= {(kind, lp, a) for kind in ("run_straddle", "pair_straddle") for a in range(4)}
    req |= {("tree261_class1",), ("tree2",), ("pair_lo_edge",), ("pair_lo_below",), ("pair_hi_edge",),
            ("pair_hi_above",), ("sparse",)}
    req |= {("plen", p) for p in (SMALL, SMALL + 1, MEDIUM, MEDIUM + 1)}
    req |= {("class_max_lead15", SMALL), ("class_max_lead15", MEDIUM)}
    req |= {("max_payload_lead15", 1, False), ("max_payload_lead15", 2, False), ("max_payload_lead15", 0, False),
            ("max_payload_lead15", 0, True)}
    return req


def test_table_covers_every_decode_path(oracle):
    """Every cell of the table's design is reached by at least one HUFF block of the oracle's streams."""
    hit, maxlen = set(), 0
    for name in ROW_NAMES:
        r = build_row(name)
        if r.kind == "hadamard":
            w, hdr = r.oracle().transform(r.frame())
            assert np.array_equal(w, r.block.astype(np.int32)) and not hdr.any(), name
        for f, k, b, off, plen, w in huff_blocks(r, batch_frames(r)):
            cells = classify(r.kind, plen, off, w)
            maxlen = max([maxlen] + [c[1] for c in cells if c[0] == "maxlen"])
            hit |= {c for c in cells if c[0] != "maxlen"}
    assert maxlen >= 20, maxlen
    missing = sorted(required_cells() - hit, key=str)
    assert not missing, missing
    n = [build_row(x).n for x in ROW_NAMES]
    assert any(v % 16 and v % 4 for v in n) and 70001 in n and min(n) <= 4


# ---- on the GPU ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def R():
    import rspt_b200  # noqa: F401
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


def dev_u8(a):
    return torch.from_numpy(np.array(a, dtype=np.uint8, copy=True).reshape(-1)).cuda()


def check_index(sc, blocks, nblk, nb_alloc, rebuilt, what):
    """The decode-index entries of every HUFF block against the host's token walk.  Entry t of a block names bit
    t * bits + (e & 0xFFF) and output byte e >> 12.
      encoder:  a token boundary at or after max(t * bits, tree bits) -- a token's start with its output byte, or the
                end of the last token with n -- the entries non-decreasing in both.
      rebuilt:  the FIRST boundary at or after max(t * bits, tree bits), where k_hzr_build_index keeps walking past the
                last token through what the zero padding decodes to (output byte n), and the payload's last bit
                (with n) when no boundary is left before it."""
    for f, k, b, off, plen, w in blocks:
        bits, nint = idx_geom(plen)
        limit = 8 * plen
        slot = (off >> 6) + (f * nb_alloc + k) * nblk + b
        e = sc[slot:slot + nint].astype(np.int64)
        t = np.arange(nint)
        bit, pos = t * bits + (e & ((1 << POS_SHIFT) - 1)), e >> POS_SHIFT
        lo = np.maximum(t * bits, w.tree_nbits)
        where = (what, f, k, b, plen)
        if rebuilt:
            bounds = np.concatenate([w.starts, w.pseudo]).astype(np.int64)
            bpos = np.concatenate([w.opos, np.full(len(w.pseudo), w.n)]).astype(np.int64)
            i = np.searchsorted(bounds, lo)
            inside = i < bounds.size
            want_bit = np.where(inside, bounds[np.minimum(i, bounds.size - 1)], limit)
            want_pos = np.where(inside, bpos[np.minimum(i, bounds.size - 1)], w.n)
            bad = np.flatnonzero((bit != want_bit) | (pos != want_pos))
            assert not bad.size, (where, "rebuilt entries", bad[:5], bit[bad[:5]], want_bit[bad[:5]], pos[bad[:5]], want_pos[bad[:5]])
        else:
            at = dict(zip(w.starts.tolist(), w.opos.tolist()))
            at[w.end_bits] = w.n
            for j in range(nint):
                assert bit[j] >= lo[j] and at.get(int(bit[j])) == pos[j], (where, "encoder entry", j, bit[j], pos[j], lo[j])
            assert np.all(np.diff(bit) >= 0) and np.all(np.diff(pos) >= 0), (where, "encoder entries decrease")


def run_decode(fn, n_out, want, status_n, what):
    """fn(out, status) writes n_out bytes into a buffer with GUARD sentinel bytes on both sides"""
    buf = torch.full((n_out + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
    status = torch.full((status_n,), 7, dtype=torch.int32, device="cuda")
    fn(buf[GUARD:GUARD + n_out], status)
    torch.cuda.synchronize()
    st = status.cpu().numpy()
    assert not st.any(), (what, "status", st)
    h = buf.cpu().numpy()
    assert (h[:GUARD] == 0xA5).all() and (h[GUARD + n_out:] == 0xA5).all(), (what, "wrote outside its output")
    got = h[GUARD:GUARD + n_out]
    bad = np.flatnonzero(got != want)
    assert not bad.size, (what, "first wrong bytes at", bad[:8], got[bad[:8]], want[bad[:8]])


def expected_output(oracle, r, comps, frames):
    if r.kind == "hzr":
        return np.concatenate(frames)
    o = r.oracle()
    return np.concatenate([np.frombuffer(o.decompress(c)[0], np.uint8) for c in comps])


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("name", ROW_NAMES)
def test_decode_path(R, oracle, monkeypatch, name):
    """One row: the GPU stream equals the oracle's; the encoder's and the rebuilt decode index equal the host walk;
    every way of decoding the batch gives the input (hadamard: the oracle's decode) with status 0 and nothing written
    outside the output; verify_batch passes."""
    r = build_row(name)
    frames = batch_frames(r)
    nfr, nblk = len(frames), (r.n + BLOCK - 1) // BLOCK
    if r.stage is not None:
        monkeypatch.setenv("RSPT_SPARSE_STAGE_BYTES", str(r.stage))   # read when the handle is created
    p = R.SignalPacker(r.kind, 1 if r.kind == "hzr" else 4, r.ch, r.ns, NB[r.kind], max_batch_frames=nfr + 2)
    raw = np.concatenate(frames)
    batch = p.compress_batch(dev_u8(raw))
    torch.cuda.synchronize()
    offs = batch.offsets.cpu().numpy()
    stream = batch.stream[:int(offs[nfr])].cpu().numpy()
    comps = [oracle_frame(r, fr) for fr in frames]
    for i in range(nfr):
        assert stream[offs[i]:offs[i + 1]].tobytes() == comps[i], (name, "frame", i)
    blocks = huff_blocks(r, frames)
    check_index(batch.sidecar.cpu().numpy().view(np.uint32), blocks, nblk, NB[r.kind], False, name)
    assert not p.verify_batch(batch).cpu().numpy().any(), name
    want = expected_output(oracle, r, comps, frames)
    fb = p.frame_bytes

    bare = R.CompressedBatch(batch.stream, batch.offsets, batch.frame_nb, None, nfr)
    st = torch.zeros(nfr, dtype=torch.int32, device="cuda")
    rebuilt = p.build_index(bare, st)
    torch.cuda.synchronize()
    assert not st.cpu().numpy().any(), name
    check_index(rebuilt.sidecar.cpu().numpy().view(np.uint32), blocks, nblk, NB[r.kind], True, name)

    n_all = nfr * fb
    run_decode(lambda o, s: p.decompress_batch(batch, out=o, status=s), n_all, want, nfr, (name, "encoder index"))
    run_decode(lambda o, s: p.decompress_batch(rebuilt, out=o, status=s), n_all, want, nfr, (name, "rebuilt index"))
    run_decode(lambda o, s: p.decompress_batch(bare, out=o, status=s, use_sidecar=False), n_all, want, nfr, (name, "implicit index"))
    ids = list(range(nfr - 1, -1, -1)) + [0, nfr - 1]
    want_g = np.concatenate([want[i * fb:(i + 1) * fb] for i in ids])
    for src, use in ((batch, True), (bare, False)):
        run_decode(lambda o, s: p.decompress_frames(src, ids, out=o, status=s, use_sidecar=use), len(ids) * fb, want_g, len(ids),
                   (name, "decompress_frames", "stored index" if use else "own index"))
    p.close()
