"""The batch inflate paths on the device, through b200z_inflate_batch_device: k_inflate_fast alone (B200Z_FAST=2), the
default pair of passes (fast kernel, then the exact pair on what it leaves), the exact pair alone (B200Z_FAST=0) at every
lane shape, and k_inflate_fast walked by two CTAs -- all against the oracle, on a seeded corpus aimed at the fast kernel's
eligibility rule and internals, in batches large enough that every persistent CTA meets every kind of unit.

Also the output bounds the entry points promise (include/b200z.h): unit u writes out_base[out_off[u] .. +out_cap[u]) and
nothing else, the device workspace is what b200z_inflate_workspace_bytes says (sized by the layout's extent), and the host
entry points leave the caller's bytes between slots alone.

With B200Z_EMU_TESTS=1 the library is the emulation build, whose "device" pointers are host pointers: the helper then uses
numpy buffers and the same tests run on the CPU (smaller batches; tests that need torch tensors are `needs_device`)."""
import heapq
import os
import random
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import oracle_lib as orc  # noqa: E402

pytestmark = pytest.mark.gpu

EMU = os.environ.get("B200Z_EMU_TESTS") == "1"
SENT_LEN, SENT_ST, SENT_USED = 0xDEADBEEF, -77, 0xFEEDF00D
FILL = 0x5A
GUARD = 1 << 20
# k_inflate_fast's limits (archive_b200/csrc/inflate_fast.cuh)
IN_CAP, MIN_IN, WIN, SUBN, LB, DB = 30720, 192, 65536, 384, 10, 8

# ====================================================================================== a small DEFLATE writer
LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEXT = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
         8193, 12289, 16385, 24577]
DEXT = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 30


def len_sym(n):
    i = max(k for k in range(29) if LBASE[k] <= n)
    return 257 + i, LEXT[i], n - LBASE[i]


def dist_sym(d):
    i = max(k for k in range(30) if DBASE[k] <= d)
    return i, DEXT[i], d - DBASE[i]


def canonical(lens):
    """RFC 1951 3.2.2: code of every symbol (MSB first); over-subscribed sets get whatever the counting gives."""
    ml = max(lens) if lens else 0
    bl = [0] * (ml + 2)
    for v in lens:
        if v:
            bl[v] += 1
    nxt, code = [0] * (ml + 2), 0
    for b in range(1, ml + 1):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    codes = [0] * len(lens)
    for s, v in enumerate(lens):
        if v:
            codes[s] = nxt[v] & ((1 << v) - 1)
            nxt[v] += 1
    return codes


def subtable_entries(lens, root):
    """Second-level entries k_inflate_fast allocates for one alphabet (inflate_fast.cuh, the table build): every root
    prefix (the first `root` bits of a code) that has codes longer than the root gets a sub-table of 2^(m - root)
    entries, m = the longest code under that prefix.  The lit/len (root 10) and distance (root 8) sub-tables share one
    pool of SUBN = 384 entries; a block that needs more is left to the exact kernels."""
    longest = {}
    for c, v in zip(canonical(lens), lens):
        if v > root:
            p = c >> (v - root)
            longest[p] = max(longest.get(p, 0), v)
    return sum(1 << (m - root) for m in longest.values())


def huffman_lengths(freq, limit):
    """Code lengths from frequencies (plain Huffman; frequencies halved until the longest code fits `limit`)."""
    f = list(freq)
    while True:
        items = [(v, i, [s]) for i, (s, v) in enumerate((s, v) for s, v in enumerate(f) if v)]
        lens = [0] * len(f)
        if len(items) == 1:
            lens[items[0][2][0]] = 1
            return lens
        heapq.heapify(items)
        k = len(f)
        while len(items) > 1:
            a, b = heapq.heappop(items), heapq.heappop(items)
            for s in a[2] + b[2]:
                lens[s] += 1
            heapq.heappush(items, (a[0] + b[0], k, a[2] + b[2]))
            k += 1
        if max(lens) <= limit:
            return lens
        f = [(v + 1) >> 1 if v else 0 for v in f]


class Bits:
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, val, n):
        self.v |= (val & ((1 << n) - 1)) << self.n
        self.n += n

    def huff(self, code, n):  # Huffman codes go MSB first
        self.put(int(format(code, f"0{n}b")[::-1], 2) if n else 0, n)

    def align(self):
        self.n = (self.n + 7) & ~7

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")


def rle_lengths(lens):
    """-> [(cl symbol, extra value)] for a run-length coded sequence of code lengths (symbols 16 / 17 / 18)."""
    out, i = [], 0
    while i < len(lens):
        v, r = lens[i], 1
        while i + r < len(lens) and lens[i + r] == v:
            r += 1
        i += r
        if v == 0:
            while r >= 11:
                k = min(r, 138); out.append((18, k - 11)); r -= k
            if r >= 3:
                out.append((17, r - 3)); r = 0
            out += [(0, 0)] * r
        else:
            out.append((v, 0)); r -= 1
            while r >= 3:
                k = min(r, 6); out.append((16, k - 3)); r -= k
            out += [(v, 0)] * r
    return out


def write_tokens(bw, tokens, lit_codes, lit_lens, d_codes, d_lens):
    for t in tokens:
        if isinstance(t, int):
            bw.huff(lit_codes[t], lit_lens[t])
        else:
            n, d = t
            s, eb, ev = len_sym(n)
            bw.huff(lit_codes[s], lit_lens[s]); bw.put(ev, eb)
            s, eb, ev = dist_sym(d)
            bw.huff(d_codes[s], d_lens[s]); bw.put(ev, eb)
    bw.huff(lit_codes[256], lit_lens[256])


def encode(blocks, final=True):
    """blocks: ("fixed", tokens) | ("dyn", tokens[, lit_lens, dist_lens]) | ("stored", bytes).  Tokens are literal byte
    values or (length, distance).  The last block is BFINAL unless final=False (a stream that ends after a flush)."""
    bw = Bits()
    for k, b in enumerate(blocks):
        bw.put(1 if (final and k == len(blocks) - 1) else 0, 1)
        if b[0] == "stored":
            bw.put(0, 2); bw.align()
            bw.put(len(b[1]), 16); bw.put(len(b[1]) ^ 0xffff, 16)
            for c in b[1]:
                bw.put(c, 8)
            continue
        if b[0] == "fixed":
            bw.put(1, 2)
            write_tokens(bw, b[1], canonical(FIXED_LIT), FIXED_LIT, canonical(FIXED_DIST), FIXED_DIST)
            continue
        tokens = b[1]
        if len(b) > 2:
            ll, dl = list(b[2]), list(b[3])
        else:
            lf, df = [0] * 286, [0] * 30
            lf[256] = 1
            for t in tokens:
                if isinstance(t, int):
                    lf[t] += 1
                else:
                    lf[len_sym(t[0])[0]] += 1
                    df[dist_sym(t[1])[0]] += 1
            ll = huffman_lengths(lf, 15)
            dl = huffman_lengths(df, 15) if any(df) else [1]
        while len(ll) > 257 and ll[-1] == 0:
            ll.pop()
        while len(dl) > 1 and dl[-1] == 0:
            dl.pop()
        seq = rle_lengths(ll + dl)
        cf = [0] * 19
        for s, _ in seq:
            cf[s] += 1
        cl = huffman_lengths(cf, 7)
        ncl = 19
        while ncl > 4 and cl[CL_ORDER[ncl - 1]] == 0:
            ncl -= 1
        bw.put(2, 2)
        bw.put(len(ll) - 257, 5); bw.put(len(dl) - 1, 5); bw.put(ncl - 4, 4)
        for i in range(ncl):
            bw.put(cl[CL_ORDER[i]], 3)
        cc = canonical(cl)
        for s, e in seq:
            bw.huff(cc[s], cl[s])
            if s >= 16:
                bw.put(e, {16: 2, 17: 3, 18: 7}[s])
        write_tokens(bw, tokens, canonical(ll), ll, canonical(dl), dl)
    return bw.bytes()


def expand(tokens, out=None):
    out = bytearray() if out is None else out
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
        else:
            n, d = t
            for _ in range(n):
                out.append(out[-d])
    return out


def gen_tokens(rng, n_out, alphabet, p_match=0.3, max_len=40, max_dist=32768, start=0):
    """Random tokens that produce exactly n_out bytes after `start` bytes of earlier output."""
    toks, pos, end = [], start, start + n_out
    while pos < end:
        left = end - pos
        if pos > 0 and left >= 3 and rng.random() < p_match:
            n = min(left, rng.randint(3, max_len))
            toks.append((n, rng.randint(1, min(pos, max_dist))))
            pos += n
        else:
            toks.append(rng.choice(alphabet))
            pos += 1
    return toks


def fill_lengths(n, space, max_len):
    """n code lengths whose Kraft sum is space / 2^15: the binary expansion of `space`, then the shortest code split in
    two until there are n (no split makes a code longer than max_len)."""
    lens = [b for b in range(1, 16) if space >> (15 - b) & 1]
    assert sum(1 << (15 - v) for v in lens) == space
    while len(lens) < n:
        i = lens.index(min(lens))
        v = lens.pop(i)
        assert v < max_len
        lens += [v + 1, v + 1]
    assert len(lens) == n
    return lens


def assign(rng, lens_multiset, n_sym, keep_short=()):
    """Lengths to symbols: the symbols in keep_short get the shortest codes, the others a seeded shuffle."""
    ls = sorted(lens_multiset)
    out = [0] * n_sym
    for s in keep_short:
        out[s] = ls.pop(0)
    rest = [s for s in range(n_sym) if s not in keep_short]
    rng.shuffle(ls)
    for s, v in zip(rest, ls):
        out[s] = v
    return out


def code_sets(rng, lit_full15, lit_tail11, dist_tail9):
    """A complete lit/len code over all 286 symbols (HLIT maximal) and a complete distance code over all 30 (HDIST
    maximal).  Canonical codes are ordered by length, so the longest codes take the last root prefixes:
      lit/len  32 * lit_full15 codes of 15 bits fill lit_full15 root prefixes of 10 bits, 2^(15-10) = 32 entries each;
               lit_tail11 codes of 11 bits sit in the prefixes before them, 2^(11-10) = 2 entries per prefix they touch
      distance a chain of 10..15-bit codes (half of one 8-bit root prefix) and the 9-bit code(s) beside it: that prefix
               needs 2^(15-8) = 128 entries; dist_tail9 more 9-bit codes spill into the prefix before, 2 entries.
    So (8, 0, 0) needs 8 * 32 + 128 = 384 = SUBN entries, exactly the pool; (8, 1, 0) and (8, 0, 2) need 386, the
    least a set can need beyond it (sub-tables are powers of two).  subtable_entries() counts it the kernel's way."""
    n15 = 32 * lit_full15
    lit_space = (1 << 15) - n15 - lit_tail11 * (1 << 4)
    lit = fill_lengths(286 - n15 - lit_tail11, lit_space, LB) + [15] * n15 + [11] * lit_tail11
    chain = [10, 11, 12, 13, 14, 15, 15]
    d_long = chain + [9] * dist_tail9
    d_space = (1 << 15) - sum(1 << (15 - v) for v in d_long)
    dist = fill_lengths(30 - len(d_long), d_space, DB) + d_long
    return assign(rng, lit, 286, keep_short=(256,)), assign(rng, dist, 30)


# ====================================================================================== the corpus
class Unit:
    __slots__ = ("cls", "data", "cap", "lead", "finish", "leave")

    def __init__(self, cls, data, cap=None, lead=None, finish=False, leave=False):
        self.cls, self.data, self.lead, self.finish, self.leave = cls, bytes(data), lead, finish, leave
        self.cap = cap


def deflate(data, level=6, wbits=15, mem=9, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, -wbits, mem, strategy)
    return co.compress(data) + co.flush()


def text(rng, n, nwords=2000):
    words = [bytes(rng.choice(b"etaoinshrdlucmfwypvbgkqjxz") for _ in range(rng.randint(2, 10))) for _ in range(nwords)]
    b = bytearray()
    while len(b) < n:
        b += rng.choice(words) + rng.choice([b" ", b" ", b", ", b".\n"])
    return bytes(b[:n])


def edge_corpus(small=False):
    """Seeded units, each with its class; finish=True: k_inflate_fast must finish it, leave=True: it must leave it."""
    from archive_b200 import synth
    rng = random.Random(20261017)
    U = []
    # benchmark shape: 64 KiB of the synthetic text, one dynamic block, + the 8-byte gzip trailer
    t = synth.text(8 * 65536, stream=5)
    for i in range(8):
        U.append(Unit("bench", synth.deflate_raw(t[i * 65536:(i + 1) * 65536].tobytes()) + bytes(8), 65536, finish=True))
    # MIN_IN: trailing junk after the final block sets in_len to the byte without changing the output
    z = deflate(text(rng, 120) * 5)
    assert len(z) < 180
    for il in (191, 192, 193):
        U.append(Unit("min_in", z + bytes(rng.randrange(256) for _ in range(il - len(z))), finish=il >= MIN_IN,
                      leave=il < MIN_IN))
    # IN_CAP: (lead + il + 15) & ~15 <= 30720 decides, for every lead 0..15 and il on both sides
    z = synth.deflate_raw(t[:65536].tobytes(), 9)
    assert len(z) < 30705, len(z)
    leads = range(16) if not small else (0, 1, 15)
    ils = range(30705, 30722) if not small else (30705, 30706, 30720, 30721)
    for lead in leads:
        for il in ils:
            ok = (lead + il + 15) & ~15 <= IN_CAP
            U.append(Unit("in_cap", z + bytes(0xA5 for _ in range(il - len(z))), 65536, lead=lead, finish=ok, leave=not ok))
    # out_cap around the output size and the 64 KiB window
    p = text(rng, 30000)
    z = deflate(p) + bytes(8)
    for cap, fin, lv in ((0, False, True), (len(p) - 1, False, True), (len(p), True, False), (65535, True, False),
                         (65536, True, False), (65537, False, True)):
        U.append(Unit("out_cap", z, cap, finish=fin, leave=lv))
    # an output of exactly 64 KiB whose last token is a match
    alpha = list(b"abcdefghijklmnop")
    toks = gen_tokens(rng, 65536 - 258, alpha, p_match=0.5, max_len=60) + [(258, 1000)]
    z = encode([("dyn", toks)]) + bytes(8)
    U.append(Unit("out_64k_last_match", z, 65536, finish=True))
    # distance 32768, length 258; distance-1 runs; overlapping copies across the 1 KiB LZ77 chunks; long chains
    toks = [rng.choice(alpha) for _ in range(32768)] + [(258, 32768)] * 100
    U.append(Unit("dist32768_len258", encode([("dyn", toks)]) + bytes(8), finish=True))
    toks = [65]
    for k in range(120):
        toks += [(258, 1), rng.choice(alpha), (rng.randint(3, 258), 1)]
    U.append(Unit("dist1_runs", encode([("dyn", toks)]) + bytes(8), finish=True))
    toks = gen_tokens(rng, 600, alpha)
    pos = 600
    for c in range(1, 60):
        edge = c * 1024 - rng.randint(1, 200)
        if edge <= pos:
            continue
        toks += gen_tokens(rng, edge - pos, alpha, start=pos)
        d = rng.choice([1, 2, 3, 7, 31, 100, 255, 257])
        toks.append((258, d))
        pos = edge + 258
    U.append(Unit("overlap_chunks", encode([("dyn", toks)]) + bytes(8), finish=True))
    toks = [rng.choice(alpha) for _ in range(2100)]
    pos = 2100
    while pos + 258 <= 60000:  # each copy reads bytes that are themselves copies, from the chunk before
        toks.append((258, rng.choice([700, 1024, 1100, 2047])))
        pos += 258
    U.append(Unit("chains", encode([("dyn", toks)]) + bytes(8), finish=True))
    # block structure: stored blocks inside eligible units, sync flushes (empty stored blocks), ends without a final
    # block, memLevel 1, fixed blocks, every window size
    for k in range(3):
        a = gen_tokens(rng, 5000, alpha)
        st = bytes(rng.randrange(256) for _ in range(rng.choice([1, 1000, 4000])))
        b = gen_tokens(rng, 3000, alpha, start=5000 + len(st))
        U.append(Unit("stored_inside", encode([("dyn", a), ("stored", st), ("fixed", b), ("stored", b"")]) + bytes(8),
                      finish=True))
    for k in range(3):
        p = text(rng, 40000)
        co = zlib.compressobj(6, zlib.DEFLATED, -15, 8)
        z = b"".join(co.compress(p[i:i + 9000]) + co.flush(zlib.Z_SYNC_FLUSH) for i in range(0, 40000, 9000))
        U.append(Unit("sync_flush", z + co.flush() + bytes(8), finish=True))
        U.append(Unit("eos_no_final", z, finish=True))
    for n in (3000, 20000):
        U.append(Unit("memlevel1", deflate(text(rng, n), 6, 15, 1) + bytes(8), finish=True))
        U.append(Unit("fixed", deflate(text(rng, n), 6, 15, 9, zlib.Z_FIXED) + bytes(8), finish=True))
    for w in range(9, 16):
        U.append(Unit("wbits", deflate(text(rng, 30000), 9, w) + bytes(8), finish=True))
    # hand-written code sets zlib never emits (HLIT 286, HDIST 30, codes of 15 bits, a single distance code)
    lit, dist = code_sets(rng, 8, 0, 0)
    assert subtable_entries(lit, LB) == 256 and subtable_entries(dist, DB) == 128  # exactly SUBN
    for k in range(2):
        toks = gen_tokens(rng, rng.randint(15000, 30000), list(range(256)), p_match=0.35)
        U.append(Unit("subn_exact", encode([("dyn", toks, lit, dist)]) + bytes(8), finish=True))
    lit2, dist2 = code_sets(rng, 8, 1, 0)
    assert subtable_entries(lit2, LB) == 258 and subtable_entries(dist2, DB) == 128
    lit3, dist3 = code_sets(rng, 8, 0, 2)
    assert subtable_entries(lit3, LB) == 256 and subtable_entries(dist3, DB) == 130
    for ll, dl in ((lit2, dist2), (lit3, dist3)):
        toks = gen_tokens(rng, 20000, list(range(256)), p_match=0.35)
        U.append(Unit("subn_over", encode([("dyn", toks, ll, dl)]) + bytes(8), leave=True))
    lit4, dist4 = code_sets(rng, 2, 5, 0)
    assert subtable_entries(lit4, LB) + subtable_entries(dist4, DB) < SUBN
    toks = gen_tokens(rng, 25000, list(range(256)), p_match=0.35)
    U.append(Unit("long_codes", encode([("dyn", toks, lit4, dist4), ("dyn", gen_tokens(rng, 5000, alpha, start=25000))])
                  + bytes(8), finish=True))
    toks = [66] + [rng.choice([(rng.randint(3, 258), 1), rng.choice(alpha)]) for _ in range(3000)]
    U.append(Unit("one_dist_code", encode([("dyn", toks, huffman_lengths([1] * 256 + [1] + [1] * 29, 15), [1])])
                  + bytes(8)))
    # mid-unit abandonment: clean blocks, then a last block that trips a fallback
    for k in range(2):
        a = gen_tokens(rng, 6000, alpha)
        over = [8] * 286  # over-subscribed: 286 codes of 8 bits
        U.append(Unit("abandon_oversubscribed", encode([("dyn", a), ("dyn", [1, 2, 3], over, [5] * 30)]) + bytes(8),
                      leave=True))
        U.append(Unit("abandon_dist_before_start", encode([("dyn", a), ("fixed", [70, (10, 20000)])]) + bytes(8), 65536,
                      leave=True))
        b = gen_tokens(rng, 5000, alpha, start=6000)
        U.append(Unit("abandon_out_cap", encode([("dyn", a), ("dyn", b)]) + bytes(8), 6000 + 100, leave=True))
    # damaged units
    base = [deflate(text(rng, rng.randint(2000, 50000)), rng.choice([1, 6, 9])) for _ in range(4)]
    for z in base:
        for _ in range(3 if small else 8):
            b = bytearray(z + bytes(8))
            pos = rng.randrange(len(z) * 8)
            b[pos >> 3] ^= 1 << (pos & 7)
            U.append(Unit("bitflip", b, 65536))
        for cut in (len(z) // 3, len(z) - 1, len(z) - 5):
            U.append(Unit("truncated", z[:cut], 65536))
    for u in U:
        st, out, _ = orc.inflate(u.data)
        if u.cap is None:
            u.cap = len(out)
        assert st == orc.OK or not u.finish, u.cls  # the clean units are clean
    return U


def batch(small=False, n_min=None):
    """The edge corpus interleaved with benchmark-shape units (and repeated) to at least n_min units, seeded."""
    from archive_b200 import synth
    edge = edge_corpus(small)
    if n_min is None:
        n_min = 64 if small else 4 * 296
    t = synth.text(16 * 65536, stream=6)
    filler = [Unit("bench", synth.deflate_raw(t[i * 65536:(i + 1) * 65536].tobytes()) + bytes(8), 65536, finish=True)
              for i in range(16)]
    rng = random.Random(99)
    units = []
    while len(units) < n_min:
        e = edge[:]
        rng.shuffle(e)
        for u in e:  # eligible, ineligible and abandoned units alternate, with benchmark units between
            units.append(u)
            if rng.random() < 0.5:
                units.append(rng.choice(filler))
    return units


# ====================================================================================== the device entry
def n_sms():
    if EMU:
        return 148
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


class Run:
    pass


def run_device(units, env=None, layout=None, ws_extent=None, seed=1, ws_pattern=False):
    """units -> Run: b200z_inflate_batch_device on device buffers (numpy buffers on the emulation build).  `env`: the
    B200Z_* settings for this call (read at every launch).  Checks the bounds the entry point promises and returns
    the per-unit arrays and the whole output buffer (and the workspace before and after, with ws_pattern: a seeded
    pattern instead of zeros)."""
    from archive_b200 import _ffi
    L = _ffi.ensure_init()
    rng = random.Random(seed)
    n = len(units)
    # input: every in_off % 16 (the lead k_inflate_fast stages in front of a unit), chosen per unit where it matters
    blob = bytearray(rng.randrange(256) for _ in range(7))
    in_off = np.zeros(n, np.uint64)
    for i, u in enumerate(units):
        lead = u.lead if u.lead is not None else i % 16
        blob += bytes(0xC3 for _ in range((lead - len(blob)) % 16))
        in_off[i] = len(blob)
        blob += u.data
    blob += bytes(64)
    in_len = np.array([len(u.data) for u in units], np.uint32)
    caps = np.array([u.cap for u in units], np.uint32)
    if layout is None:
        out_off = np.zeros(n, np.uint64)
        o = rng.randrange(16)
        for i in range(n):
            o += rng.randint(0, 40)
            out_off[i] = o
            o += int(caps[i])
        if n >= 64:
            assert len(set(int(x) % 16 for x in out_off)) == 16
    else:
        out_off = np.array(layout, np.uint64)
    extent = int(max(int(out_off[i]) + int(caps[i]) for i in range(n)))
    out_bytes = extent + 97
    ws = L.b200z_inflate_workspace_bytes(n, len(blob), extent if ws_extent is None else ws_extent)
    guard = (np.arange(GUARD, dtype=np.uint32) * 2654435761 >> 13).astype(np.uint8)
    init = [np.full(n, SENT_LEN, np.uint32), np.full(n, SENT_ST, np.int32), np.full(n, SENT_USED, np.uint32)]
    host = dict(inp=np.frombuffer(bytes(blob), np.uint8), in_off=in_off, in_len=in_len, out=np.full(out_bytes, FILL, np.uint8),
                out_off=out_off, cap=caps, ol=init[0], st=init[1], iu=init[2],
                ws=np.concatenate([np.random.default_rng(seed).integers(0, 256, ws, np.uint8) if ws_pattern
                                   else np.zeros(ws, np.uint8), guard]))
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        if EMU:
            keep = {k: np.ascontiguousarray(v).copy() for k, v in host.items()}
            ptr = {k: v.ctypes.data for k, v in keep.items()}
            rc = L.b200z_inflate_batch_device(ptr["inp"], ptr["in_off"], ptr["in_len"], ptr["out"], ptr["out_off"], ptr["cap"],
                                              ptr["ol"], ptr["st"], ptr["iu"], n, ptr["ws"], ws, None)
            assert rc == 0, _ffi.last_error()
            back = keep
        else:
            import torch
            dev = {k: torch.from_numpy(v.view(np.uint8).copy()).cuda() for k, v in host.items()}
            assert dev["inp"].data_ptr() % 256 == 0  # so that lead = in_off & 15
            ptr = {k: v.data_ptr() for k, v in dev.items()}
            torch.cuda.synchronize()
            rc = L.b200z_inflate_batch_device(ptr["inp"], ptr["in_off"], ptr["in_len"], ptr["out"], ptr["out_off"], ptr["cap"],
                                              ptr["ol"], ptr["st"], ptr["iu"], n, ptr["ws"], ws,
                                              torch.cuda.current_stream().cuda_stream)
            assert rc == 0, _ffi.last_error()
            torch.cuda.synchronize()
            back = {k: dev[k].cpu().numpy().view(host[k].dtype) for k in ("out", "ol", "st", "iu", "ws")}
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    r = Run()
    r.out, r.out_off, r.cap = back["out"], out_off, caps
    r.ws_before, r.ws_after = host["ws"][:ws], back["ws"][:ws]
    r.out_len, r.status, r.in_used = back["ol"].copy(), back["st"].copy(), back["iu"].copy()
    r.left = (r.out_len == SENT_LEN) & (r.status == SENT_ST) & (r.in_used == SENT_USED)
    assert np.array_equal(back["ws"][ws:], guard), "a write past the end of the workspace"
    # nothing outside the units' slots changes; a unit that is left keeps its slot as it was
    mask = np.zeros(out_bytes, bool)
    for i in range(n):
        a, c = int(out_off[i]), int(caps[i])
        if r.left[i]:
            assert (r.out[a:a + c] == FILL).all(), f"unit {i} ({units[i].cls}) is left but its slot was written"
        mask[a:a + c] = True
    assert (r.out[~mask] == FILL).all(), "a write outside every unit's output slot"
    r.bytes = [r.out[int(out_off[i]):int(out_off[i]) + min(int(r.out_len[i]), int(caps[i]))].tobytes() for i in range(n)]
    return r


def tuples(r):
    return [(int(r.status[i]), int(r.out_len[i]), int(r.in_used[i]), r.bytes[i]) for i in range(len(r.bytes))]


_ORC = {}


def oracle(u):
    k = (u.data, u.cap)
    if k not in _ORC:
        _ORC[k] = (orc.inflate(u.data), orc.emul_inflate(u.data, u.cap))
    return _ORC[k]


def check_vs_oracle(units, r):
    """Every unit against the oracle, by the rules of test_inflate_gpu.py::test_batch_bad_data_vs_oracle."""
    for i, u in enumerate(units):
        st, out, used = int(r.status[i]), r.bytes[i], int(r.in_used[i])
        (ost, oout, oused), _ = oracle(u)
        where = f"unit {i} ({u.cls}, in_len {len(u.data)}, cap {u.cap})"
        assert int(r.out_len[i]) <= u.cap or st == -2, where
        if st == -2:
            assert oout[:len(out)] == out and (len(oout) > u.cap or ost != orc.OK), where
        elif ost == orc.OK:
            if st in (0, 1, -1):
                assert out == oout, where
                if st == 0:
                    assert used == oused, where
            else:
                assert st in (-3, -4) and oout[:len(out)] == out, (where, st)
        elif ost == orc.RUNAWAY:
            assert st == -4, (where, st)
        else:
            assert st in (-3, -4, -5), (where, st)


# ====================================================================================== tests
@pytest.fixture(scope="module")
def units():
    return batch(small=EMU)


@pytest.fixture(scope="module")
def exact(units):
    return run_device(units, {"B200Z_FAST": "0"})


@pytest.fixture(scope="module")
def fast_only(units):
    return run_device(units, {"B200Z_FAST": "2"})


def test_writer_round_trips_through_zlib():
    """The hand-written encoder is itself checked against zlib before it is trusted with edge cases."""
    rng = random.Random(4)
    alpha = list(b"xyz01")
    toks = gen_tokens(rng, 5000, alpha, p_match=0.4, max_len=258)
    lit, dist = code_sets(rng, 8, 0, 0)
    for blocks in ([("fixed", toks)], [("dyn", toks)], [("dyn", toks, lit, dist)], [("stored", b"abc"), ("dyn", toks)]):
        z = encode(blocks)
        want = bytes(expand([t for b in blocks for t in (list(b[1]) if b[0] == "stored" else b[1])]))
        assert zlib.decompress(z, -15) == want


def test_fast_only(units, fast_only, capsys):
    """B200Z_FAST=2: what k_inflate_fast finishes is exact; what it leaves is untouched; the units it must take it takes,
    and the ones it must leave (out_cap > 64 KiB, in_len < 192, more than IN_CAP staged bytes, more than SUBN sub-table
    entries, a last block that falls back) it leaves."""
    r = fast_only
    counts = {}
    for i, u in enumerate(units):
        c = counts.setdefault(u.cls, [0, 0])
        c[1] += 1
        where = f"unit {i} ({u.cls}, in_len {len(u.data)}, lead {u.lead}, cap {u.cap})"
        if r.left[i]:
            assert not u.finish, f"{where}: must finish in k_inflate_fast"
            continue
        c[0] += 1
        assert not u.leave, f"{where}: must be left to the exact kernels"
        (ost, oout, oused), (est, eout, eused, _) = oracle(u)
        assert est in (0, 1), f"{where}: finished although the exact logic reports {est}"
        assert ost == orc.OK and oout == eout, where
        assert r.bytes[i] == eout, f"{where}: bytes"
        assert int(r.out_len[i]) == len(eout), f"{where}: out_len"
        assert int(r.status[i]) == est, f"{where}: status"
        assert int(r.in_used[i]) == eused, f"{where}: in_used"
        if est == 0:
            assert oused == eused, where
        # the tail of a finished unit's slot is not written
        a = int(r.out_off[i])
        assert (r.out[a + len(eout):a + u.cap] == FILL).all(), f"{where}: write past out_len"
    with capsys.disabled():
        print("\nk_inflate_fast finished (of units) by class: " +
              ", ".join(f"{k} {v[0]}/{v[1]}" for k, v in sorted(counts.items())))
    for cls in ("bench", "in_cap", "min_in", "out_cap", "subn_exact", "subn_over", "abandon_oversubscribed"):
        assert cls in counts


@pytest.mark.parametrize("mode", ["default", "spare"])
def test_paths_agree(units, exact, fast_only, mode):
    """The default pair of passes, and k_inflate_fast walked by two CTAs only (B200Z_FAST_SPARE_SMS = SMs - 1: the
    header parsed ahead and the bulk loads pipelined across hundreds of consecutive units), give what the exact pair
    alone gives, unit for unit; and every unit agrees with the oracle."""
    env = {"B200Z_FAST": "1"} if mode == "default" else {"B200Z_FAST": "1", "B200Z_FAST_SPARE_SMS": str(n_sms() - 1)}
    r = run_device(units, env, ws_pattern=True)
    check_vs_oracle(units, exact)
    # a unit k_inflate_fast finished costs the exact pair nothing: k_inflate_decode skips it, so its token region (4
    # bytes per output byte from 4 * out_off, the workspace layout of inflate_ws_carve) keeps the pattern it had
    for i in np.flatnonzero(~fast_only.left):
        a, c = 4 * int(r.out_off[i]), 4 * int(r.cap[i])
        assert np.array_equal(r.ws_after[a:a + c], r.ws_before[a:a + c]), \
            f"unit {i} ({units[i].cls}) was finished by k_inflate_fast and decoded again by k_inflate_decode"
    a, b = tuples(r), tuples(exact)
    for i in range(len(units)):
        assert a[i] == b[i], f"unit {i} ({units[i].cls}): {a[i][:3]} vs the exact pair's {b[i][:3]}"


LANE_SHAPES = [{"B200Z_UPW": "32"}, {"B200Z_UPW": "8"}, {"B200Z_UPW": "4"}, {"B200Z_UPW": "8", "B200Z_SPEC_G": "2"}]


@pytest.mark.parametrize("shape", LANE_SHAPES, ids=lambda s: "_".join(f"{k[6:]}{v}" for k, v in s.items()))
def test_exact_pair_lane_shapes(units, exact, shape):
    """The exact pair at 1, 4 and 8 lanes per stream, and 8 streams of 2 lanes: the settings are read once per process,
    so each shape runs in a process of its own, which writes its results to a file."""
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "r.npz")
        env = dict(os.environ, **shape, B200Z_FAST="0")
        subprocess.run([sys.executable, os.path.abspath(__file__), path], env=env, cwd=ROOT, check=True,
                       timeout=900 if EMU else 300)
        got = np.load(path, allow_pickle=False)
        n = len(units)
        assert len(got["status"]) == n
        for i in range(n):
            ol = int(got["out_len"][i])
            o = int(got["off"][i])
            t = (int(got["status"][i]), ol, int(got["in_used"][i]), got["bytes"][o:o + min(ol, units[i].cap)].tobytes())
            want = tuples(exact)[i]
            if t[0] in (-2, -3) and t[0] == want[0]:
                # A match past out_cap or before the start, found in k_inflate_expand in tokens a helper lane decoded:
                # in_used is where the decode lane stopped, which depends on the lanes per stream.  Only in_used.
                t, want = t[:2] + t[3:], want[:2] + want[3:]
            assert t == want, f"unit {i} ({units[i].cls}) under {shape}"


def test_sparse_layout_workspace_by_extent():
    """Slots far apart, in an order that is not the units' order, the last one at the top of the extent with a 64 KiB
    output of literals (a token per byte: the most tokens a slot can hold); the workspace is sized by the extent, as
    the header says, and nothing is written past it."""
    rng = random.Random(8)
    from archive_b200 import synth
    t = synth.text(4 * 65536, stream=8).tobytes()
    us = [Unit("bench", synth.deflate_raw(t[i * 65536:(i + 1) * 65536]) + bytes(8), 65536) for i in range(4)]
    lit = bytes(rng.randrange(256) for _ in range(65536))
    us.append(Unit("literals", encode([("dyn", list(lit))]) + bytes(8), 65536))
    us.append(Unit("literals_fixed", encode([("fixed", list(lit[:30000]))]) + bytes(8), 30000))
    for extra in (0, 64, 100, 200, 255):  # extents on every side of the workspace's 256-byte rounding
        layout = [0, 300000 + extra, 150001, 77777, 500000 + extra, 420000]
        for env in ({"B200Z_FAST": "0"}, {"B200Z_FAST": "1"}, {"B200Z_FAST": "0", "B200Z_UPW": "1"}):
            r = run_device(us, env, layout=layout)
            check_vs_oracle(us, r)
            assert all(int(s) == 0 for s in r.status), (extra, env, list(r.status))


# ---------------------------------------------------------------------------- host entry points
def host_call(L, fn, units, out, out_off, caps, multi=False):
    from archive_b200 import _ffi
    n = len(units)
    blob = b"".join(u.data for u in units)
    in_off = np.cumsum([0] + [len(u.data) for u in units[:-1]]).astype(np.uint64)
    in_len = np.array([len(u.data) for u in units], np.uint32)
    caps = np.array(caps, np.uint32)
    out_off = np.array(out_off, np.uint64)
    ol, st, iu = np.zeros(n, np.uint32), np.zeros(n, np.int32), np.zeros(n, np.uint32)
    addr, nb, keep = _ffi.as_buffer(blob)
    p = lambda a: a.ctypes.data
    args = [addr, nb, p(in_off), p(in_len), p(out), out.size, p(out_off), p(caps), p(ol), p(st), p(iu), n]
    rc = fn(*args, 0) if multi else fn(*args)
    assert rc == 0, _ffi.last_error()
    return ol, st


@pytest.mark.parametrize("entry", ["batch", "batch_multi"])
def test_host_entries_leave_gaps_alone(entry):
    """b200z_inflate_batch / b200z_inflate_batch_multi (one device) write the units' slots and nothing between them,
    even when the library's device buffer still holds an earlier call's output there."""
    from archive_b200 import _ffi, synth
    L = _ffi.ensure_init()
    t = synth.text(6 * 65536, stream=11).tobytes()
    us = [Unit("bench", synth.deflate_raw(t[i * 65536:(i + 1) * 65536]) + bytes(8), 65536) for i in range(6)]
    multi = entry == "batch_multi"
    if multi:
        assert L.b200z_multi_init(1, 0) == 0, L.b200z_last_error()
    fn = L.b200z_inflate_batch_multi if multi else L.b200z_inflate_batch
    try:
        # first call: a contiguous layout fills the device buffer with decoded text
        out = np.zeros(6 * 65536, np.uint8)
        host_call(L, fn, us, out, [i * 65536 for i in range(6)], [65536] * 6, multi)
        assert out.tobytes() == t
        # second call: slots with gaps of 1..4000 bytes, caller bytes everywhere else
        rng = random.Random(3)
        caps = [65536, 30000, 65536, 65536 + 100]
        sel = [us[0], Unit("short", deflate(t[:30000]) + bytes(8), 30000), us[2], us[3]]
        offs, o = [], 5
        for c in caps:
            o += rng.randint(1, 4000)
            offs.append(o)
            o += c
        out = np.full(o + 777, FILL, np.uint8)
        ol, st = host_call(L, fn, sel, out, offs, caps, multi)
        assert list(st) == [0] * 4
        mask = np.zeros(out.size, bool)
        for a, c, u, n in zip(offs, caps, sel, ol):
            assert out[a:a + n].tobytes() == orc.inflate(u.data)[1]
            mask[a:a + c] = True
        assert (out[~mask] == FILL).all(), "the caller's bytes between slots were overwritten"
    finally:
        if multi:
            L.b200z_multi_shutdown()


def _child(path):
    """A fresh process for the once-per-process settings (B200Z_UPW / B200Z_SPEC_G): the same batch, B200Z_FAST=0."""
    us = batch(small=EMU)
    r = run_device(us)
    offs = np.cumsum([0] + [len(b) for b in r.bytes[:-1]]).astype(np.int64)
    np.savez(path, status=r.status, out_len=r.out_len, in_used=r.in_used, off=offs,
             bytes=np.frombuffer(b"".join(r.bytes) + b"\0", np.uint8))


if __name__ == "__main__":
    if EMU:
        sys.path.insert(0, os.path.join(HERE, "host_emul"))
        import build_emu_lib
        os.environ.setdefault("B200Z_LIB", build_emu_lib.build())
    _child(sys.argv[1])
