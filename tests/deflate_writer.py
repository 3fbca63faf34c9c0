"""A small RFC 1951 (DEFLATE) writer for tests: it writes exactly the blocks, headers and tokens it is given, so a test
can ask for streams zlib never writes (15-bit codes that are used, minimal and maximal dynamic headers, hundreds of blocks
in one member, incomplete or over-subscribed codes, forbidden symbols).  Nothing here chooses for the caller beyond the
defaults documented on each argument.

Tokens of a compressed block:
  int b                    literal byte b
  (length, dist)           a match, coded with the standard length / distance symbols and extra bits
  ("ll", sym, extra)       literal/length symbol `sym` as is (any 0..287), followed by `extra` in the symbol's extra bits
  ("d", sym, extra)        distance symbol `sym` as is (any 0..31), followed by `extra` in its extra bits
End-of-block (256) is appended unless eob=False."""
import struct
import zlib

# length symbols 257..285 and distance symbols 0..29: (base, extra bits)
LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [i // 2 for i in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LL = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_D = [5] * 32


def len_extra(sym):
    """Extra bits of literal/length symbol `sym` (0 for literals, end-of-block and the undefined 286 / 287)."""
    return LEN_EXTRA[sym - 257] if 257 <= sym <= 285 else 0


def dist_extra(sym):
    return DIST_EXTRA[sym] if sym < 30 else 0


def length_symbol(length):
    """(symbol, extra value) of a match length 3..258; 258 is symbol 285, never 284 + 31."""
    assert 3 <= length <= 258, length
    if length == 258:
        return 285, 0
    i = max(i for i in range(28) if LEN_BASE[i] <= length)
    return 257 + i, length - LEN_BASE[i]


def dist_symbol(dist):
    assert 1 <= dist <= 32768, dist
    i = max(i for i in range(30) if DIST_BASE[i] <= dist)
    return i, dist - DIST_BASE[i]


def canonical_codes(lengths):
    """RFC 1951 section 3.2.2 codes (MSB-first integers) for code lengths; 0 = unused.  Incomplete and over-subscribed
    length sets get codes too (the latter then collide or overflow their length), which is what a test of a decoder's
    rejection needs."""
    maxl = max(lengths, default=0)
    bl_count = [0] * (maxl + 2)
    for l in lengths:
        if l:
            bl_count[l] += 1
    code, next_code = 0, [0] * (maxl + 2)
    for bits in range(1, maxl + 1):
        code = (code + bl_count[bits - 1]) << 1
        next_code[bits] = code
    codes = [0] * len(lengths)
    for s, l in enumerate(lengths):
        if l:
            codes[s] = next_code[l] & ((1 << l) - 1)
            next_code[l] += 1
    return codes


def kraft(lengths):
    """Sum of 2^-len over the used codes, times 2^15: 32768 = complete, less = incomplete, more = over-subscribed."""
    return sum(1 << (15 - l) for l in lengths if l)


def limited_lengths(freqs, max_len=15):
    """Optimal code lengths of at most max_len bits for the symbols with freqs > 0 (package-merge).  One used symbol
    gets length 1; no used symbol gives all zeros."""
    used = [s for s, f in enumerate(freqs) if f > 0]
    lengths = [0] * len(freqs)
    if len(used) <= 1:
        for s in used:
            lengths[s] = 1
        return lengths
    assert len(used) <= 1 << max_len
    leaves = sorted(((freqs[s], (s,)) for s in used), key=lambda t: t[0])
    items = leaves
    for _ in range(max_len - 1):
        packages = [(items[i][0] + items[i + 1][0], items[i][1] + items[i + 1][1]) for i in range(0, len(items) - 1, 2)]
        items = sorted(leaves + packages, key=lambda t: t[0])
    for _, syms in items[:2 * len(used) - 2]:
        for s in syms:
            lengths[s] += 1
    return lengths


def _rev(code, n):
    return int(format(code, f"0{n}b")[::-1], 2) if n else 0


class BitWriter:
    """LSB-first bit packer into one Python integer."""

    def __init__(self):
        self.acc = 0
        self.n = 0

    def bits(self, value, n):
        assert 0 <= value < (1 << n) or n == 0 and value == 0, (value, n)
        self.acc |= value << self.n
        self.n += n

    def huff(self, code, length):  # Huffman codes go MSB first
        self.bits(_rev(code, length), length)

    def align(self, pad_value=0):
        """Pads to the next byte boundary (pad_value: the padding bits, for tests of readers that must skip them)."""
        k = -self.n & 7
        self.bits(pad_value & ((1 << k) - 1), k)

    def raw(self, data):
        assert self.n % 8 == 0
        self.acc |= int.from_bytes(data, "little") << self.n
        self.n += 8 * len(data)

    def getvalue(self):
        return self.acc.to_bytes((self.n + 7) // 8, "little")


def rle_code_lengths(lens, mode="greedy"):
    """Run-length codes of a code-length sequence as a list of (symbol, extra value).
    mode "greedy": 18 / 17 for zero runs (longest first), 16 for repeats of the previous length (a run may cross the
    literal/distance boundary, as RFC 1951 allows); "literal": one symbol 0..15 per length."""
    ops, i = [], 0
    while i < len(lens):
        v = lens[i]
        run = 1
        while i + run < len(lens) and lens[i + run] == v:
            run += 1
        if mode == "literal":
            ops.append((v, 0))
            i += 1
            continue
        if v == 0 and run >= 3:
            n = min(run, 138)
            ops.append((18, n - 11) if n >= 11 else (17, n - 3))
            i += n
            continue
        ops.append((v, 0))
        i += 1
        run -= 1
        while run >= 3:
            n = min(run, 6)
            ops.append((16, n - 3))
            i += n
            run -= n
    return ops


CL_EXTRA = {16: 2, 17: 3, 18: 7}


class Deflate:
    """One DEFLATE stream built block by block.  BFINAL is set only where a block asks for it."""

    def __init__(self):
        self.w = BitWriter()

    def stored(self, data, final=False, pad_value=0, nlen=None):
        """A stored block; pad_value fills the bits up to the byte boundary; nlen overrides the one's complement."""
        self.w.bits(int(final), 1)
        self.w.bits(0, 2)
        self.w.align(pad_value)
        self.w.bits(len(data), 16)
        self.w.bits((~len(data) & 0xFFFF) if nlen is None else nlen, 16)
        self.w.raw(data)
        return self

    def fixed(self, tokens, final=False, eob=True):
        self.w.bits(int(final), 1)
        self.w.bits(1, 2)
        self._tokens(tokens, FIXED_LL, FIXED_D, eob)
        return self

    def dynamic(self, tokens, final=False, eob=True, ll_lens=None, d_lens=None, max_bits=15, hlit=None, hdist=None,
                cl_lens=None, hclen=None, rle="greedy", fields=None):
        """A dynamic block.
        ll_lens / d_lens: code lengths (default: length-limited codes of max_bits from the tokens' symbol counts; no
          match -> one distance code of length 1, as zlib writes).  HLIT / HDIST default to the lists' lengths trimmed
          of trailing zeros (at least 257 / 1); larger values send the zeros.
        cl_lens: the 19 code-length-code lengths (default: 7-bit limited code of the symbols used); hclen: how many of
          them to send, in RFC order (default: up to the last non-zero, at least 4).
        rle: "greedy", "literal", or an explicit list of (symbol, extra value) for the concatenated length sequence.
        fields: raw (HLIT-257, HDIST-1, HCLEN-4) values to write instead of the computed ones (invalid headers)."""
        syms = self._symbols(tokens, eob)
        if ll_lens is None:
            f = [0] * 286
            for s, _ in syms:
                if s[0] == "ll":
                    f[s[1]] += 1
            ll_lens = limited_lengths(f, max_bits)
        if d_lens is None:
            f = [0] * 30
            for s, _ in syms:
                if s[0] == "d":
                    f[s[1]] += 1
            d_lens = limited_lengths(f, max_bits) if any(f) else [1]
        ll_lens, d_lens = list(ll_lens), list(d_lens)
        if hlit is None:
            hlit = max(257, max((i + 1 for i, l in enumerate(ll_lens) if l), default=0))
        if hdist is None:
            hdist = max(1, max((i + 1 for i, l in enumerate(d_lens) if l), default=0))
        ll_lens = (ll_lens + [0] * hlit)[:hlit]
        d_lens = (d_lens + [0] * hdist)[:hdist]
        seq = ll_lens + d_lens
        ops = rle if isinstance(rle, list) else rle_code_lengths(seq, rle)
        if cl_lens is None:
            f = [0] * 19
            for s, _ in ops:
                f[s] += 1
            cl_lens = limited_lengths(f, 7)
        if hclen is None:
            hclen = max(4, max((i + 1 for i, s in enumerate(CL_ORDER) if cl_lens[s]), default=0))
        w = self.w
        w.bits(int(final), 1)
        w.bits(2, 2)
        fh, fd, fc = fields if fields is not None else (hlit - 257, hdist - 1, hclen - 4)
        w.bits(fh, 5)
        w.bits(fd, 5)
        w.bits(fc, 4)
        for i in range(hclen):
            w.bits(cl_lens[CL_ORDER[i]], 3)
        cl_codes = canonical_codes(cl_lens)
        for s, extra in ops:
            w.huff(cl_codes[s], cl_lens[s])
            if s in CL_EXTRA:
                w.bits(extra, CL_EXTRA[s])
        self._emit(syms, ll_lens, d_lens)
        return self

    def bits(self, value, n):
        """Raw bits (e.g. a bare block header or a corrupt tail)."""
        self.w.bits(value, n)
        return self

    def getvalue(self):
        return self.w.getvalue()

    # ---- internals ----
    @staticmethod
    def _symbols(tokens, eob):
        """[(("ll"|"d", symbol), (extra value, extra bits)), ...] for a token list."""
        out = []
        for t in tokens:
            if isinstance(t, int):
                out.append((("ll", t), (0, 0)))
            elif t[0] == "ll":
                out.append((("ll", t[1]), (t[2], len_extra(t[1]))))
            elif t[0] == "d":
                out.append((("d", t[1]), (t[2], dist_extra(t[1]))))
            else:
                ls, le = length_symbol(t[0])
                ds, de = dist_symbol(t[1])
                out.append((("ll", ls), (le, len_extra(ls))))
                out.append((("d", ds), (de, dist_extra(ds))))
        if eob:
            out.append((("ll", 256), (0, 0)))
        return out

    def _tokens(self, tokens, ll_lens, d_lens, eob):
        self._emit(self._symbols(tokens, eob), ll_lens, d_lens)

    def _emit(self, syms, ll_lens, d_lens):
        llc, dc = canonical_codes(ll_lens), canonical_codes(d_lens)
        w = self.w
        for (kind, s), (ev, en) in syms:
            lens, codes = (ll_lens, llc) if kind == "ll" else (d_lens, dc)
            assert s < len(lens) and lens[s], f"{kind} symbol {s} has no code"
            w.huff(codes[s], lens[s])
            w.bits(ev, en)


def lz77(data, window=32768, max_len=258, min_len=3, max_chain=64):
    """Greedy LZ77 tokens of `data` (hash chains on 3-byte prefixes): the longest match among the last max_chain
    candidates, else a literal."""
    toks, heads, i, n = [], {}, 0, len(data)
    while i < n:
        best_len, best_dist = 0, 0
        if i + min_len <= n:
            key = data[i:i + 3]
            for j in reversed(heads.get(key, [])[-max_chain:]):
                if i - j > window:
                    break
                L = 0
                lim = min(max_len, n - i)
                while L < lim and data[j + L] == data[i + L]:
                    L += 1
                if L > best_len:
                    best_len, best_dist = L, i - j
                    if L == lim:
                        break
        step = best_len if best_len >= min_len else 1
        for k in range(i, min(i + step, n - 2)):
            heads.setdefault(data[k:k + 3], []).append(k)
        if best_len >= min_len:
            toks.append((best_len, best_dist))
        else:
            toks.append(data[i])
        i += step
    return toks


def expand(tokens):
    """The bytes a token list decodes to (raw symbols excluded)."""
    out = bytearray()
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
        else:
            L, d = t
            assert d <= len(out)
            for _ in range(L):
                out.append(out[-d])
    return bytes(out)


def bgzf_wrap(deflate_bytes, payload, isize=None, crc=None):
    """One BGZF block around a raw DEFLATE stream; CRC32 and ISIZE are those of the intended payload unless given.
    The header is the one bamutil.bgzf_block writes."""
    bsize = 12 + 6 + len(deflate_bytes) + 8 - 1
    assert bsize < 65536
    hdr = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize)
    return hdr + deflate_bytes + struct.pack("<II", (zlib.crc32(payload) if crc is None else crc) & 0xFFFFFFFF,
                                             len(payload) if isize is None else isize)
