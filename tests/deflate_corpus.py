"""Seeded, named DEFLATE conformance corpus built with deflate_writer: streams zlib never writes, aimed at the GPU
inflate's decoder (inflate_lane.cuh) and resolve kernel (inflate2.cuh).

valid_cases()    -> [(name, [(bgzf block, payload), ...])]   zlib decodes every block to its payload
invalid_cases()  -> [(name, bgzf block)]                       zlib rejects the block (stream error or ISIZE mismatch)

Not pinned (zlib and the reference's miniz_oxide are recalled to disagree, so no expectation is written down):
  * a literal/length or distance code with exactly one used symbol of length 2 or more (zlib rejects any incomplete
    code but a single 1-bit one; miniz_oxide accepts any one-symbol code);
  * a code-length code with exactly one used symbol (zlib rejects every incomplete code-length code);
  * length symbol 284 with extra bits 31, i.e. length 258 not written as symbol 285 (RFC 1951 leaves it undefined);
  * bytes after the final block of a BGZF member."""
import random

from deflate_writer import (CL_ORDER, DIST_BASE, DIST_EXTRA, LEN_BASE, LEN_EXTRA, Deflate, bgzf_wrap, expand, kraft,
                            limited_lengths, lz77, rle_code_lengths)

SEED = 20261020


def _match(ls, le, ds, de):
    """(length, dist) of length symbol ls with extra value le and distance symbol ds with extra de."""
    return LEN_BASE[ls - 257] + le, DIST_BASE[ds] + de


def _rand_bytes(rng, n, alphabet=None):
    if alphabet is None:
        return bytes(rng.randrange(256) for _ in range(n))
    return bytes(rng.choice(alphabet) for _ in range(n))


def _block(d, payload):
    return bgzf_wrap(d.getvalue(), payload), payload


def _one(d, tokens_or_payload):
    payload = tokens_or_payload if isinstance(tokens_or_payload, bytes) else expand(tokens_or_payload)
    return [_block(d, payload)]


def _assign(n_syms, lens_by_sym):
    lens = [0] * n_syms
    for s, l in lens_by_sym.items():
        lens[s] = l
    return lens


# ------------------------------------------------------------------ decoder: code lengths
def case_len15_codes(rng):
    """Complete literal/length and distance codes of lengths 1..15, 15 where the 15-bit symbols are used (literal 'z',
    length symbol 284, distance symbols 14 and 15)."""
    ll_syms = [ord(c) for c in "ACGTNacg"] + [257, 258, 265, 270, 285, 256, ord("z"), 284]
    ll = _assign(286, {s: min(i + 1, 15) for i, s in enumerate(ll_syms)})
    d_syms = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15]
    dl = _assign(30, {s: min(i + 1, 15) for i, s in enumerate(d_syms)})
    assert kraft(ll) == kraft(dl) == 1 << 15 and ll[256] == 14
    toks, out = [], 0
    for c in b"ACGTNacgz" * 3:
        toks.append(c)
        out += 1
    for i in range(400):
        r = rng.random()
        if r < 0.4 or out < 300:
            toks.append(ord(rng.choice("ACGTNacgz")))
            out += 1
            continue
        ls = rng.choice([257, 258, 265, 270, 285, 284])
        le = rng.randrange(1 << LEN_EXTRA[ls - 257]) if ls != 284 else rng.randrange(31)
        ds = rng.choice([s for s in d_syms if DIST_BASE[s] + (1 << DIST_EXTRA[s]) - 1 <= out] + [14, 15] * (out > 256))
        de = rng.randrange(1 << DIST_EXTRA[ds])
        L, D = _match(ls, le, ds, de)
        toks.append((L, D))
        out += L
    assert out <= 65536
    d = Deflate().dynamic(toks, final=True, ll_lens=ll, d_lens=dl)
    return _one(d, toks)


def case_sym48_every_phase(rng):
    """The 48-bit worst case of one decoder step (15-bit length code of symbol 284 + 5 extra bits, 15-bit distance code
    of symbol 29 + 13 extra bits), two back to back after a 1-bit literal: each repetition advances the bit position
    by 97 = 33 mod 64, so the pairs start at every bit phase of the reader's 64-bit window."""
    prefix = _rand_bytes(rng, 24577 + 100)
    ll_syms = [ord("x")] + [ord(c) for c in "abcdefghijkl"] + [256, 257, 284]
    ll = _assign(286, {s: min(i + 1, 15) for i, s in enumerate(ll_syms)})
    d_syms = list(range(15)) + [29]
    dl = _assign(30, {s: min(i + 1, 15) for i, s in enumerate(d_syms)})
    assert kraft(ll) == kraft(dl) == 1 << 15 and ll[284] == 15 and dl[29] == 15
    toks = []
    for rep in range(64):
        toks.append(ord("x"))
        for _ in range(2):
            toks.append(_match(284, rng.randrange(31), 29, rng.randrange(100)))
    d = Deflate().stored(prefix).dynamic(toks, final=True, ll_lens=ll, d_lens=dl)
    payload = expand(list(prefix) + toks)
    assert len(payload) <= 65536
    return [_block(d, payload)]


# ------------------------------------------------------------------ decoder: headers and block sequences
def case_header_min(rng):
    """The smallest dynamic header that can code a block: HLIT 257, HDIST 1 (length 0) and HCLEN 5 (HCLEN 4 sends only
    the lengths of 16, 17, 18 and 0, which leave end-of-block without a code: see invalid 'hclen4_no_eob').  All 256
    codes are 8 bits: literals 0..254 and end-of-block."""
    ll = [8] * 255 + [0, 8]
    toks = list(_rand_bytes(rng, 3000, bytes(range(255))))
    d = Deflate().dynamic(toks, final=True, ll_lens=ll, d_lens=[0], cl_lens=_cl({8: 1, 16: 2, 0: 2}), hclen=5)
    return _one(d, toks)


def _cl(m):
    return [m.get(s, 0) for s in range(19)]


def case_header_max(rng):
    """HLIT 286, HDIST 30, HCLEN 19: every literal/length and distance symbol has a code, and all 19 code-length-code
    lengths are sent (untrimmed trailing zeros)."""
    data = _rand_bytes(rng, 20000, b"ACGT" * 8 + bytes(range(256)))
    toks = lz77(data)
    ll = [8] * 226 + [9] * 60  # 226 * 2^7 + 60 * 2^6 = 2^15
    dl = [4, 4] + [5] * 28     # 2 * 2^11 + 28 * 2^10 = 2^15
    assert kraft(ll) == kraft(dl) == 1 << 15
    d = Deflate().dynamic(toks, final=True, ll_lens=ll, d_lens=dl, hlit=286, hdist=30, hclen=19)
    return _one(d, toks)


def case_literal_only_no_distance_code(rng):
    toks = list(_rand_bytes(rng, 5000, b"ACGTN"))
    d = Deflate().dynamic(toks, final=True, d_lens=[0], hdist=1)
    return _one(d, toks)


def case_single_distance_code(rng):
    """One distance code of length 1 (distance symbol 3: distance 4), the one incomplete code zlib accepts."""
    toks = list(b"ACGT")
    for _ in range(300):
        toks.append((rng.randrange(3, 259), 4) if rng.random() < 0.5 else rng.choice(b"ACGT"))
    d = Deflate().dynamic(toks, final=True, d_lens=[0, 0, 0, 1])
    return _one(d, toks)


def case_eob_and_one_literal(rng):
    toks = [ord("Q")] * 4000
    ll = _assign(286, {ord("Q"): 1, 256: 1})
    d = Deflate().dynamic(toks, final=True, ll_lens=ll, d_lens=[0])
    return _one(d, toks)


def _complete(lens, free):
    """Gives symbols of `free` the longest lengths that fill the code up to exactly 2^15 (a complete code)."""
    for s in free:
        rest = (1 << 15) - kraft(lens)
        if not rest:
            break
        lens[s] = 16 - rest.bit_length()  # the largest power of two <= rest
    assert kraft(lens) == 1 << 15
    return lens


def case_rle_longest_runs(rng):
    """Code-length run-length codes at their limits: 18 repeating 138 zeros, 17 repeating 10 zeros, 16 repeating 6 —
    one 16 runs across the literal/length / distance boundary — then the same codes again with every length sent as a
    literal 0..15."""
    lits = [0, 139] + list(range(150, 161))  # zeros 1..138 -> one 18 x 138; zeros 140..149 -> one 17 x 10
    ll = [0] * 286
    for s in lits + [256]:
        ll[s] = 5
    for s in range(280, 286):
        ll[s] = 6
    dl = [6, 6, 6] + [0] * 27  # lengths 6 from literal/length 280 to distance 2: 6, then 16 x 6 across the boundary
    _complete(ll, range(200, 250))
    _complete(dl, range(3, 30))
    ops = rle_code_lengths(ll + dl)
    assert (18, 127) in ops and (17, 7) in ops
    i, crossing = 0, False
    for s, e in ops:
        n = {16: 3 + e, 17: 3 + e, 18: 11 + e}.get(s, 1)
        crossing |= s == 16 and i < 286 < i + n
        i += n
    assert crossing
    toks = [rng.choice(lits) for _ in range(300)]
    out = 300
    for _ in range(150):
        L = rng.choice([115, 130, 131, 162, 163, 194, 195, 226, 227, 257, 258])  # length symbols 280..285
        ds = rng.choice([s for s in range(30) if dl[s] and DIST_BASE[s] <= out])
        D = min(DIST_BASE[ds] + rng.randrange(1 << DIST_EXTRA[ds]), out)
        toks += [(L, D), rng.choice(lits)]
        out += L + 1
    payload = expand(toks)
    d = Deflate().dynamic(toks, ll_lens=ll, d_lens=dl, hlit=286, hdist=30)
    d.dynamic(toks[:60], final=True, ll_lens=ll, d_lens=dl, hlit=286, hdist=30, rle="literal")
    return [_block(d, payload + _tail(payload, toks[:60]))]


def _tail(prev, toks):
    """Bytes of `toks` decoded after `prev` (matches may reach into prev)."""
    out = bytearray(prev)
    for t in toks:
        if isinstance(t, int):
            out.append(t)
        else:
            for _ in range(t[0]):
                out.append(out[-t[1]])
    return bytes(out[len(prev):])


def case_hundreds_of_blocks(rng):
    """400 DEFLATE blocks in one BGZF block, cycling stored / fixed / dynamic, matches reaching into earlier blocks."""
    d = Deflate()
    payload = b""
    for i in range(400):
        chunk = _rand_bytes(rng, rng.randrange(20, 120), b"ACGT")
        toks = _tokens_after(payload, chunk, rng)
        final = i == 399
        k = i % 3
        if k == 0:
            d.stored(chunk, final)
        elif k == 1:
            d.fixed(toks, final)
        else:
            d.dynamic(toks, final, max_bits=rng.choice([7, 9, 15]))
        payload += chunk
    return [_block(d, payload)]


def _tokens_after(history, chunk, rng):
    """Tokens for `chunk` given `history`: literals, and (half of the time) a match at the nearest earlier occurrence of
    the next 3 bytes within 4 KiB, extended as far as it goes (overlapping its own destination when it does)."""
    buf, h = history + chunk, len(history)
    toks, i = [], 0
    while i < len(chunk):
        p = h + i
        j = buf.rfind(chunk[i:i + 3], max(0, p - 4096), p + 2) if rng.random() < 0.5 and i + 3 <= len(chunk) else -1
        if j >= 0:
            L = 3
            while L < min(258, len(chunk) - i) and buf[j + L] == buf[p + L]:
                L += 1
            toks.append((L, p - j))
            i += L
        else:
            toks.append(chunk[i])
            i += 1
    assert _tail(history, toks) == chunk
    return toks


def case_mixed_and_empty_blocks(rng):
    """Stored, fixed and dynamic blocks in one member, with empty stored blocks between them and an empty final stored
    block (the shape of a sync flush followed by a finish)."""
    d = Deflate()
    payload = b""
    for i in range(12):
        chunk = _rand_bytes(rng, rng.randrange(1, 400), b"ACGTN\t:")
        toks = _tokens_after(payload, chunk, rng)
        [lambda: d.stored(chunk), lambda: d.fixed(toks), lambda: d.dynamic(toks)][i % 3]()
        if i % 2:
            d.stored(b"")
        payload += chunk
    d.stored(b"", final=True)
    return [_block(d, payload)]


def case_stored_pad_and_address(rng):
    """Stored blocks behind fixed blocks of 10 + 9 j bits (j 9-bit literals): the stored header is followed by every
    padding of 0..7 bits, and the stored payloads start at every address mod 8 of the stream, in all 64 pairs."""
    d = Deflate()
    payload = b""
    seen = set()
    blocks = 0
    while len(seen) < 64:
        j = rng.randrange(8)
        lits = [rng.randrange(144, 256) for _ in range(j)]
        d.fixed(lits)
        payload += bytes(lits)
        start = d.w.n + 3
        pad = -start & 7
        addr = ((start + pad) // 8 + 4) & 7
        n = rng.randrange(0, 24)
        data = _rand_bytes(rng, n)
        d.stored(data)
        payload += data
        seen.add((pad, addr))
        blocks += 1
        assert blocks < 5000
    d.fixed([], final=True)
    assert len(payload) <= 65536
    return [_block(d, payload)]


# ------------------------------------------------------------------ decoder: fixed blocks
def case_fixed_every_symbol(rng):
    """A fixed block that uses every length symbol 257..285 and every distance symbol 0..29, each at its smallest and
    largest extra value, behind a stored block of 32768 bytes so that distance 32768 reaches the stream's first byte."""
    prefix = _rand_bytes(rng, 32768, b"ACGTN")
    lens = []
    for ls in range(257, 286):
        for e in sorted({0, (1 << LEN_EXTRA[ls - 257]) - 1 - (ls == 284)}):
            lens.append(LEN_BASE[ls - 257] + e)
    dists = []
    for ds in range(30):
        for e in sorted({0, (1 << DIST_EXTRA[ds]) - 1}):
            dists.append(DIST_BASE[ds] + e)
    toks = []
    for i in range(max(len(lens), len(dists))):
        toks.append((lens[i % len(lens)], dists[i % len(dists)]))
        toks.append(rng.choice(b"ACGT"))
    d = Deflate().stored(prefix).fixed(toks, final=True)
    payload = prefix + _tail(prefix, toks)
    assert len(payload) <= 65536
    return [_block(d, payload)]


# ------------------------------------------------------------------ resolve kernel
def case_dist_1_to_16_every_length(rng):
    """Every distance 1..16 with every length 3..258 (the overlap-doubling path of resolve_copy), one BGZF block per
    distance, lengths in a shuffled order so that the matches start at every alignment."""
    out = []
    for dist in range(1, 17):
        lens = list(range(3, 259))
        rng.shuffle(lens)
        toks = list(_rand_bytes(rng, 16, b"ACGTN"))
        for L in lens:
            toks.append((L, dist))
            if rng.random() < 0.3:
                toks.append(rng.choice(b"acgt"))
        d = Deflate().dynamic(toks, final=True)
        out += _one(d, toks)
    return out


def case_dist_32768(rng):
    prefix = _rand_bytes(rng, 32768)
    toks = []
    for _ in range(120):
        toks.append((rng.randrange(3, 259), 32768))
        toks.append(rng.randrange(256))
    d = Deflate().stored(prefix).dynamic(toks, final=True)
    payload = prefix + _tail(prefix, toks)
    assert len(payload) <= 65536
    return [_block(d, payload)]


def case_match_chains(rng):
    """Chains of matches that each read the previous match's destination: 40 inside one 32-token batch of one
    super-window (3-byte matches at distance 3), and long chains with mixed lengths that cross batches and the resolve
    kernel's 1024-byte super-windows."""
    out = []
    toks = list(b"xyz") + [(3, 3)] * 40 + list(b"q")
    out += _one(Deflate().dynamic(toks, final=True), toks)
    toks = list(_rand_bytes(rng, 7))
    prev, pos = 7, 7
    while pos < 30000:
        L = rng.choice([3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 64, 100, 258])
        toks.append((L, prev))  # the source is the start of the previous match's destination
        prev = L
        pos += L
    out += _one(Deflate().dynamic(toks, final=True), toks)
    # short distances inside a chain (source overlaps both the previous match and the current one)
    toks = list(_rand_bytes(rng, 5))
    prev = 5
    for _ in range(3000):
        L = rng.randrange(3, 12)
        toks.append((L, rng.randrange(1, prev + 1)))
        prev = L
    out += _one(Deflate().fixed(toks, final=True), toks)
    return out


def case_densest_super_window(rng):
    """3-byte matches back to back through whole 1024-byte super-windows: 342 match starts in window 1 (the most any
    window can hold; the resolve kernel's list has room for kResList = 352), 341 in windows 2 and 3, distances mixing
    the chain (3) and random reaches back."""
    toks = list(_rand_bytes(rng, 1024, b"ACGT"))
    pos = 1024
    while pos < 4096:
        D = 3 if rng.random() < 0.5 else rng.randrange(1, pos + 1)
        toks.append((3, D))
        pos += 3
    d = Deflate().dynamic(toks, final=True)
    return _one(d, toks)


def case_match_ends_at_65536(rng):
    """A full 64 KiB block whose last token is a 258-byte match ending on byte 65536."""
    toks = list(_rand_bytes(rng, 300, b"ACGT"))
    pos = 300
    while pos < 65536 - 258 - 300:
        L = rng.randrange(3, 259)
        toks.append((L, rng.randrange(1, min(pos, 32768) + 1)))
        pos += L
        toks.append(rng.choice(b"ACGT"))
        pos += 1
    toks += list(_rand_bytes(rng, 65536 - 258 - pos, b"ACGT"))
    toks.append((258, rng.randrange(1, 32769)))
    d = Deflate().dynamic(toks, final=True)
    payload = expand(toks)
    assert len(payload) == 65536
    return [_block(d, payload)]


def case_isize_1_to_15(rng):
    out = []
    for n in range(1, 16):
        toks = [rng.choice(b"ACGT")]
        if n >= 4:
            toks.append((n - 1, 1))
        else:
            toks += [rng.choice(b"ACGT") for _ in range(n - 1)]
        d = Deflate().fixed(toks, final=True) if n % 2 else Deflate().dynamic(toks, final=True)
        out += _one(d, toks)
    return out


def case_all_output_residues(rng):
    """Blocks of 16 k + 1 bytes: consecutive blocks start at all 16 residues mod 16 of the output (the first / last
    chunk stores of the decoder and unaligned loads of the resolve kernel)."""
    out = []
    for i in range(17):
        n = 16 * rng.choice([0, 1, 2, 7, 60, 300, 1000, 4000]) + 1
        data = _rand_bytes(rng, n, b"ACGT")
        toks = _tokens_after(b"", data, rng)
        d = Deflate().dynamic(toks, final=True) if i % 2 else Deflate().fixed(toks, final=True)
        out += _one(d, toks)
    return out


VALID = [case_len15_codes, case_sym48_every_phase, case_header_min, case_header_max, case_literal_only_no_distance_code,
         case_single_distance_code, case_eob_and_one_literal, case_rle_longest_runs, case_hundreds_of_blocks,
         case_mixed_and_empty_blocks, case_stored_pad_and_address, case_fixed_every_symbol, case_dist_1_to_16_every_length,
         case_dist_32768, case_match_chains, case_densest_super_window, case_match_ends_at_65536, case_isize_1_to_15,
         case_all_output_residues]


def valid_cases():
    out = []
    for i, f in enumerate(VALID):
        out.append((f.__name__[5:], f(random.Random(SEED + i))))
    return out


# ------------------------------------------------------------------ invalid streams
def _inv(d, payload, **kw):
    return bgzf_wrap(d.getvalue(), payload, **kw)


def invalid_cases():
    """One BGZF block per case; CRC32 and ISIZE are those of the bytes the encoder meant, so only the DEFLATE stream
    itself (or ISIZE) can make a decoder reject it."""
    c = {}
    AC = _assign(286, {ord("A"): 2, ord("C"): 2, 256: 2})  # code 11 unassigned
    # incomplete literal/length code (3 of 4 two-bit codes): the repro of the bug, then the unassigned code read
    p = b"ACCAACCA"
    c["incomplete_ll_unused"] = _inv(Deflate().dynamic(list(p), final=True, ll_lens=AC, d_lens=[0]), p)
    d = Deflate().dynamic(list(b"ACCA"), final=True, eob=False, ll_lens=AC, d_lens=[0]).bits(0b11, 2).bits(0, 16)
    c["incomplete_ll_hit"] = _inv(d, b"ACCAC")
    # incomplete distance code: distances 1 (1 bit) and 2 (2 bits), code 11 unassigned
    ll = _assign(286, {ord("A"): 2, ord("C"): 2, 256: 2, 257: 2})
    dl = [1, 2]
    toks = list(b"AC") + [(3, 1), (3, 2)] + list(b"A")
    c["incomplete_dist_unused"] = _inv(Deflate().dynamic(toks, final=True, ll_lens=ll, d_lens=dl), expand(toks))
    d = Deflate().dynamic(list(b"AC"), final=True, eob=False, ll_lens=ll, d_lens=dl)
    d.bits(0b11, 2)  # length symbol 257 (code 11)
    d.bits(0b11, 2).bits(0, 16)  # the unassigned distance code 11
    c["incomplete_dist_hit"] = _inv(d, b"ACACA")
    # incomplete code-length code: 8 -> '0', 0 -> '10', '11' unassigned
    ll8 = [8] * 255 + [0, 8]
    ops = [(8, 0)] * 255 + [(0, 0), (8, 0), (0, 0)]
    cl = _cl({8: 1, 0: 2})
    p = bytes(range(40))
    c["incomplete_cl_unused"] = _inv(Deflate().dynamic(list(p), final=True, ll_lens=ll8, d_lens=[0], rle=ops, cl_lens=cl), p)
    d = Deflate().bits(1, 1).bits(2, 2).bits(0, 5).bits(0, 5).bits(1, 4)  # HLIT 257, HDIST 1, HCLEN 5
    for i in range(5):
        d.bits(cl[CL_ORDER[i]], 3)  # 16 17 18 0 8
    d.bits(0, 1).bits(0, 1).bits(0b11, 2).bits(0, 16)  # two 8s, then the unassigned code
    c["incomplete_cl_hit"] = _inv(d, p)
    # over-subscribed codes
    over_ll = _assign(286, {ord("A"): 1, ord("C"): 1, 256: 1})
    p = b"ACCA"
    c["oversubscribed_ll"] = _inv(Deflate().dynamic(list(p), final=True, ll_lens=over_ll, d_lens=[0]), p)
    toks = list(b"AC") + [(3, 1)]
    c["oversubscribed_dist"] = _inv(Deflate().dynamic(toks, final=True, ll_lens=ll, d_lens=[1, 1, 1]), expand(toks))
    p = bytes(range(40))
    c["oversubscribed_cl"] = _inv(Deflate().dynamic(list(p), final=True, ll_lens=ll8, d_lens=[0], rle=ops,
                                                    cl_lens=_cl({8: 1, 0: 1, 18: 1})), p)
    # header fields
    p = b"ACGT" * 10
    c["first_length_is_16"] = _inv(Deflate().dynamic(list(p), final=True, rle=[(16, 0)] + rle_code_lengths(_default_lens(p))), p)
    lens = _default_lens(p)
    ops = rle_code_lengths(lens)
    ops[-1] = (18, 127)  # the last run of zeros overruns HLIT + HDIST
    c["repeat_overruns_hlit_hdist"] = _inv(Deflate().dynamic(list(p), final=True, rle=ops, hlit=257, hdist=1), p)
    for hlit in (287, 288):
        c[f"hlit_field_{hlit - 257}"] = _inv(Deflate().dynamic(list(p), final=True, hlit=hlit), p)
    for hdist in (31, 32):
        c[f"hdist_{hdist}"] = _inv(Deflate().dynamic(list(p), final=True, hdist=hdist), p)
    c["eob_length_0"] = _inv(Deflate().dynamic(list(p), final=True, eob=False).bits(0, 16), p)
    # HCLEN 4: only 16, 17, 18 and 0 have lengths (17: '0', 18: '1'), so all 258 lengths are 0: no end-of-block
    c["hclen4_no_eob"] = _inv(Deflate().bits(1, 1).bits(2, 2).bits(0, 5).bits(0, 5).bits(0, 4)
                              .bits(0, 3).bits(1, 3).bits(1, 3).bits(0, 3)
                              .bits(1, 1).bits(127, 7).bits(1, 1).bits(109, 7).bits(0, 24), p)
    c["btype_3"] = _inv(Deflate().bits(1, 1).bits(3, 2).bits(0, 29), p)
    c["stored_nlen_mismatch"] = _inv(Deflate().stored(p, final=True, nlen=(~len(p) & 0xFFFF) ^ 0x10), p)
    # fixed-code symbols with no meaning
    c["fixed_ll_286"] = _inv(Deflate().fixed(list(b"ACG") + [("ll", 286, 0)] + list(b"T"), final=True), b"ACGTACG")
    c["fixed_ll_287"] = _inv(Deflate().fixed(list(b"ACG") + [("ll", 287, 0)] + list(b"T"), final=True), b"ACGTACG")
    c["fixed_d_30"] = _inv(Deflate().fixed(list(b"ACG") + [("ll", 257, 0), ("d", 30, 0)], final=True), b"ACGACG")
    c["fixed_d_31"] = _inv(Deflate().fixed(list(b"ACG") + [("ll", 257, 0), ("d", 31, 0)], final=True), b"ACGACG")
    # distances before the block start
    c["dist_at_position_0"] = _inv(Deflate().fixed([(3, 1)] + list(b"ACGT"), final=True), b"AAAACGT")
    c["dist_one_too_far"] = _inv(Deflate().dynamic(list(b"ACGTN") + [(4, 6)], final=True), b"ACGTNACGT")
    # size and truncation
    p = b"ACGTTGCA" * 20
    c["output_longer_than_isize_literal"] = _inv(Deflate().fixed(list(p), final=True), p, isize=len(p) - 1)
    toks = list(b"ACGTTGCA") + [(152, 8)]
    c["output_longer_than_isize_match"] = _inv(Deflate().dynamic(toks, final=True), expand(toks), isize=150)
    rng = random.Random(SEED - 1)
    data = _rand_bytes(rng, 4000)
    full = Deflate().dynamic(list(data), final=True, max_bits=15).getvalue()
    c["truncated_inside_a_symbol"] = bgzf_wrap(full[:len(full) // 2], data)
    return sorted(c.items())


def _default_lens(p):
    """Code lengths the writer picks for literal-only tokens `p` (HLIT 257, one 1-bit distance code)."""
    f = [0] * 286
    for b in p:
        f[b] += 1
    f[256] += 1
    return limited_lengths(f, 15)[:257] + [1]


def write_corpus(path, cases):
    """Writes the BGZF blocks of `cases` (valid_cases() form) to `path`; returns (n_blocks, concatenated payloads)."""
    blob, want, n = b"", b"", 0
    for _, blocks in cases:
        for blk, payload in blocks:
            blob += blk
            want += payload
            n += 1
    with open(path, "wb") as f:
        f.write(blob)
    return n, want
