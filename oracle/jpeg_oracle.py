"""numpy restatement of the baseline JPEG decoder of csrc/jpeg.cu, bit-exact with libjpeg-turbo's defaults (ISLOW IDCT,
fancy upsampling, jdcolor.c's YCbCr -> RGB), which is what PIL's Image.open(f).convert("RGB") and tf.image.decode_jpeg
produce.

Stages, in the order the library runs them:
  parse()              header parse: SOI, APPn, DQT, DHT, SOF0/1, DRI, SOS, EOI; the entropy data cut at RSTn into segments
  destuff()            the compact bit stream of one segment (a run of FF followed by 00 becomes one FF)
  decode_sequential()  Huffman decode of one segment from state (0, 0, 0)
  decode_subsequences() the same result from subsequences of L bits: speculative pass, checkpoints, repair (Weissenberger &
                       Schmidt, ICPP 2018)
  dc_prefix()          DC values from DC differences, per component, reset at every segment
  idct_islow()         dequantisation + jidctint.c with jdmaster.c's range-limit table
  upsample / colour    jdsample.c h2v1 / h2v2 fancy upsampling, jdcolor.c ycc_rgb_convert

Corrupt entropy data never raises: an invalid Huffman code decodes as symbol 0 and consumes 16 bits, bits past the end of a
segment read as 0, a run past k = 63 writes coefficient 63 (jpeg_natural_order's padding), blocks past a segment's MCU count
are dropped and missing ones stay zero (their DC difference is 0).
"""
from __future__ import annotations

import re

import numpy as np


class JpegError(ValueError):
    pass


# Entropy-coded bytes of one restart segment at most: its bit positions stay below 2^31 - 8192 (int32 on the device)
MAX_SEGMENT_BYTES = (1 << 28) - 1024


ZIGZAG = np.array([
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
    28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
    47, 55, 62, 63], np.int64)       # jpeg_natural_order: zigzag index -> natural (row-major) index


# ---------------------------------------------------------------------------------------------------------------------
# header parse
# ---------------------------------------------------------------------------------------------------------------------
def _huff_table(counts, symbols, is_dc):
    """(maxcode[17], valoffset[17], huffval) of jdhuff.c jpeg_make_d_derived_tbl; JpegError for an invalid table."""
    if sum(counts) > 256:
        raise JpegError("bad Huffman table: more than 256 symbols")
    maxcode = [-1] * 18
    valoff = [0] * 18
    code, p = 0, 0
    for l in range(1, 17):
        n = counts[l - 1]
        if n:
            valoff[l] = p - code
            code += n
            p += n
            if code >= (1 << l):                 # no code may be all ones (jpeg_make_d_derived_tbl)
                raise JpegError("bad Huffman table: code lengths overflow")
            maxcode[l] = code - 1
        code <<= 1
    maxcode[17] = 0x7FFFFFFF
    if is_dc and any(s > 15 for s in symbols):
        raise JpegError("bad Huffman table: DC symbol above 15")
    return maxcode, valoff, list(symbols)


def parse(data: bytes) -> dict:
    """Header parse and the cut of the entropy data into restart segments; JpegError with the reason for any file outside
    the accepted subset (baseline/extended sequential Huffman, 8-bit, 1 or 3 components, luma (1,1) / (2,1) / (2,2) with
    chroma (1,1), one interleaved scan)."""
    d = bytes(data)
    n = len(d)
    if n < 4 or d[0] != 0xFF or d[1] != 0xD8:
        raise JpegError("not a JPEG file (no SOI)")
    p = 2
    q = {}
    huff = {}
    frame = None
    jfif = adobe = False
    transform = -1
    ri = 0
    while True:
        if p >= n:
            raise JpegError("truncated before the scan")
        if d[p] != 0xFF:
            raise JpegError("expected a marker")
        while p < n and d[p] == 0xFF:
            p += 1
        if p >= n:
            raise JpegError("truncated before the scan")
        m = d[p]
        p += 1
        if m == 0xD9:
            raise JpegError("EOI before any scan")
        if m in (0xD8, 0x01) or 0xD0 <= m <= 0xD7:
            raise JpegError(f"unexpected marker 0x{m:02X}")
        if p + 2 > n:
            raise JpegError("truncated before the scan")
        ln = (d[p] << 8) | d[p + 1]
        if ln < 2 or p + ln > n:
            raise JpegError("truncated before the scan")
        seg = d[p + 2:p + ln]
        p += ln
        if m == 0xE0:
            if len(seg) >= 14 and seg[:5] == b"JFIF\0":
                jfif = True
        elif m == 0xEE:
            if len(seg) >= 12 and seg[:5] == b"Adobe":
                adobe, transform = True, seg[11]
        elif m == 0xDB:
            i = 0
            while i < len(seg):
                pq, tq = seg[i] >> 4, seg[i] & 15
                if pq > 1 or tq > 3:
                    raise JpegError("bad quantisation table")
                sz = 64 * (pq + 1)
                if i + 1 + sz > len(seg):
                    raise JpegError("truncated quantisation table")
                raw = np.frombuffer(seg[i + 1:i + 1 + sz], np.uint8 if pq == 0 else ">u2").astype(np.int64)
                tab = np.zeros(64, np.int64)
                tab[ZIGZAG] = raw
                q[tq] = tab
                i += 1 + sz
        elif m == 0xC4:
            i = 0
            while i < len(seg):
                if i + 17 > len(seg):
                    raise JpegError("truncated Huffman table")
                tc, th = seg[i] >> 4, seg[i] & 15
                if tc > 1 or th > 3:
                    raise JpegError("bad Huffman table class or id")
                counts = list(seg[i + 1:i + 17])
                tot = sum(counts)
                if i + 17 + tot > len(seg):
                    raise JpegError("truncated Huffman table")
                huff[(tc, th)] = _huff_table(counts, list(seg[i + 17:i + 17 + tot]), tc == 0)
                i += 17 + tot
        elif m in (0xC0, 0xC1):
            if frame is not None:
                raise JpegError("more than one frame header")
            if len(seg) < 6:
                raise JpegError("truncated frame header")
            if seg[0] != 8:
                raise JpegError(f"{seg[0]}-bit precision (only 8-bit is supported)")
            h, w, nc = (seg[1] << 8) | seg[2], (seg[3] << 8) | seg[4], seg[5]
            if nc not in (1, 3):
                raise JpegError(f"{nc} components (only 1 or 3 are supported)")
            if len(seg) < 6 + 3 * nc:
                raise JpegError("truncated frame header")
            comps = [(seg[6 + 3 * c], seg[7 + 3 * c] >> 4, seg[7 + 3 * c] & 15, seg[8 + 3 * c]) for c in range(nc)]
            if h == 0:
                raise JpegError("height defined by DNL (not supported)")
            if w == 0:
                raise JpegError("zero width")
            frame = (h, w, comps)
        elif m == 0xC2 or m == 0xC6 or m == 0xCA or m == 0xCE:
            raise JpegError("progressive JPEG (not supported)")
        elif m == 0xC3 or m == 0xC7 or m == 0xCB or m == 0xCF:
            raise JpegError("lossless JPEG (not supported)")
        elif m in (0xC5, 0xC9, 0xCC, 0xCD):
            raise JpegError("arithmetic-coded or hierarchical JPEG (not supported)")
        elif m == 0xDD:
            if len(seg) < 2:
                raise JpegError("truncated DRI")
            ri = (seg[0] << 8) | seg[1]
        elif m == 0xDC:
            raise JpegError("DNL marker (not supported)")
        elif m == 0xDA:
            if frame is None:
                raise JpegError("scan before the frame header")
            break
        # other APPn, COM and unknown markers are skipped by their length
    h, w, comps = frame
    ns = seg[0] if seg else 0
    if len(seg) < 1 + 2 * ns + 3:
        raise JpegError("truncated scan header")
    if ns != len(comps):
        raise JpegError("scan does not hold every component (several scans are not supported)")
    sc = [(seg[1 + 2 * i], seg[2 + 2 * i] >> 4, seg[2 + 2 * i] & 15) for i in range(ns)]
    if [c[0] for c in sc] != [c[0] for c in comps]:
        raise JpegError("scan components are not in frame order")
    ss, se, ahal = seg[1 + 2 * ns], seg[2 + 2 * ns], seg[3 + 2 * ns]
    if ss != 0 or se != 63 or ahal != 0:
        raise JpegError("not a sequential scan")
    # sampling
    if len(comps) == 1:
        hs, vs = [1], [1]
    else:
        hs, vs = [c[1] for c in comps], [c[2] for c in comps]
        if (hs[0], vs[0]) not in ((1, 1), (2, 1), (2, 2)) or any((hs[c], vs[c]) != (1, 1) for c in (1, 2)):
            raise JpegError("unsupported sampling factors " + ",".join(f"{c[1]}x{c[2]}" for c in comps))
    for ci, (_, td, ta) in enumerate(sc):
        if (0, td) not in huff or (1, ta) not in huff:
            raise JpegError(f"component {ci}: Huffman table referenced but never defined")
        if comps[ci][3] not in q:
            raise JpegError(f"component {ci}: quantisation table referenced but never defined")
    # colour space: libjpeg's default_decompress_parms
    if len(comps) == 1:
        space = "gray"
    elif jfif:
        space = "ycc"
    elif adobe:
        space = "rgb" if transform == 0 else "ycc"
    elif [c[0] for c in comps] == [82, 71, 66]:
        space = "rgb"
    else:
        space = "ycc"
    # entropy data: segments at RSTn, up to EOI.  Inside the data a run of FF followed by 00 is one FF byte (jdhuff.c
    # jpeg_fill_bit_buffer skips fill bytes); a run of FF followed by anything else is a marker.
    segs = []
    start = p
    while True:
        f = d.find(b"\xFF", p)
        if f < 0 or f + 1 >= n:
            raise JpegError("truncated inside the entropy-coded data (no EOI)")
        r = f
        while r + 1 < n and d[r + 1] == 0xFF:
            r += 1
        if r + 1 >= n:
            raise JpegError("truncated inside the entropy-coded data (no EOI)")
        mk = d[r + 1]
        if mk == 0x00:
            p = r + 2
            continue
        if f - start > MAX_SEGMENT_BYTES:
            raise JpegError(f"a restart segment holds {f - start} bytes of entropy-coded data (at most {MAX_SEGMENT_BYTES})")
        segs.append((start, f))
        p = r + 2
        if 0xD0 <= mk <= 0xD7:
            start = p
            continue
        if mk == 0xD9:
            break
        if mk == 0xDC:
            raise JpegError("DNL marker (not supported)")
        if mk == 0xDA or 0xC0 <= mk <= 0xCF or mk == 0xDB or mk == 0xDD:
            raise JpegError("several scans (not supported)")
        raise JpegError(f"unexpected marker 0x{mk:02X} after the scan")
    hmax, vmax = max(hs), max(vs)
    mcux, mcuy = -(-w // (8 * hmax)), -(-h // (8 * vmax))
    blocks = []                     # per block of an MCU: component, x and y within the component's MCU cell
    for c in range(len(comps)):
        for by in range(vs[c]):
            for bx in range(hs[c]):
                blocks.append((c, bx, by))
    nmcu = mcux * mcuy
    if ri == 0:
        ri = nmcu
    nseg = -(-nmcu // ri)
    segs = (segs + [(start, start)] * nseg)[:nseg]         # extra RSTn segments are dropped, missing ones are empty
    return dict(height=h, width=w, ncomp=len(comps), space=space, hs=hs, vs=vs, hmax=hmax, vmax=vmax, mcux=mcux,
                mcuy=mcuy, blocks=blocks, restart=ri, segments=segs, data=d,
                quant=[q[c[3]] for c in comps],
                dc=[huff[(0, c[1])] for c in sc], ac=[huff[(1, c[2])] for c in sc])


def info(data: bytes) -> tuple[int, int, int]:
    j = parse(data)
    return j["height"], j["width"], j["ncomp"]


# ---------------------------------------------------------------------------------------------------------------------
# entropy decode
# ---------------------------------------------------------------------------------------------------------------------
def destuff(d: bytes, a: int, b: int) -> bytes:
    return re.sub(rb"\xFF+\x00", b"\xFF", d[a:b])


class _Bits:
    def __init__(self, buf: bytes):
        self.v = int.from_bytes(buf, "big") if buf else 0
        self.n = 8 * len(buf)

    def peek(self, pos: int, cnt: int) -> int:
        """cnt bits at pos, MSB first; bits past the end are 0."""
        if pos >= self.n:
            return 0
        end = pos + cnt
        if end <= self.n:
            return (self.v >> (self.n - end)) & ((1 << cnt) - 1)
        return ((self.v & ((1 << (self.n - pos)) - 1)) << (end - self.n))


def _decode_huff(bits, pos, tab):
    """(symbol, code length); an invalid code is symbol 0 of length 16."""
    maxcode, valoff, vals = tab
    look = bits.peek(pos, 16)
    for l in range(1, 17):
        code = look >> (16 - l)
        if code <= maxcode[l]:
            return vals[code + valoff[l]], l
    return 0, 16


def _extend(r, s):
    return r - (1 << s) + 1 if s and r < (1 << (s - 1)) else r


def step(j, bits, st):
    """One symbol from state (pos, u, k): returns the next state, the coefficient (natural index, value) it writes or None,
    and whether it completed a block.  DC values are differences."""
    pos, u, k = st
    c = j["blocks"][u][0]
    if k == 0:
        s, l = _decode_huff(bits, pos, j["dc"][c])
        r = bits.peek(pos + l, s) if s else 0
        pos += l + s
        out = (0, _extend(r, s))
        k = 1
    else:
        rs, l = _decode_huff(bits, pos, j["ac"][c])
        r, s = rs >> 4, rs & 15
        out = None
        if s:
            k += r
            v = bits.peek(pos + l, s)
            out = (int(ZIGZAG[min(k, 63)]), _extend(v, s))
            k += 1
        elif r == 15:
            k += 16
        else:
            k = 64
        pos += l + s
    done = k >= 64
    if done:
        u = (u + 1) % len(j["blocks"])
        k = 0
    return (pos, u, k), out, done


def decode_sequential(j, seg_index):
    """int64 [nblocks, 64] coefficients of one segment (DC as differences), decoded from (0, 0, 0)."""
    a, b = j["segments"][seg_index]
    bits = _Bits(destuff(j["data"], a, b))
    nb = _seg_blocks(j, seg_index)
    coef = np.zeros((nb, 64), np.int64)
    st, blk = (0, 0, 0), 0
    while st[0] < bits.n and blk < nb:
        st, out, done = step(j, bits, st)
        if out is not None:
            coef[blk, out[0]] = out[1]
        blk += done
    return coef


def _seg_blocks(j, s):
    nmcu = j["mcux"] * j["mcuy"]
    return (min(nmcu, (s + 1) * j["restart"]) - s * j["restart"]) * len(j["blocks"])


def decode_subsequences(j, seg_index, L, stats=None):
    """decode_sequential()'s result through subsequences of L bits (L a multiple of 32): the exact start state of every
    subsequence is the fixed point S_0 = (0, 0, 0), S_{i+1} = exit(D(S_i)).  A speculative pass decodes each subsequence
    from its first bit with u = k = 0 and keeps a checkpoint at the first symbol boundary at or past every 32-bit word; the
    repair re-decodes subsequence i from the exit of i - 1 when that differs from the start it used, until a checkpoint
    agrees (from there on the speculative result holds) or the subsequence ends."""
    assert L % 32 == 0
    a, b = j["segments"][seg_index]
    bits = _Bits(destuff(j["data"], a, b))
    nbits = bits.n
    nsub = -(-nbits // L)

    def run(i, st, checks=None):
        """Decodes subsequence i from st; returns (exit, blocks, checkpoints {word boundary: (state, blocks)}, symbols).
        With checks, stops at the first checkpoint that agrees and completes the result from it."""
        end = min((i + 1) * L, nbits)
        cps, blk, nsym = {}, 0, 0
        nextb = (st[0] // 32 + 1) * 32
        while st[0] < end:
            st, _, done = step(j, bits, st)
            blk += done
            nsym += 1
            while nextb <= st[0] and nextb <= (i + 1) * L:
                if checks is not None and nextb in checks and checks[nextb][0] == st:
                    ex, ex_blk, _ = spec[i]
                    return ex, blk + ex_blk - checks[nextb][1], cps, nsym
                cps[nextb] = (st, blk)
                nextb += 32
        return st, blk, cps, nsym

    spec = []
    for i in range(nsub):
        ex, blk, cps, _ = run(i, (i * L, 0, 0))
        spec.append((ex, blk, cps))
    starts, counts = [], []
    st = (0, 0, 0)
    for i in range(nsub):
        starts.append(st)
        if st == (i * L, 0, 0):
            ex, blk = spec[i][0], spec[i][1]
        else:
            ex, blk, _, nsym = run(i, st, spec[i][2])
            if stats is not None:
                stats["subsequences"] = stats.get("subsequences", 0) + 1
                stats["symbols"] = stats.get("symbols", 0) + nsym
        counts.append(blk)
        st = ex
    # the write pass: every subsequence from its agreed start, blocks placed by the exclusive prefix of the counts
    nb = _seg_blocks(j, seg_index)
    coef = np.zeros((nb, 64), np.int64)
    base = 0
    for i in range(nsub):
        st, blk = starts[i], base
        end = min((i + 1) * L, nbits)
        while st[0] < end:
            st, out, done = step(j, bits, st)
            if out is not None and blk < nb:
                coef[blk, out[0]] = out[1]
            blk += done
        base += counts[i]
    return coef


def dc_prefix(j, coef):
    """DC differences -> DC values in place, per component, restarting at 0 (int32 wrap-around, int16 store as libjpeg)."""
    bpm = len(j["blocks"])
    last = [0] * j["ncomp"]
    for bi in range(coef.shape[0]):
        c = j["blocks"][bi % bpm][0]
        last[c] = (last[c] + int(coef[bi, 0]) + 2 ** 31) % 2 ** 32 - 2 ** 31
        coef[bi, 0] = (last[c] + 2 ** 15) % 2 ** 16 - 2 ** 15
    return coef


def coefficients(j, L=None):
    """int64 [mcuy * mcux * blocks per MCU, 64] dequantisation-ready coefficients of the whole image, in MCU order."""
    parts = []
    for s in range(len(j["segments"])):
        c = decode_sequential(j, s) if L is None else decode_subsequences(j, s, L)
        parts.append(dc_prefix(j, c))
    return np.concatenate(parts, 0) if parts else np.zeros((0, 64), np.int64)


# ---------------------------------------------------------------------------------------------------------------------
# IDCT, upsampling, colour
# ---------------------------------------------------------------------------------------------------------------------
def range_limit(v):
    """jdmaster.c's post-IDCT table indexed by (v & RANGE_MASK), v the descaled IDCT output before the +128 centre."""
    x = np.asarray(v, np.int64) & 1023
    return np.where(x < 128, x + 128, np.where(x < 512, 255, np.where(x < 896, 0, x - 896))).astype(np.uint8)


def _idct_1d(s0, s1, s2, s3, s4, s5, s6, s7):
    z1 = (s2 + s6) * 4433
    tmp2 = z1 + s6 * -15137
    tmp3 = z1 + s2 * 6270
    tmp0 = (s0 + s4) << 13
    tmp1 = (s0 - s4) << 13
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    t0, t1, t2, t3 = s7, s5, s3, s1
    z1, z2, z3, z4 = t0 + t3, t1 + t2, t0 + t2, t1 + t3
    z5 = (z3 + z4) * 9633
    t0, t1, t2, t3 = t0 * 2446, t1 * 16819, t2 * 25172, t3 * 12299
    z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069 + z5, z4 * -3196 + z5
    t0 += z1 + z3
    t1 += z2 + z4
    t2 += z2 + z3
    t3 += z1 + z4
    return [t10 + t3, t11 + t2, t12 + t1, t13 + t0, t13 - t0, t12 - t1, t11 - t2, t10 - t3]


def idct_islow(coef, qtab):
    """[n, 64] natural-order coefficients, [64] quantisation table -> [n, 8, 8] uint8 (jidctint.c jpeg_idct_islow)."""
    x = (np.asarray(coef, np.int64) * np.asarray(qtab, np.int64)).reshape(-1, 8, 8)
    cols = _idct_1d(*[x[:, r, :] for r in range(8)])                        # pass 1 on columns
    ws = np.stack([(c + (1 << 10)) >> 11 for c in cols], 1)                 # DESCALE(, CONST_BITS - PASS1_BITS)
    rows = _idct_1d(*[ws[:, :, c] for c in range(8)])                       # pass 2 on rows
    return np.stack([range_limit((r + (1 << 17)) >> 18) for r in rows], 2)  # DESCALE(, CONST_BITS + PASS1_BITS + 3)


def planes(j, coef):
    """Component planes [c] of (mcuy * v * 8, mcux * h * 8) uint8, whole blocks including the MCU padding."""
    out = []
    bpm = len(j["blocks"])
    for c in range(j["ncomp"]):
        h, v = j["hs"][c], j["vs"][c]
        pl = np.zeros((j["mcuy"] * v * 8, j["mcux"] * h * 8), np.uint8)
        us = [u for u, b in enumerate(j["blocks"]) if b[0] == c]
        for u in us:
            _, bx, by = j["blocks"][u]
            px = idct_islow(coef[u::bpm], j["quant"][c]).reshape(j["mcuy"], j["mcux"], 8, 8)
            for my in range(j["mcuy"]):
                for mx in range(j["mcux"]):
                    y0, x0 = (my * v + by) * 8, (mx * h + bx) * 8
                    pl[y0:y0 + 8, x0:x0 + 8] = px[my, mx]
        out.append(pl)
    return out


def upsample(j, plane, c):
    """One chroma plane to the image's size: jdsample.c h2v1 / h2v2 fancy upsampling (plain replication when the
    component is at most 2 samples wide, as jinit_upsampler chooses), int32 arithmetic."""
    H, W = j["height"], j["width"]
    he, ve = j["hmax"] // j["hs"][c], j["vmax"] // j["vs"][c]
    if he == 1 and ve == 1:
        return plane[:H, :W]
    dw = -(-W * j["hs"][c] // j["hmax"])
    dh = -(-H * j["vs"][c] // j["vmax"])
    p = plane.astype(np.int64)
    x = np.arange(W)
    i = x >> 1
    if dw <= 2:
        return plane[(np.arange(H) // ve)[:, None], i[None, :]]
    even = (x & 1) == 0
    nb = np.where(even, i - 1, i + 1)                        # the other column of the pair: never out of [0, dw) here
    first, last = even & (i == 0), ~even & (i == dw - 1)
    if ve == 1:
        v = p[:H]
        near, far = v[:, i], v[:, np.clip(nb, 0, dw - 1)]
        out = np.where(even, (near * 3 + far + 1) >> 2, (near * 3 + far + 2) >> 2)
        out = np.where(first | last, near, out)
        return out.astype(np.uint8)
    y = np.arange(H)
    r = y >> 1
    r2 = np.clip(np.where((y & 1) == 0, r - 1, r + 1), 0, dh - 1)           # context rows replicate the first / last row
    cs = p[r][:, :dw + 1] * 3 + p[r2][:, :dw + 1]
    this, other = cs[:, i], cs[:, np.clip(nb, 0, dw - 1)]
    out = np.where(even, (this * 3 + other + 8) >> 4, (this * 3 + other + 7) >> 4)
    out = np.where(first, (this * 4 + 8) >> 4, np.where(last, (this * 4 + 7) >> 4, out))
    return out.astype(np.uint8)


def ycc_to_rgb(y, cb, cr):
    """jdcolor.c ycc_rgb_convert with its fixed-point tables (SCALEBITS 16)."""
    y, cb, cr = (np.asarray(a, np.int64) for a in (y, cb, cr))
    half = 1 << 15
    xb, xr = cb - 128, cr - 128
    r = y + ((91881 * xr + half) >> 16)
    g = y + ((-22554 * xb + half - 46802 * xr) >> 16)
    b = y + ((116130 * xb + half) >> 16)
    return np.stack([np.clip(a, 0, 255) for a in (r, g, b)], -1).astype(np.uint8)


def pixels_from_coefficients(j, coef):
    pl = planes(j, coef)
    H, W = j["height"], j["width"]
    if j["ncomp"] == 1:
        g = pl[0][:H, :W]
        return np.stack([g, g, g], -1)
    y, cb, cr = pl[0][:H, :W], upsample(j, pl[1], 1), upsample(j, pl[2], 2)
    if j["space"] == "rgb":
        return np.stack([y, cb, cr], -1)
    return ycc_to_rgb(y, cb, cr)


def decode(data: bytes, L=None) -> np.ndarray:
    """uint8 (h, w, 3) RGB, what np.asarray(Image.open(f).convert("RGB")) gives for an accepted file."""
    j = parse(data)
    return pixels_from_coefficients(j, coefficients(j, L))
