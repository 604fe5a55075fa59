"""Reference of the read-pair ingest (tadpole_b200/csrc/pairs.cu, DESIGN S0f): the checker the pairs tests compare the GPU
with.  bin_pairs_text restates the spec one line at a time, errors included; bin_pairs_np is a vectorised restatement
(pandas + numpy) for genome-sized, well-formed inputs, held equal to the line-by-line one by the CPU tests.
write_pairs writes seeded synthetic pair files in the three layouts: distance-decaying cis pairs, trans pairs, unplaced
names, and (quirks=True) the comment, header, CRLF, blank, mixed-separator, swapped, duplicate and edge-position lines."""
from __future__ import annotations

import re

import numpy as np

# 0-based (chrom1, pos1, chrom2, pos2) columns of the three layouts
LAYOUTS = {"4dn": (1, 2, 3, 4), "hicpro": (1, 2, 4, 5), "juicer": (1, 2, 5, 6)}
FIELDS = {"4dn": 7, "hicpro": 8, "juicer": 10}      # fields per line of write_pairs
WINDOW = 64 << 20                        # the library's default device window
UNPLACED = ["chrM", "!", "chr1_KI270706v1_random"]


class PairsError(ValueError):
    """An error of the spec: the file and line (1-based; 0 for a whole-file error) and the kind."""

    def __init__(self, path, line, kind):
        super().__init__(f"'{path}' line {line}: {kind}" if line else f"'{path}': {kind}")
        self.path, self.line, self.kind = path, line, kind


def n_bins(chromsizes, binsize):
    return [-(-int(ln) // int(binsize)) for _, ln in chromsizes]


def _cells_out(cells, chromsizes):
    out = []
    for c in range(len(chromsizes)):
        kept = sorted(cells[c].items())
        out.append((np.array([k[0] for k, _ in kept], dtype=np.int64), np.array([k[1] for k, _ in kept], dtype=np.int64),
                    np.array([float(v) for _, v in kept], dtype=np.float64)))
    return out


def bin_pairs_text(paths, chromsizes, binsize, columns=(1, 2, 3, 4), index_base=1, window=WINDOW):
    """tp_genome_ingest_pairs_file, one line at a time.  chromsizes: [(name, length in bp)].  Returns
    ([(I, J, count) of each chromosome, sorted by (I, J)], dict(lines, cis, trans, unplaced)); raises PairsError with
    the first file's lowest bad line (or the whole-file error) in path order."""
    index = {nm.encode(): c for c, (nm, _) in enumerate(chromsizes)}
    lens = [int(ln) for _, ln in chromsizes]
    c1col, p1col, c2col, p2col = columns
    maxcol = max(columns)
    cells = [dict() for _ in chromsizes]
    counts = dict(lines=0, cis=0, trans=0, unplaced=0)
    for path in paths:
        with open(path, "rb") as fh:
            data = fh.read()
        if data[:2] == b"\x1f\x8b":
            raise PairsError(path, 0, "compressed input is not read")
        before = counts["lines"]
        pieces = data.split(b"\n")
        ends = [True] * (len(pieces) - 1) + [False]
        if pieces and pieces[-1] == b"":
            pieces, ends = pieces[:-1], ends[:-1]
        for n, (raw, nl) in enumerate(zip(pieces, ends), 1):
            if len(raw) + nl > window:
                raise PairsError(path, n, "longer than the device window")
            line = raw[:-1] if raw.endswith(b"\r") else raw
            if line.strip(b" \t\r") == b"" or line[:1] == b"#":
                continue
            fields = [f for f in re.split(rb"[ \t]+", line) if f]
            if len(fields) <= maxcol:
                raise PairsError(path, n, "fewer fields than the columns need")
            pos = []
            for col in (p1col, p2col):
                if not re.fullmatch(rb"[0-9]{1,18}", fields[col]):
                    raise PairsError(path, n, "a position is not 1 to 18 digits")
                pos.append(int(fields[col]))
            chroms = [index.get(fields[c1col], -1), index.get(fields[c2col], -1)]
            for c, p in zip(chroms, pos):
                if c >= 0 and not index_base <= p <= lens[c] - 1 + index_base:
                    raise PairsError(path, n, "a position lies outside its chromosome")
            counts["lines"] += 1
            if chroms[0] < 0 or chroms[1] < 0:
                counts["unplaced"] += 1
            elif chroms[0] != chroms[1]:
                counts["trans"] += 1
            else:
                counts["cis"] += 1
                b1, b2 = ((p - index_base) // binsize for p in pos)
                key = (min(b1, b2), max(b1, b2))
                cells[chroms[0]][key] = cells[chroms[0]].get(key, 0) + 1
        if counts["lines"] == before:
            raise PairsError(path, 0, "holds no pair lines")
    return _cells_out(cells, chromsizes), counts


def bin_pairs_np(paths, chromsizes, binsize, columns=(1, 2, 3, 4), index_base=1):
    """bin_pairs_text for genome-sized, well-formed files (pandas reads them; a '#' only starts header lines): the same
    result, without the error checks."""
    import pandas as pd
    names = [nm for nm, _ in chromsizes]
    lens = np.array([int(ln) for _, ln in chromsizes], dtype=np.int64)
    nb = np.array(n_bins(chromsizes, binsize), dtype=np.int64)
    starts = np.concatenate(([0], np.cumsum(nb)))
    c1col, p1col, c2col, p2col = columns
    keys, counts = [], dict(lines=0, cis=0, trans=0, unplaced=0)
    for path in paths:
        df = pd.read_csv(path, sep=r"\s+", comment="#", header=None, usecols=list(columns),
                         dtype={c1col: str, c2col: str, p1col: np.int64, p2col: np.int64}, engine="c")
        index = pd.Index(names)
        c1 = index.get_indexer(df[c1col]).astype(np.int64)                 # -1: not in the table
        c2 = index.get_indexer(df[c2col]).astype(np.int64)
        p1, p2 = df[p1col].to_numpy() - index_base, df[p2col].to_numpy() - index_base
        for c, p in ((c1, p1), (c2, p2)):
            ok = c >= 0
            assert np.all((p[ok] >= 0) & (p[ok] < lens[c[ok]])), "a position outside its chromosome"
        placed = (c1 >= 0) & (c2 >= 0)
        cis = placed & (c1 == c2)
        counts["lines"] += int(c1.size)
        counts["unplaced"] += int((~placed).sum())
        counts["trans"] += int((placed & (c1 != c2)).sum())
        counts["cis"] += int(cis.sum())
        b1, b2 = p1[cis] // binsize, p2[cis] // binsize
        s = starts[c1[cis]]
        keys.append(((s + np.minimum(b1, b2)) << 31) | (s + np.maximum(b1, b2)))
    k, v = np.unique(np.concatenate(keys) if keys else np.zeros(0, np.int64), return_counts=True)
    gi, gj = k >> 31, k & 0x7fffffff
    c = np.searchsorted(starts, gi, side="right") - 1
    out = []
    for ch in range(len(chromsizes)):
        m = c == ch
        out.append((gi[m] - starts[ch], gj[m] - starts[ch], v[m].astype(np.float64)))
    return out, counts


# ---- synthetic pair files -------------------------------------------------------------------------------------------

def _right(vals, width):
    """right-aligned decimal digits of vals (non-negative) in `width` columns, space-padded: an [n, width] uint8 array"""
    v = np.asarray(vals, dtype=np.int64)
    out = np.full((v.size, width), ord(" "), dtype=np.uint8)
    for k in range(width):
        d = (v // 10 ** k) % 10
        show = (v >= 10 ** k) | (k == 0)
        out[:, width - 1 - k] = np.where(show, d + ord("0"), ord(" "))
    return out


def _left(names, idx, width):
    tab = np.full((len(names), width), ord(" "), dtype=np.uint8)
    for r, nm in enumerate(names):
        b = nm.encode()
        tab[r, :len(b)] = np.frombuffer(b, dtype=np.uint8)
    return tab[np.asarray(idx)]


def synth_pairs(chromsizes, n_cis, n_trans, n_unplaced, seed, index_base=1, max_dist=2_000_000):
    """(names, chrom1, pos1, chrom2, pos2) of seeded pairs: cis pairs whose distance decays like 1/d (up to max_dist,
    clipped to the chromosome; a fifth swapped so pos1 > pos2), trans pairs between two table chromosomes, and unplaced
    pairs with one end on a name outside the table.  Names index `names` (the table's, then UNPLACED)."""
    rng = np.random.default_rng(seed)
    names = [nm for nm, _ in chromsizes] + UNPLACED
    lens = np.array([ln for _, ln in chromsizes], dtype=np.int64)
    nc = len(chromsizes)
    w = lens / lens.sum()
    c = rng.choice(nc, n_cis, p=w)
    a = (rng.random(n_cis) * lens[c]).astype(np.int64)
    d = np.floor(np.exp(rng.random(n_cis) * np.log(max_dist))).astype(np.int64) - 1
    b = np.minimum(a + d, lens[c] - 1)
    sw = rng.random(n_cis) < 0.2
    a, b = np.where(sw, b, a), np.where(sw, a, b)
    t1 = rng.choice(nc, n_trans, p=w)
    t2 = (t1 + rng.integers(1, nc, n_trans)) % nc if nc > 1 else t1
    ta = (rng.random(n_trans) * lens[t1]).astype(np.int64)
    tb = (rng.random(n_trans) * lens[t2]).astype(np.int64)
    u1 = rng.choice(nc, n_unplaced, p=w)
    u2 = nc + rng.integers(0, len(UNPLACED), n_unplaced)
    ua = (rng.random(n_unplaced) * lens[u1]).astype(np.int64)
    ub = rng.integers(0, 10 ** 6, n_unplaced)
    flip = rng.random(n_unplaced) < 0.5
    u1, u2, ua, ub = np.where(flip, u2, u1), np.where(flip, u1, u2), np.where(flip, ub, ua), np.where(flip, ua, ub)
    c1 = np.concatenate([c, t1, u1]); c2 = np.concatenate([c, t2, u2])
    p1 = np.concatenate([a, ta, ua]); p2 = np.concatenate([b, tb, ub])
    o = rng.permutation(c1.size)
    return names, c1[o], p1[o] + index_base, c2[o], p2[o] + index_base


def pair_lines(layout, names, c1, p1, c2, p2, first_id=0):
    """The lines of the pairs in `layout` as bytes: space-padded fixed-width fields separated by tabs"""
    n = c1.size
    wn = max(len(nm) for nm in names)
    wp = max(2, len(str(int(max(p1.max(initial=0), p2.max(initial=0))))))
    tab, sp = np.full((n, 1), 9, np.uint8), np.full((n, 1), 32, np.uint8)
    rid = np.concatenate([np.full((n, 1), ord("r"), np.uint8), _right(np.arange(first_id, first_id + n), 10)], axis=1)
    rid[rid == 32] = ord("0")
    s1 = np.where(np.arange(n) % 2 == 0, ord("+"), ord("-")).astype(np.uint8)[:, None]
    s2 = np.where(np.arange(n) % 3 == 0, ord("+"), ord("-")).astype(np.uint8)[:, None]
    C1, P1, C2, P2 = _left(names, c1, wn), _right(p1, wp), _left(names, c2, wn), _right(p2, wp)
    frag = _right(np.arange(n) % 977, 4)
    if layout == "4dn":                     # readID chrom1 pos1 chrom2 pos2 strand1 strand2
        parts = [rid, tab, C1, tab, P1, tab, C2, tab, P2, tab, s1, tab, s2]
    elif layout == "hicpro":                # readID chr1 pos1 strand1 chr2 pos2 strand2 size
        parts = [rid, tab, C1, tab, P1, tab, s1, tab, C2, tab, P2, tab, s2, tab, frag]
    elif layout == "juicer":                # str1 chr1 pos1 frag1 str2 chr2 pos2 frag2 mapq1 mapq2
        z, o = np.full((n, 1), ord("0"), np.uint8), np.full((n, 1), ord("1"), np.uint8)
        parts = [z, sp, C1, sp, P1, sp, frag, sp, o, sp, C2, sp, P2, sp, frag, sp, _right(np.full(n, 60), 2), sp,
                 _right(np.full(n, 42), 2)]
    else:
        raise ValueError(layout)
    arr = np.concatenate(parts + [np.full((n, 1), 10, np.uint8)], axis=1)
    return arr.tobytes()


def header(layout, chromsizes):
    if layout == "4dn":
        h = "## pairs format v1.0\n" + "".join(f"#chromsize: {nm} {ln}\n" for nm, ln in chromsizes)
        return (h + "#columns: readID chr1 pos1 chr2 pos2 strand1 strand2\n").encode()
    return f"# synthetic {layout} pairs\n".encode()


def quirk_lines(layout, chromsizes, index_base, seed):
    """Hand-made lines around the edges of the spec, in `layout`: CRLF endings, blank and whitespace-only lines,
    comments, mixed tabs and spaces, leading blanks, swapped pairs, duplicates, positions at index_base and at each
    chromosome's last base, chr1 / chr10 prefixes and every unplaced name."""
    rng = np.random.default_rng(seed)
    cols = LAYOUTS[layout]
    width = FIELDS[layout]
    out = []

    def line(c1, p1, c2, p2, sep="\t", lead="", end="\n"):
        f = [f"x{k}" for k in range(width)]
        f[cols[0]], f[cols[1]], f[cols[2]], f[cols[3]] = c1, str(p1), c2, str(p2)
        out.append(lead + sep.join(f) + end)

    lo = index_base
    for nm, ln in chromsizes[:6]:
        hi = ln - 1 + index_base
        line(nm, lo, nm, hi)
        line(nm, hi, nm, lo, sep=" \t ")
        line(nm, hi, nm, hi, end="\r\n")
        line(nm, lo, nm, lo, lead="  \t")
    nm0, ln0 = chromsizes[0]
    for _ in range(3):
        line(nm0, 5 + index_base, nm0, 3 + index_base)      # duplicates, swapped
    out.append("\n")
    out.append(" \t \r\n")
    out.append("\r\n")
    out.append("# a comment in the middle\n")
    out.append("#\n")
    for u in UNPLACED:
        line(u, 7, nm0, lo)
        line(nm0, lo + 1, u, 99999999999)
    if len(chromsizes) > 1:
        line(chromsizes[1][0], lo, nm0, ln0 - 1 + index_base, sep="  ")
    for _ in range(20):
        c = int(rng.integers(0, len(chromsizes)))
        nm, ln = chromsizes[c]
        a, b = (int(x) + index_base for x in rng.integers(0, ln, 2))
        line(nm, a, nm, b, sep=rng.choice(["\t", " ", "\t\t", " \t"]), end=rng.choice(["\n", "\r\n"]))
    return "".join(out).encode()


def write_pairs(path, layout, chromsizes, n_cis, n_trans, n_unplaced, seed, index_base=1, quirks=False, head=True,
                chunk=4_000_000):
    """A seeded synthetic pair file in `layout` ("4dn", "hicpro", "juicer"): header lines, then the pairs of
    synth_pairs (and the quirk lines, when asked), written in chunks of `chunk` pairs."""
    with open(path, "wb") as fh:
        if head:
            fh.write(header(layout, chromsizes))
        if quirks:
            fh.write(quirk_lines(layout, chromsizes, index_base, seed))
        total, done = n_cis + n_trans + n_unplaced, 0
        nchunk = max(1, -(-total // chunk))
        for k in range(nchunk):
            part = [x * (k + 1) // nchunk - x * k // nchunk for x in (n_cis, n_trans, n_unplaced)]
            names, c1, p1, c2, p2 = synth_pairs(chromsizes, *part, seed * 1000 + k, index_base)
            if c1.size:
                fh.write(pair_lines(layout, names, c1, p1, c2, p2, first_id=done))
                done += c1.size
        if quirks:
            fh.write(b"# the end\n")
