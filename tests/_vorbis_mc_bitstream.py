"""Multichannel Vorbis stream WRITER for the front-end tests: tests/_vorbis_bitstream.py's setup headers and audio packets (same codebooks,
floor-1 and residue configurations, same ground truth), extended to C channels with a list of coupling steps (chained steps allowed, one
list per mapping if asked for), 1..n sub-maps with a random multiplex for any C, and truth arrays of max(2, C) planes.  Builders only;
nothing here reads a bitstream."""
import numpy as np

from tests._streams import BitWriterRtl, _ilog, vorbis_ident
from tests._vorbis_bitstream import Book

f32 = np.float32


class Stream:
    """A whole logical stream's headers + a packet generator with ground truth, for any channel count (the two-channel writer of
    tests/_vorbis_bitstream.py with coupling lists, sub-maps for any channel count and an optional floor 0; its own streams are
    not these)."""

    def __init__(self, rng, channels=2, bs_exp=(7, 9), residue_type=None, per_word=None, residue_begin=None, couplings=(), max_submaps=1,
                 mapping_couplings=None, extra_floor0=False):
        """couplings: the (magnitude, angle) steps written into every mapping (chained steps allowed).  max_submaps: 1..max_submaps
        sub-maps per mapping with a random multiplex.  mapping_couplings: one step list per mapping (mapping k takes entry k modulo the
        list's length) instead of `couplings`.  extra_floor0: one more floor, of type 0, that no mapping uses."""
        self.rng, self.channels, self.bs_exp = rng, channels, bs_exp
        self.planes = max(2, channels)   # truth arrays: [planes][65] / [planes][slot]
        self.ident = vorbis_ident(channels=channels, bs0=bs_exp[0], bs1=bs_exp[1])
        books = []
        # floor books: scalar, small alphabets
        n_floor_books = int(rng.integers(2, 5))
        for _ in range(n_floor_books):
            books.append(Book(rng, int(rng.integers(1, 40)), 1))
        # residue class book: dims = partitions per class word, entries = classifications^dims exactly
        self.classifications = int(rng.integers(1, 5))
        # class words of several partitions: when the partition count is not a multiple of it, the reference lets the last word spill
        # into the next channel's classes (residue.rs:451-477 bounds the write by the vector's end) -- the truth kept here follows
        # the specification, so comparisons against it use per_word = 1; reader-vs-reader comparisons use any
        self.per_word = int(rng.integers(1, 4)) if per_word is None else per_word
        class_book = len(books)
        books.append(Book(rng, self.classifications ** self.per_word, self.per_word, style="plain"))
        vq_first = len(books)
        for _ in range(int(rng.integers(2, 5))):
            dims = int(rng.choice([1, 2, 4, 8]))
            books.append(Book(rng, int(rng.integers(2, 30)), dims, vq=(int(rng.integers(1, 3)), bool(rng.integers(2)))))
        self.books = books
        w = BitWriterRtl()
        w.put(len(books) - 1, 8)
        for b in books:
            w.v |= b.bits.v << w.n
            w.n += b.bits.n
        w.put(0, 6), w.put(0, 16)
        # floors (type 1)
        self.floors = []
        n_floors = int(rng.integers(1, 4))
        w.put(n_floors - 1 + int(extra_floor0), 6)
        for _ in range(n_floors):
            w.put(1, 16)
            rangebits = bs_exp[0] - 1
            parts = int(rng.integers(0, 6))
            pclass = [int(rng.integers(0, 3)) for _ in range(parts)]
            classes = {}
            w.put(parts, 5)
            for c in pclass:
                w.put(c, 4)
            if parts:
                for c in range(max(pclass) + 1):
                    dims, sub = int(rng.integers(1, 4)), int(rng.integers(0, 3))
                    w.put(dims - 1, 3), w.put(sub, 2)
                    main = int(rng.integers(n_floor_books))
                    if sub:
                        w.put(main, 8)
                    subbooks = []
                    for _k in range(1 << sub):
                        sb = int(rng.integers(0, n_floor_books + 1))  # 0 = none
                        w.put(sb, 8)
                        subbooks.append(sb - 1 if sb else None)
                    classes[c] = dict(dims=dims, sub=sub, main=main, subbooks=subbooks)
            mult = int(rng.integers(1, 5))
            w.put(mult - 1, 2), w.put(rangebits, 4)
            n_x = sum(classes[c]["dims"] for c in pclass)
            xs = [int(v) for v in rng.choice(np.arange(1, 1 << rangebits), size=n_x, replace=False)]
            for x in xs:
                w.put(x, rangebits)
            self.floors.append(dict(multiplier=mult, pclass=pclass, classes=classes, n_posts=2 + n_x))
        if extra_floor0:   # order, rate, bark map size, amplitude bits, amplitude offset, one book
            w.put(0, 16), w.put(8, 8), w.put(44100, 16), w.put(256, 16), w.put(6, 6), w.put(100, 8), w.put(0, 4), w.put(0, 8)
        # residues
        self.residues = []
        n_res = int(rng.integers(1, 3))
        w.put(n_res - 1, 6)
        for _ in range(n_res):
            rtype = int(rng.integers(3)) if residue_type is None else residue_type
            n2_short = (1 << bs_exp[0]) >> 1
            part_size = int(rng.choice([8, 16]))
            begin = int(rng.choice([0, part_size])) if residue_begin is None else residue_begin
            end = int(rng.choice([n2_short, (1 << bs_exp[1]) >> 1, 1 << bs_exp[1], 3 * part_size + begin]))
            if end < begin:   # (a setup header with end < begin is refused, residue.rs:88-90)
                end = begin + 3 * part_size
            w.put(rtype, 16), w.put(begin, 24), w.put(end, 24), w.put(part_size - 1, 24)
            w.put(self.classifications - 1, 6), w.put(class_book, 8)
            used = []
            for _c in range(self.classifications):
                u = int(rng.integers(0, 8)) | (int(rng.integers(2)) << int(rng.integers(3, 8)))
                w.put(u & 7, 3)
                if u >> 3:
                    w.put(1, 1), w.put(u >> 3, 5)
                else:
                    w.put(0, 1)
                used.append(u)
            vbooks = [[None] * 8 for _ in used]
            for ci, u in enumerate(used):
                for j in range(8):
                    if u >> j & 1:
                        vbooks[ci][j] = int(rng.integers(vq_first, len(books)))
                        w.put(vbooks[ci][j], 8)
            self.residues.append(dict(type=rtype, begin=begin, end=end, part_size=part_size, used=used, books=vbooks))
        if mapping_couplings is not None:
            couplings = mapping_couplings[0]
        self.couplings = [(int(m), int(a)) for m, a in couplings]
        n_map = int(rng.integers(1, 3))
        w.put(n_map - 1, 6)
        self.mappings = []
        for k_map in range(n_map):
            steps = self.couplings if mapping_couplings is None else [(int(m), int(a)) for m, a in mapping_couplings[k_map % len(mapping_couplings)]]
            w.put(0, 16)
            submaps = int(rng.integers(1, max_submaps + 1))
            if submaps > 1:
                w.put(1, 1), w.put(submaps - 1, 4)
            else:
                w.put(0, 1)
            if steps:
                w.put(1, 1), w.put(len(steps) - 1, 8)
                for m, a in steps:
                    w.put(m, _ilog(channels - 1)), w.put(a, _ilog(channels - 1))
            else:
                w.put(0, 1)
            w.put(0, 2)
            mux = [0] * channels
            if submaps > 1:
                mux = [int(rng.integers(submaps)) for _ in range(channels)]
                for m in mux:
                    w.put(m, 4)
            sm = []
            for _k in range(submaps):
                fl, rs = int(rng.integers(n_floors)), int(rng.integers(n_res))
                w.put(0, 8), w.put(fl, 8), w.put(rs, 8)
                sm.append((fl, rs))
            self.mappings.append(dict(mux=mux, submaps=sm, couplings=steps))
        n_modes = int(rng.integers(1, 5))
        w.put(n_modes - 1, 6)
        self.modes = []
        for _ in range(n_modes):
            flag, mp = int(rng.integers(2)), int(rng.integers(n_map))
            w.put(flag, 1), w.put(0, 16), w.put(0, 16), w.put(mp, 8)
            self.modes.append((bool(flag), mp))
        w.put(1, 1)
        self.setup = b"\x05vorbis" + w.bytes()
        self.prev_flag = None

    def packet(self, unused_prob=0.15):
        """One audio packet: (bytes, truth dict like the oracle's decode result)."""
        rng = self.rng
        w = BitWriterRtl()
        w.put(0, 1)
        mode = int(rng.integers(len(self.modes)))
        w.put(mode, _ilog(len(self.modes) - 1))
        long_block, mp = self.modes[mode]
        if long_block:
            w.put(int(rng.integers(2)), 1), w.put(int(rng.integers(2)), 1)
        mapping = self.mappings[mp]
        n2 = (1 << (self.bs_exp[1] if long_block else self.bs_exp[0])) >> 1
        slot = (1 << self.bs_exp[1]) >> 1
        floor_y = np.zeros((self.planes, 65), dtype=np.uint16)
        dnd, floor_idx = [True] * self.planes, [None] * self.planes
        for ch in range(self.channels):
            fi = mapping["submaps"][mapping["mux"][ch]][0]
            f = self.floors[fi]
            if rng.random() < unused_prob:
                w.put(0, 1)
                continue
            w.put(1, 1)
            rng_ = {1: 256, 2: 128, 3: 86, 4: 64}[f["multiplier"]]
            bits = _ilog(rng_ - 1)
            y = [int(rng.integers(rng_)), int(rng.integers(rng_))]
            w.put(y[0], bits), w.put(y[1], bits)
            for c in f["pclass"]:
                cl = f["classes"][c]
                cval = 0
                if cl["sub"]:
                    book = self.books[cl["main"]]
                    cval = int(rng.choice(book.usable))
                    book.put(w, cval)
                for _d in range(cl["dims"]):
                    sub = cval & ((1 << cl["sub"]) - 1)
                    cval >>= cl["sub"]
                    sb = cl["subbooks"][sub]
                    if sb is None:
                        y.append(0)
                    else:
                        e = int(rng.choice(self.books[sb].usable))
                        self.books[sb].put(w, e)
                        y.append(e)
            dnd[ch], floor_idx[ch] = False, fi
            floor_y[ch, :len(y)] = y
        for m, a in mapping["couplings"]:   # non-zero vector propagate, step by step (Vorbis I 4.3.2 step 6)
            if dnd[m] != dnd[a]:
                dnd[m] = dnd[a] = False
        residue = np.zeros((self.planes, slot), dtype=np.float32)
        for sm, (_fl, ri) in enumerate(mapping["submaps"]):
            chans = [c for c in range(self.channels) if mapping["mux"][c] == sm]
            if not chans:
                continue
            r = self.residues[ri]
            count = len(chans)
            full = n2 * count if r["type"] == 2 else n2
            begin, end = min(r["begin"], full), min(r["end"], full)
            parts = (end - begin) // r["part_size"]
            if not any(not dnd[c] for c in chans):
                continue
            buf = np.zeros(full, dtype=np.float32)
            lanes = [None] if r["type"] == 2 else [c for c in chans]
            active = [True] if r["type"] == 2 else [not dnd[c] for c in chans]
            classes = {k: [0] * (parts + self.per_word) for k in range(len(lanes))}
            max_pass = max([j for u in r["used"] for j in range(8) if u >> j & 1], default=0)
            class_book = self.books[[k for k, b in enumerate(self.books) if b.dims == self.per_word and b.entries == self.classifications ** self.per_word and b.vq is None][-1]]
            for p in range(max_pass + 1):
                for first in range(0, parts, self.per_word):
                    if p == 0:
                        for k in range(len(lanes)):
                            if not active[k]:
                                continue
                            group = [int(rng.integers(self.classifications)) for _ in range(self.per_word)]
                            val = 0
                            for g in group:
                                val = val * self.classifications + g
                            class_book.put(w, val)
                            classes[k][first:first + self.per_word] = group
                    for part in range(first, min(parts, first + self.per_word)):
                        for k in range(len(lanes)):
                            if not active[k]:
                                continue
                            cls = classes[k][part]
                            if not r["used"][cls] >> p & 1:
                                continue
                            book = self.books[r["books"][cls][p]]
                            start = begin + r["part_size"] * part
                            target = buf if r["type"] == 2 else residue[lanes[k]]
                            n = r["part_size"]
                            if r["type"] == 0:
                                step = n // book.dims
                                for i in range(step):
                                    e = int(rng.integers(book.entries)) if len(book.usable) == book.entries else int(rng.choice(book.usable))
                                    book.put(w, e)
                                    for d, o in zip(range(book.dims), range(i, n, step)):
                                        target[start + o] = f32(target[start + o] + book.vq[e, d])
                            else:
                                for o in range(0, n - book.dims + 1, book.dims):
                                    e = int(rng.choice(book.usable))
                                    book.put(w, e)
                                    for d in range(book.dims):
                                        target[start + o + d] = f32(target[start + o + d] + book.vq[e, d])
            if r["type"] == 2:
                for i, c in enumerate(chans):
                    residue[c, :n2] = buf[i::count][:n2]
        prev = long_block if self.prev_flag is None else self.prev_flag
        self.prev_flag = long_block
        return w.bytes(), dict(block_flag=long_block, prev_block_flag=prev, do_not_decode=dnd, floor=floor_idx, floor_y=floor_y, residue=residue)
