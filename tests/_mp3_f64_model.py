"""Float64 model of MPEG Layer III synthesis: an independent check of the oracle (oracle/oracle_mp3.cpp).

Same contract as `oracle_mp3_batch`: units [F,2,2], spectra [F,2,2,576] (sign * |q|^(4/3) as the Huffman stage emits them)
and runs in, PCM [F,2,1152] out, with fresh per-stream state (hybrid overlap and polyphase FIFO) that carries across the
granules and frames of a stream.

Same decisions as the reference.  Every data-dependent choice the reference (symphonia-bundle-mp3 @ ee35874) makes is
followed and cited below: which bands are requantised, the intensity-stereo bound searches, the `rzero` bookkeeping
that decides how far alias reduction and the IMDCTs reach.  These choices are taken on exact inputs (scale factors,
flags and zero tests on the spectra), so the model and the oracle take the same branches and any difference between
them is arithmetic.

Different arithmetic from the reference.  Every stage is evaluated in float64 from its defining formula, not with the
reference's fast algorithms or f32 tables: requantisation as x * 2^((A-B)/4); mid/side with 1/sqrt(2); MPEG-1 intensity
ratios from tan(pos * pi/12), MPEG-2 ratios as powers of 2^(-1/4) or 2^(-1/2); the alias butterflies from the normative
Ci list; IMDCT-36 and IMDCT-12 as direct cosine sums with the four windows from their sine formulas; the polyphase bank
as the ISO 11172-3 matrixing V = N * S followed by the windowing.

Shared data.  Two tables are not recomputed here: the 512-tap synthesis window D (taken from `oracle_mp3_tables`) and
the scale-factor band edges with the mixed-block switch points (parsed from oracle/mp3_iso_data.h).  Neither has a
closed form -- both are normative lists -- and tools/verify_constants_vs_reference.py checks both bit for bit against
the reference's literals, so sharing them cannot hide an arithmetic error in the oracle.

Where the reference departs from the ISO text, the model follows the reference:
  * a mixed block's long part is requantised over bands[..switch] (requantize.rs:374), one band short of the switch
    point: the last long band (samples 30..36 at 44.1 kHz) keeps its unscaled |q|^(4/3) values;
  * alias reduction of a mixed block sets rzero to 36 (hybrid_synthesis.rs:225, :240), so hybrid synthesis treats
    sub-bands 2..31 as zero (:287, :351-358): the short part of a mixed block never reaches the output.

Speed: every stateless stage runs vectorised over all granule-channels of the batch at once; only the intensity-stereo
bound search loops over granules (in Python), and the two stateful stages (overlap-add, polyphase) run per stream and
channel over that lane's granules.
"""
import os
import re

import numpy as np

from symphonia_b200._native import (F_INTENSITY, F_MID_SIDE, F_MIXED, F_MPEG1, F_PREFLAG, F_SCALEFAC_SCALE, F_SFC_LSB,
                                    MP3_END, MP3_SHORT, MP3_START)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Plausible bugs the model can be asked to make (`mutation=`); the suite shows each one misses the tolerance.
MUTATIONS = (
    "band_edge",            # long band 5 starts one line late in requantisation
    "pretab_shift",         # pretab applied one band early
    "short_window_gain",    # sub-block gain of the wrong window in short bands
    "mixed_long_per_iso",   # mixed long part requantised up to the switch point (the ISO text, not the reference)
    "is_ratio_pos",         # MPEG-1 intensity ratio of pos 2 taken from pos 3
    "is_pos21",             # is_pos[21] read from scalefacs[21] instead of copied from band 20
    "mpeg2_is_scale",       # MPEG-2 intensity ratios with the two SFC_LSB scales swapped
    "short_is_sfi",         # short-block intensity scan reads is_pos[sfi] instead of is_pos[sfi - 1]
    "ms_above_is",          # mid/side applied up to rzero, above the intensity bound too
    "rzero_no_merge",       # joint stereo leaves each channel its own rzero
    "alias_into_short",     # alias reduction of a mixed block also runs at the boundary of sub-bands 1 and 2
    "cs_ca_sign",           # sign error in the ca term of butterfly 3 (upper sample)
    "freq_inv_skip",        # frequency inversion skips slot 17
    "overlap_other_ch",     # channel 1 overlap-adds channel 0's IMDCT tail
)


# ---- shared tables -------------------------------------------------------------------------------------------------
def _parse_header():
    src = open(os.path.join(ROOT, "oracle", "mp3_iso_data.h")).read()

    def table(name):
        m = re.search(r"\b" + name + r"\[9\](?:\[\d+\])? = \{(.*?)\};", src, re.S)
        body = re.sub(r"//.*", "", m.group(1))
        rows = re.findall(r"\{(.*?)\}", body, re.S)
        if rows:
            return [[int(x) for x in r.split(",") if x.strip()] for r in rows]
        return [int(x) for x in body.split(",") if x.strip()]

    long_e, short_e, mixed_e = table("kLongEdges"), table("kShortEdges"), table("kMixedEdges")
    count, switch = table("kMixedCount"), table("kMixedSwitch")
    mixed_e = [row[:count[sr]] for sr, row in enumerate(mixed_e)]
    return long_e, short_e, mixed_e, switch


LONG_EDGES, SHORT_EDGES, MIXED_EDGES, MIXED_SWITCH = _parse_header()
# ISO/IEC 11172-3 Table B.6 (requantize.rs:255-256)
PRETAB = [0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 3, 2, 0]
# ISO/IEC 11172-3 Table B.9: the alias-reduction coefficients Ci
ALIAS_C = np.array([-0.6, -0.535, -0.33, -0.185, -0.095, -0.041, -0.0142, -0.0037])

_D = None


def synth_window():
    """The 512-tap synthesis window D, as the f32 values the reference parses (shared with the oracle)."""
    global _D
    if _D is None:
        from tests import _oracle
        lib = _oracle.load()
        n = lib.oracle_mp3_tables(None, 0)
        tab = np.zeros(n, dtype=np.float32)
        lib.oracle_mp3_tables(_oracle.ptr(tab), n)
        _D = tab[:512].astype(np.float64)
    return _D


# ---- closed forms ----------------------------------------------------------------------------------------------------
def imdct_windows():
    """The four IMDCT windows of ISO/IEC 11172-3 2.4.3.4.10.3: normal, start, short, stop."""
    i = np.arange(36) + 0.5
    w = np.zeros((4, 36))
    w[0] = np.sin(np.pi / 36 * i)
    w[1, :18] = w[0, :18]
    w[1, 18:24] = 1.0
    w[1, 24:30] = np.sin(np.pi / 12 * (i[24:30] - 18))
    w[2, :12] = np.sin(np.pi / 12 * i[:12])
    w[3, 6:12] = np.sin(np.pi / 12 * (i[6:12] - 6))
    w[3, 12:18] = 1.0
    w[3, 18:] = w[0, 18:]
    return w


_WIN = imdct_windows()
_C36 = np.cos(np.pi / 72 * np.outer(2 * np.arange(36) + 1 + 18, 2 * np.arange(18) + 1))  # [36, 18]
_C12 = np.cos(np.pi / 24 * np.outer(2 * np.arange(12) + 1 + 6, 2 * np.arange(6) + 1))    # [12, 6]
_N = np.cos(np.pi / 64 * np.outer(16 + np.arange(64), 2 * np.arange(32) + 1))              # [64, 32]


def is_ratios(pos, mpeg1, lsb, mutation=None):
    """(k_l, k_r) of intensity position `pos` (ISO/IEC 11172-3 2.4.3.4.9.3, 13818-3 2.4.3.2)."""
    if mpeg1:
        if mutation == "is_ratio_pos" and pos == 2:
            pos = 3
        if pos == 6:  # tan(pi/2): the limit (1, 0), as the reference tabulates it (stereo.rs:118)
            return 1.0, 0.0
        t = np.tan(pos * np.pi / 12)
        return t / (1 + t), 1 / (1 + t)
    if mutation == "mpeg2_is_scale":
        lsb = not lsb
    step = 0.5 if lsb else 0.25  # i0 = 2^(-1/4) for scalefac_compress & 1 == 0, 2^(-1/2) for 1 (stereo.rs:59-63)
    if pos & 1:
        return 2.0 ** (-step * (pos + 1) / 2), 1.0
    return 1.0, 2.0 ** (-step * pos / 2)


# ---- per-(sample rate, block kind) line tables -------------------------------------------------------------------------
KIND_LONG, KIND_SHORT, KIND_MIXED = 0, 1, 2


def _line_tables(mutation):
    """For every sample-rate index and block kind, per spectral line: the scale-factor index whose gain scales it (-1: not
    requantised), its short window (-1: long band), its pretab value; and the short-block reorder permutation and the
    rzero it leaves for every rzero in 0..576."""
    sfi = np.full((9, 3, 576), -1, dtype=np.int64)
    win = np.full((9, 3, 576), -1, dtype=np.int64)
    pre = np.zeros((9, 3, 576), dtype=np.int64)
    perm = np.tile(np.arange(576), (9, 3, 1))
    rz_after = np.tile(np.arange(577), (9, 3, 1))
    pretab = PRETAB[1:] + [0] if mutation == "pretab_shift" else PRETAB

    def long_bands(k, sr, edges):
        for i in range(len(edges) - 1):
            sfi[sr, k, edges[i]:edges[i + 1]] = i
            pre[sr, k, edges[i]:edges[i + 1]] = pretab[i]

    def short_bands(k, sr, edges, first_sf):
        for i in range(len(edges) - 1):
            sfi[sr, k, edges[i]:edges[i + 1]] = first_sf + i
            # A = global_gain - 210 - 8 * subblock_gain[i % 3] (requantize.rs:317-321, :343)
            win[sr, k, edges[i]:edges[i + 1]] = (i + 1) % 3 if mutation == "short_window_gain" else i % 3

    def reorder(k, sr, bands):
        # hybrid_synthesis.rs:183-213: window-major quads interleaved; quads starting at or above rzero are skipped
        quads = [bands[q:q + 4] for q in range(0, len(bands) - 3, 3)]
        for s0, s1, s2, s3 in quads:
            n = min(s1 - s0, s2 - s1, s3 - s2)
            for w, sw in enumerate((s0, s1, s2)):
                perm[sr, k, s0 + w + 3 * np.arange(n)] = sw + np.arange(n)
        for rz in range(577):
            i = bands[0]
            for s0, s1, s2, s3 in quads:
                if s0 >= rz:
                    break
                i += 3 * min(s1 - s0, s2 - s1, s3 - s2)
            rz_after[sr, k, rz] = max(rz, i)  # :213

    for sr in range(9):
        edges = list(LONG_EDGES[sr])
        if mutation == "band_edge":
            edges[5] += 1
        long_bands(KIND_LONG, sr, edges)                                     # requantize.rs:378
        short_bands(KIND_SHORT, sr, SHORT_EDGES[sr], 0)                     # :361
        sw, mixed = MIXED_SWITCH[sr], MIXED_EDGES[sr]
        long_bands(KIND_MIXED, sr, mixed[:sw + 1] if mutation == "mixed_long_per_iso" else mixed[:sw])  # :374
        short_bands(KIND_MIXED, sr, mixed[sw:], sw)                          # :375
        reorder(KIND_SHORT, sr, SHORT_EDGES[sr])
        reorder(KIND_MIXED, sr, mixed[sw:])
    return sfi, win, pre, perm, rz_after


_TABLES = {}


def _tables(mutation):
    key = mutation if mutation in ("band_edge", "pretab_shift", "short_window_gain", "mixed_long_per_iso") else None
    if key not in _TABLES:
        _TABLES[key] = _line_tables(key)
    return _TABLES[key]


# ---- joint stereo (stereo.rs), one granule ----------------------------------------------------------------------------
def _mid_side(l, r):
    m, s = l.copy(), r.copy()
    l[:] = (m + s) / np.sqrt(2.0)
    r[:] = (m - s) / np.sqrt(2.0)


def _intensity_band(pos, inv_pos, ratio, ms, l, r):
    # stereo.rs:168-188
    if pos < inv_pos:
        kl, kr = ratio(pos)
        r[:] = kr * l
        l[:] = kl * l
    elif ms:
        _mid_side(l, r)


def _intensity(u1, rz1, ms, end, l, r, mutation):
    """Intensity stereo of one granule; returns the intensity bound.  Zero tests read channel 1 before it is rewritten."""
    sr = int(u1["sample_rate_idx"])
    mpeg1 = bool(u1["flags"] & F_MPEG1)
    lsb = bool(u1["flags"] & F_SFC_LSB)
    inv_pos = 7 if mpeg1 else 31  # INTENSITY_INV_POS_MPEG1 / _MPEG2 (stereo.rs:216-222, :342-348)
    ratio = lambda p: is_ratios(p, mpeg1, lsb, mutation)  # noqa: E731
    sf = [int(v) for v in u1["scalefacs"]]
    bound = end
    if u1["block_type"] != MP3_SHORT:
        # stereo.rs:198-261: bands from the top down while channel 1 is zero; is_pos[21] = is_pos[20] (:228-230)
        pos = sf[:22]
        if mutation != "is_pos21":
            pos[21] = pos[20]
        edges = LONG_EDGES[sr]
        for b in range(21, -1, -1):
            s, e = edges[b], edges[b + 1]
            if not (s >= rz1 or not r[s:e].any()):  # :240
                break
            _intensity_band(pos[b], inv_pos, ratio, ms, l[s:e], r[s:e])
            bound = s
        return bound
    # stereo.rs:265-482: short bands in quads of three windows from the top down, each window with its own bound; a
    # mixed block then continues into its long bands.  is_pos[36..39] = scalefacs[33..36] (:352-354).
    pos = sf[:36] + sf[33:36]
    if u1["flags"] & F_MIXED:
        sw, bands = MIXED_SWITCH[sr], MIXED_EDGES[sr]
        short, long_, sfi = bands[sw:], bands[:sw + 1], len(bands) - 1  # :330-335
    else:
        short, long_, sfi = SHORT_EDGES[sr], None, 39                    # :336-339
    at = (lambda i: pos[i]) if mutation != "short_is_sfi" else (lambda i: pos[min(i + 1, 38)])
    zero = [True, True, True]
    found = False
    for q in reversed(range(0, len(short) - 3, 3)):                      # zip of four shifted iterators, step_by(3), rev
        for w in (2, 1, 0):
            s, e = short[q + w], short[q + w + 1]
            zero[w] = zero[w] and not r[s:e].any()                       # :375, :397, :416
            if zero[w]:
                _intensity_band(at(sfi - 1), inv_pos, ratio, ms, l[s:e], r[s:e])
            elif ms:
                _mid_side(l[s:e], r[s:e])
            sfi -= 1
        bound = short[q]                                                 # :438
        found = not any(zero)
        if found:
            break
    if not found and long_ is not None:                                   # :452-477
        for b in range(len(long_) - 2, -1, -1):
            s, e = long_[b], long_[b + 1]
            if r[s:e].any():
                break
            _intensity_band(at(sfi - 1), inv_pos, ratio, ms, l[s:e], r[s:e])
            sfi -= 1
            bound = s
    return bound


# ---- the batch -------------------------------------------------------------------------------------------------------
def _lanes(runs):
    """(stream, channel) -> the rows (frame * 2 + granule) * 2 + channel that lane synthesises, in decode order."""
    lanes = {}
    for run in runs:
        gpf = int(run["granules_per_frame"]) or 2
        n_ch = int(run["channels"]) or 2
        for f in range(int(run["first_frame"]), int(run["first_frame"]) + int(run["n_frames"])):
            for gr in range(gpf):
                for ch in range(n_ch):
                    lanes.setdefault((int(run["stream"]), ch), []).append((f * 2 + gr) * 2 + ch)
    return lanes


def polyphase(slots):
    """ISO 11172-3 2.4.3.4.10 synthesis of one channel from a fresh state: sub-band samples [T, 32] -> PCM [T, 32].
    V_t = N S_t; U takes V_{t-2a}[0:32] and V_{t-2a-1}[32:64] for a = 0..7; PCM_t = sum over the 16 U blocks of U * D."""
    D = synth_window()
    T = len(slots)
    V = np.zeros((T + 16, 64))
    V[16:] = np.asarray(slots, dtype=np.float64) @ _N.T
    out = np.zeros((T, 32))
    for a in range(8):
        out += V[16 - 2 * a: 16 - 2 * a + T, :32] * D[64 * a: 64 * a + 32]
        out += V[15 - 2 * a: 15 - 2 * a + T, 32:] * D[64 * a + 32: 64 * a + 64]
    return out


def mp3_batch(units, spectra, runs, mutation=None):
    """units [F,2,2] MP3_GC_DTYPE, spectra [F,2,2,576], runs -> PCM [F,2,1152] float64 (untouched slots stay 0)."""
    assert mutation is None or mutation in MUTATIONS, mutation
    units = np.ascontiguousarray(units).reshape(-1)
    F = len(units) // 4
    x = np.asarray(spectra, dtype=np.float32).reshape(F * 4, 576).astype(np.float64)
    lanes = _lanes(runs)
    rows = np.array(sorted(r for rr in lanes.values() for r in rr), dtype=np.int64)
    u = units[rows]
    sr = u["sample_rate_idx"].astype(np.int64)
    bt = u["block_type"]
    flags = u["flags"]
    kind = np.where(bt != MP3_SHORT, KIND_LONG, np.where(flags & F_MIXED, KIND_MIXED, KIND_SHORT))
    rz = u["rzero"].astype(np.int64)
    sfi_t, win_t, pre_t, perm_t, rz_after_t = _tables(mutation)

    # requantisation (requantize.rs:239-381): x * 2^((A - B) / 4), A = global_gain - 210 - 8 * subblock_gain[window],
    # B = ((scalefac + preflag * pretab) << (scalefac_scale ? 2 : 1)) as u8
    sfi, win, pre = sfi_t[sr, kind], win_t[sr, kind], pre_t[sr, kind]
    sf = np.take_along_axis(u["scalefacs"].astype(np.int64), np.maximum(sfi, 0), axis=1)
    shift = np.where(flags & F_SCALEFAC_SCALE, 2, 1)[:, None]
    b = ((sf + pre * ((flags & F_PREFLAG) != 0)[:, None]) << shift) & 0xFF
    sbg = np.take_along_axis(u["subblock_gain"].astype(np.int64), np.maximum(win, 0), axis=1)
    a = u["global_gain"].astype(np.int64)[:, None] - 210 - 8 * np.where(win >= 0, sbg, 0)
    y = x[rows] * np.where(sfi >= 0, np.exp2((a - b) / 4.0), 1.0)

    # joint stereo (stereo.rs:485-556) on the granules of two-channel runs; flags are replicated in both units
    where = {int(r): i for i, r in enumerate(rows)}
    for i, row in enumerate(rows):
        if row & 1 or row + 1 not in where:
            continue
        j = where[row + 1]
        ms, is_ = bool(flags[i] & F_MID_SIDE), bool(flags[i] & F_INTENSITY)
        if not (ms or is_):
            continue
        end = max(rz[i], rz[j])                                               # :521
        bound = _intensity(u[j], rz[j], ms, end, y[i], y[j], mutation) if is_ else end
        if ms and bound > 0:                                                  # :542-544
            hi = end if mutation == "ms_above_is" else bound
            _mid_side(y[i, :hi], y[j, :hi])
        if mutation != "rzero_no_merge":
            rz[i] = rz[j] = end                                               # :550-553

    # short-block reorder (hybrid_synthesis.rs:153-215)
    y = np.take_along_axis(y, perm_t[sr, kind], axis=1)
    rz = rz_after_t[sr, kind, rz]

    # alias reduction (:218-277): butterflies at the boundaries 18k, k < min(sb_limit, rzero / 18 + 2), where sb_limit is
    # 32 for long blocks, 2 for mixed blocks and 0 (nothing) for short blocks; rzero becomes 18 * that limit (:240)
    sb_limit = np.where(kind == KIND_LONG, 32, np.where(kind == KIND_MIXED, 2, 0))
    n_bound = np.minimum(sb_limit, rz // 18 + 2)
    rz = np.where(kind == KIND_SHORT, rz, 18 * n_bound)
    if mutation == "alias_into_short":
        n_bound = np.where(kind == KIND_MIXED, 3, n_bound)
    cs, ca = 1 / np.sqrt(1 + ALIAS_C ** 2), ALIAS_C / np.sqrt(1 + ALIAS_C ** 2)
    k = np.arange(1, 32)[:, None]
    lo, up = (18 * k - 1 - np.arange(8)).ravel(), (18 * k + np.arange(8)).ravel()
    cs8, ca8 = np.tile(cs, 31), np.tile(ca, 31)
    aliased = y.copy()
    aliased[:, lo] = y[:, lo] * cs8 - y[:, up] * ca8
    ca_up = ca8.copy()
    if mutation == "cs_ca_sign":
        ca_up[3::8] = -ca_up[3::8]
    aliased[:, up] = y[:, up] * cs8 + y[:, lo] * ca_up
    line_boundary = np.zeros(576, dtype=np.int64)  # the boundary a line's butterfly belongs to (0: none)
    line_boundary[lo], line_boundary[up] = np.repeat(np.arange(1, 32), 8), np.repeat(np.arange(1, 32), 8)
    y = np.where((line_boundary > 0) & (line_boundary < n_bound[:, None]), aliased, y)

    # hybrid synthesis (:280-359): sub-bands at or above ceil(rzero / 18) are zero; the first sb_split sub-bands take the
    # 36-point IMDCT with the block type's window, the rest three 12-point IMDCTs with the short window
    sb = y.reshape(-1, 32, 18) * (np.arange(32)[None, :] < -(-rz // 18)[:, None])[..., None]
    wsel = np.where(bt == MP3_START, 1, np.where(bt == MP3_END, 3, 0))
    long_out = (sb @ _C36.T) * _WIN[wsel][:, None, :]
    short_out = np.zeros_like(long_out)
    for w in range(3):
        short_out[..., 6 + 6 * w: 18 + 6 * w] += (sb[..., w::3] @ _C12.T) * _WIN[2, :12]
    split = np.where(kind == KIND_LONG, 32, np.where(kind == KIND_MIXED, 2, 0))
    z = np.where((np.arange(32)[None, :] < split[:, None])[..., None], long_out, short_out)  # [rows, 32, 36]

    pcm = np.zeros((F, 2, 1152))
    for (stream, ch), lane in lanes.items():
        idx = np.array([where[r] for r in lane])
        tail = z[idx, :, 18:]
        if mutation == "overlap_other_ch" and ch == 1 and (stream, 0) in lanes:
            tail = z[np.array([where[r - 1] for r in lane]), :, 18:]
        s = z[idx, :, :18].copy()
        s[1:] += tail[:-1]                                                    # overlap-add across granules
        # frequency inversion (:458-485): odd time slots of odd sub-bands
        odd = np.arange(1, 18, 2)
        if mutation == "freq_inv_skip":
            odd = odd[:-1]
        s[:, 1::2][..., odd] *= -1.0
        out = polyphase(s.transpose(0, 2, 1).reshape(-1, 32)).reshape(len(lane), 576)
        for n, r in enumerate(lane):
            f, gr = r // 4, (r // 2) & 1
            pcm[f, ch, gr * 576:(gr + 1) * 576] = out[n]
    return pcm
