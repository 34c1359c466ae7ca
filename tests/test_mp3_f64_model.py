"""The MP3 oracle's whole Layer III chain against the float64 model (tests/_mp3_f64_model.py).

The oracle is the bit-exact target of every MP3 kernel, and tests/test_oracle_kat_mp3.py pins only its building blocks
(dct32, the IMDCTs, the polyphase bank).  Here the stages that join them -- requantisation, mid/side and intensity
stereo, the short-block reorder, alias reduction, frequency inversion and the overlap carried between granules and
frames -- are checked end to end on a corpus of mixed batches that reaches every decision those stages take.  The model
takes the same decisions with different arithmetic (float64, defining formulas), so the two agree to f32 rounding; a
restatement error in the oracle, which the kernels would have copied, shows up as a difference far above it.
"""
import numpy as np
import pytest

from symphonia_b200._native import (F_INTENSITY, F_MID_SIDE, F_MIXED, F_MPEG1, F_PREFLAG, F_SCALEFAC_SCALE, F_SFC_LSB,
                                    MP3_END, MP3_LONG, MP3_RUN_DTYPE, MP3_SHORT, MP3_START)
from tests import _mp3_f64_model as model
from tests import _oracle

# Oracle vs model, max over the corpus of max|oracle - model| / RMS(model) per granule-channel (576 samples): measured
# 7.3e-06 (f32 rounding through the chain; 99th percentile 4.9e-06).  The bound leaves a factor ~2.7 above it.
BOUND = 2e-5
# Every mutation of the model must miss the bound by this factor.
MARGIN = 10.0


# ---- corpus --------------------------------------------------------------------------------------------------------
def concat(parts):
    """Concatenates (units, spectra, runs) batches into one, re-basing first_frame and stream."""
    units = np.concatenate([p[0] for p in parts])
    spectra = np.concatenate([p[1] for p in parts])
    runs, frame0, stream0 = [], 0, 0
    for u, _, r in parts:
        n_streams = int(r["stream"].max()) + 1 if len(r) else 0
        r = r.copy()
        r["first_frame"] += frame0
        r["stream"] += stream0
        runs.append(r)
        frame0 += len(u)
        stream0 += n_streams
    return units, spectra, np.concatenate(runs).astype(MP3_RUN_DTYPE)


def _set_rzero(u, s, rz):
    """rzero of one granule-channel, with the spectrum +0.0 from there on as the Huffman stage leaves it."""
    u["rzero"] = rz
    s[rz:] = 0.0


def _specials(sample_rate_idx, seed):
    """Hand-built edge cases the generator does not reach, on top of one stereo stream of 12 frames."""
    from symphonia_b200 import _native, workloads
    units, spectra, runs = workloads.mp3_batch(1, 12, seed=seed, sample_rate_idx=sample_rate_idx)
    pow43 = _native.mp3_pow43()
    gpf = int(runs["granules_per_frame"][0])
    rng = np.random.default_rng(seed)
    edges = model.LONG_EDGES[sample_rate_idx]

    def frame(f, block_type=None, mixed=False, joint=None):
        """The live units and spectra of frame f, with a common block type and joint-stereo mode."""
        for gr in range(gpf):
            for ch in range(2):
                u = units[f, gr, ch]
                if block_type is not None:
                    u["block_type"] = block_type
                    u["flags"] = (u["flags"] & (0xFF ^ F_MIXED)) | (F_MIXED if mixed else 0)
                if joint is not None:
                    u["flags"] = (u["flags"] & (0xFF ^ F_MID_SIDE ^ F_INTENSITY)) | joint
        return [(units[f, gr, ch], spectra[f, gr, ch]) for gr in range(gpf) for ch in range(2)]

    for u, _ in frame(0):
        u["global_gain"] = 0
    for u, _ in frame(1):
        u["global_gain"] = 255
    for u, s in frame(2):
        _set_rzero(u, s, 0)
    for u, s in frame(3, block_type=MP3_LONG, joint=0):
        u["rzero"] = 576
        s[574:] = pow43[[3, 1]] * np.array([-1, 1])
    for k, (u, s) in enumerate(frame(4, block_type=MP3_LONG)):
        _set_rzero(u, s, min(int(u["rzero"]), edges[15 + k]))  # rzero exactly on a band edge
    # intensity stereo with channel 1 silent (rzero 0): every band is intensity coded, in long, short and mixed blocks,
    # with and without mid/side; intensity positions across the whole range, the illegal ones included
    top = 8 if sample_rate_idx < 3 else 32
    for f, bt, mixed, joint in ((5, MP3_LONG, False, F_INTENSITY), (6, MP3_SHORT, False, F_INTENSITY | F_MID_SIDE),
                                (7, MP3_SHORT, True, F_INTENSITY), (8, MP3_START, False, F_INTENSITY | F_MID_SIDE),
                                (9, MP3_SHORT, True, F_INTENSITY | F_MID_SIDE)):
        for k, (u, s) in enumerate(frame(f, block_type=bt, mixed=mixed, joint=joint)):
            if k % 2:
                _set_rzero(u, s, 0)
                u["scalefacs"][:36] = rng.integers(0, top, size=36)
    for u, _ in frame(10, block_type=MP3_SHORT, mixed=True):
        u["flags"] |= F_PREFLAG  # pretab in the long part of a mixed block (requantize.rs:272)
        u["subblock_gain"] = (7, 0, 7)
    for u, _ in frame(11, block_type=MP3_END):
        u["flags"] |= F_PREFLAG | F_SCALEFAC_SCALE
    return units, spectra, runs


def build_corpus():
    from symphonia_b200 import workloads
    parts = []
    for sr in range(9):  # every sample rate, joint stereo with block switching and mixed blocks
        parts.append(workloads.mp3_batch(3, 10, seed=500 + sr, sample_rate_idx=sr))
    parts.append(workloads.mp3_batch(2, 8, seed=510, channels=1))
    parts.append(workloads.mp3_batch(2, 8, seed=511, sample_rate_idx=5, channels=1))
    parts.append(workloads.mp3_batch(2, 6, seed=512, sample_rate_idx=1, joint=False))
    # MPEG-1 and MPEG-2 granules in which intensity stereo is common, so that both SFC_LSB scales and every joint mode
    # appear in numbers
    for sr in (2, 4, 7):
        u, s, r = workloads.mp3_batch(2, 10, seed=520 + sr, sample_rate_idx=sr)
        rng = np.random.default_rng(520 + sr)
        for f in range(len(u)):
            joint = [F_INTENSITY, F_INTENSITY | F_MID_SIDE, F_MID_SIDE][int(rng.integers(0, 3))]
            u["flags"][f] = (u["flags"][f] & (0xFF ^ F_MID_SIDE ^ F_INTENSITY)) | joint
            rz1 = int(rng.integers(0, 200)) & ~1
            for gr in range(int(r["granules_per_frame"][0])):
                if u["rzero"][f, gr, 1] > rz1:
                    _set_rzero(u[f, gr, 1], s[f, gr, 1], rz1)
        parts.append((u, s, r))
    for sr, seed in ((0, 530), (2, 531), (3, 532), (6, 533), (8, 534)):
        parts.append(_specials(sr, seed))
    return concat(parts)


@pytest.fixture(scope="module")
def corpus(oracle):
    import symphonia_b200 as sb
    units, spectra, runs = build_corpus()
    assert sb.lib().symgpu_mp3_units_check(units.ctypes.data, runs.ctypes.data, len(runs), len(units)) == 0
    rc, want, _ = _oracle.mp3_batch(oracle, units, spectra, runs, int(runs["stream"].max()) + 1)
    assert rc == 0
    return units, spectra, runs, want


def live_rows(units, runs):
    """Row ids (frame * 2 + granule) * 2 + channel of the granule-channels the runs synthesise."""
    rows = []
    for r in runs:
        gpf, n_ch = int(r["granules_per_frame"]) or 2, int(r["channels"]) or 2
        f = np.arange(int(r["first_frame"]), int(r["first_frame"]) + int(r["n_frames"]))
        rows.append(((f[:, None, None] * 2 + np.arange(gpf)[None, :, None]) * 2 + np.arange(n_ch)[None, None, :]).ravel())
    return np.sort(np.concatenate(rows)) if rows else np.zeros(0, dtype=np.int64)


def rel_error(pcm, ref, units, runs):
    """Per live granule-channel: max |pcm - ref| / RMS(ref) over its 576 samples (the absolute error where ref is silent)."""
    rows = live_rows(units, runs)
    f, gr, ch = rows // 4, (rows // 2) & 1, rows & 1
    seg = lambda a: np.asarray(a, dtype=np.float64).reshape(-1, 2, 2, 576)[f, ch, gr]  # noqa: E731  [F,2,1152] -> rows
    p, r = seg(pcm), seg(ref)
    rms = np.sqrt((r ** 2).mean(axis=1))
    err = np.abs(p - r).max(axis=1)
    return np.where(rms > 0, err / np.where(rms > 0, rms, 1.0), err)


# ---- tests ---------------------------------------------------------------------------------------------------------
def test_corpus_reaches_every_case(corpus):
    """The corpus holds every case the model comparison is meant to cover (counted on the live granule-channels)."""
    units, spectra, runs, _ = corpus
    rows = live_rows(units, runs)
    u = units.reshape(-1)[rows]
    fl, bt = u["flags"], u["block_type"]
    assert set(u["sample_rate_idx"]) == set(range(9))
    assert {1, 2} <= set(runs["channels"])
    assert {MP3_LONG, MP3_START, MP3_SHORT, MP3_END} <= set(bt) and ((bt == MP3_SHORT) & (fl & F_MIXED > 0)).any()
    ch1 = u[(rows & 1) == 1]
    for mpeg1, lsbs in ((True, (0,)), (False, (0, F_SFC_LSB))):
        for lsb in lsbs:
            sel = ch1[((ch1["flags"] & F_MPEG1) > 0) == mpeg1]
            if not mpeg1:
                sel = sel[(sel["flags"] & F_SFC_LSB) == lsb]
            modes = {int(m) for m in sel["flags"] & (F_MID_SIDE | F_INTENSITY)}
            assert {F_MID_SIDE, F_INTENSITY, F_MID_SIDE | F_INTENSITY} <= modes, (mpeg1, lsb, modes)
    assert (fl & F_PREFLAG > 0).any() and (fl & F_SCALEFAC_SCALE > 0).any()
    short = u[bt == MP3_SHORT]
    assert (short["subblock_gain"] == 0).any() and (short["subblock_gain"] == 7).any()
    assert {0, 255} <= set(u["global_gain"])
    rz = u["rzero"].astype(int)
    assert (rz == 0).any() and (rz == 576).any()
    interior = {e for sr in range(9) for e in model.LONG_EDGES[sr][1:-1]}
    assert any(int(r) in interior and b == MP3_LONG for r, b in zip(rz, bt))
    is_silent_ch1 = (ch1["flags"] & F_INTENSITY > 0) & (ch1["rzero"] == 0)
    kinds = {(int(b), bool(f & F_MIXED)) for b, f in zip(ch1["block_type"][is_silent_ch1], ch1["flags"][is_silent_ch1])}
    assert {(MP3_LONG, False), (MP3_SHORT, False), (MP3_SHORT, True)} <= kinds
    assert np.abs(corpus[3]).max() > 1e-3


def test_oracle_matches_float64_model(corpus):
    units, spectra, runs, want = corpus
    err = rel_error(want, model.mp3_batch(units, spectra, runs), units, runs)
    assert err.max() < BOUND, f"oracle vs model: {err.max():.3g} of the granule RMS (bound {BOUND:g})"


@pytest.mark.parametrize("mutation", model.MUTATIONS)
def test_model_mutations_miss_the_bound(corpus, mutation):
    """Each plausible restatement bug, made in the model, misses the bound by at least MARGIN on this corpus: the
    corpus reaches the case and the bound is tight enough to see it."""
    units, spectra, runs, want = corpus
    err = rel_error(want, model.mp3_batch(units, spectra, runs, mutation=mutation), units, runs).max()
    assert err > MARGIN * BOUND, f"{mutation}: {err:.3g} is only {err / BOUND:.1f} x the bound"


def test_model_follows_batch_layout(corpus):
    """The model's state is per stream: the same frames in a batch whose runs are shuffled and whose stream indices are
    permuted give the same PCM."""
    units, spectra, runs, _ = corpus
    base = model.mp3_batch(units, spectra, runs)
    rng = np.random.default_rng(3)
    r = runs[rng.permutation(len(runs))].copy()
    r["stream"] = rng.permutation(len(runs))[r["stream"]]
    assert np.array_equal(model.mp3_batch(units, spectra, r), base)
