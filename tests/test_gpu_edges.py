"""The places where the scan kernels could be subtly wrong and random or workload-shaped inputs reach only by chance.

- The fast-phase filter thresholds (build_ktab: WORD r_min >= 63, HALF 31-62, BYTE 15-30, ERODE below, dilated by
  min(r_min, 8)), the exact phase's erosion by min(r_min, 32) and the homopolymer suppression of k 2-16: runs of exactly
  r_min and r_min - 1 matches planted at all 32 bit phases, at strip and tile ends, in tiles with and without N, in a
  load with an exotic letter, under every kernel shape.
- Motif sizes far above the usual 50: up to 65 535 in full mode, the six-divisor sizes 30 030 and 39 270, interval mode at
  -max 1000, and crf_interval_stop at every launch shape (and beyond what it takes: the single-interval path).
- The overflow paths of crf_scan, each asserted taken through crf_scan_stats: the bitonic spill sort, result-buffer
  reruns, the long-run and start queues, the open-row list, and a multi-rank step voided by a long spill list.

Every comparison is exact: against the C oracle, or the numpy statement of the same closed form.  The CPU tests check the
generators themselves (the planted rows are what the oracle reports) and the numpy stop loop against the literal one."""
import os
import random
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))

from crf_b200 import _cabi, api, cli, intervals  # noqa: E402
from oracle import oracle  # noqa: E402
from tests.helpers import ns  # noqa: E402
from tests.test_intervals import _runs_single_copy, _stop_literal, _write_fasta  # noqa: E402

gpu = pytest.mark.gpu

#: every kernel shape: library default, block tiles of 1 / 2 / 4 / 16 words per thread, warp tiles, two strips
SHAPES = [{}, {"words_per_thread": 1}, {"words_per_thread": 2}, {"words_per_thread": 4}, {"words_per_thread": 16},
          {"flags": _cabi.SCAN_WARP_TILES}, {"flags": _cabi.SCAN_TWO_STRIPS}]

ACGT = b"ACGT"
HBIT = {ord("A"): 0, ord("C"): 0, ord("G"): 1, ord("T"): 1}      # the H plane (crf_pack.h): A, C -> 0; G, T -> 1


def r_min(k, min_repeats, min_span):
    """build_ktab's threshold: the fewest matches of M_k a reported run has."""
    b = (min_repeats - 1) * k if min_repeats > 1 else k - 1
    return max(min_span - k, b, 1)


def filter_of(rmin):
    return "WORD" if rmin >= 63 else "HALF" if rmin >= 31 else "BYTE" if rmin >= 15 else "ERODE"


def primitive_unit(rng, k):
    while True:
        u = bytes(rng.choice(ACGT) for _ in range(k))
        if api._is_primitive(u):
            return u


class Planter:
    """A sequence of random ACGT spacers and planted runs of M_k of an exact length.  A run of r matches of motif u
    (len k) at st is u repeated over [st, st + r + k), with S[st-1] != S[st-1+k] and S[st+r] != S[st+r+k]; record 0
    starts at layout position 0 (the load path puts record r at the sum of the earlier (length + max_motif_cap)), so st
    mod 32 is the bit phase of the run's first match.  plants = [(st, end, k, present)]."""

    def __init__(self, seed, n_every=0, exotic=False):
        self.rng = random.Random(seed)
        self.np = np.random.default_rng(seed)
        self.buf = bytearray()
        self.plants = []
        self.n_every, self.last_n, self.exotic = n_every, 0, exotic

    def spacer(self, n):
        sp = bytearray(self.np.choice(np.frombuffer(ACGT, np.uint8), n).tobytes())
        if self.n_every and n >= 6 and len(self.buf) - self.last_n >= self.n_every:
            sp[n // 2] = ord("N")                                    # away from both flanks
            self.last_n = len(self.buf)
        if self.exotic and n >= 6:
            sp[n // 2] = ord("R")                                    # one exotic letter in the whole load
            self.exotic = False
        self.buf += sp

    def plant(self, u, r, phase, word_mod=1, word_rem=0, hflank=True, present=True, left_a=0, right_a=0, n_last=False):
        rng, k = self.rng, len(u)
        lead = max(1, left_a)                                       # the left flank (or its A stretch)
        c = len(self.buf) + 8 + lead
        w = c >> 5
        if (w << 5) + phase < c:
            w += 1
        while w % word_mod != word_rem:
            w += 1
        st = (w << 5) + phase
        self.spacer(st - lead - len(self.buf))
        body = bytearray((u * (r // k + 2))[:r + k])
        if n_last:
            body[k - 1] = ord("N")                                   # the base a run of k-1 matches leaves untested

        def flank(other):
            opts = [b for b in ACGT if b != other and (not hflank or other not in HBIT or HBIT[b] != HBIT[other])]
            return rng.choice(opts)
        if left_a:
            assert u[k - 1] != ord("A")
            if self.buf[-1:] == b"A":
                self.buf[-1] = rng.choice(b"CGT")                    # the stretch is exactly left_a + k - 1 long
            self.buf += b"A" * left_a                                 # S[st-1] = A != S[st-1+k]
        else:
            self.buf.append(flank(body[k - 1]))
        assert len(self.buf) == st
        self.buf += body
        if right_a:
            assert u[r % k] != ord("A")
            self.buf += b"A" * right_a + bytes([rng.choice(b"CGT")])
        else:
            self.buf.append(flank(u[r % k]))
        self.plants.append((st, st + r + k, k, present))

    def seq(self):
        self.spacer(40)
        return bytes(self.buf)


# ---- A. threshold sweep ----------------------------------------------------------------------------------------------

#: r_min values at a filter boundary: every ERODE dilation step, BYTE / ERODE, HALF / BYTE, WORD / HALF, the erosion cap
TARGETS = list(range(1, 9)) + [14, 15, 30, 31, 32, 33, 62, 63]
K_CANDIDATES = [1, 2, 3, 8, 13, 16, 32, 33, 63, 64]
#: (word_mod, word_rem) of the run's first word, in turn: anywhere, the last / first word of a 16-word strip (T = 16;
#: with T = 1 every word is a strip), the last word of a T = 1 tile
POSITIONS = [(1, 0), (16, 15), (16, 0), (256, 255)]


def sweep_settings():
    """{(min_repeats, min_span): [(k, r_min)]} that put r_min(k) on every TARGET for k = 1, some 2 <= k <= 16 and, where
    r_min >= k - 1 allows it (r_min >= 31), k >= 32 and a multiple of 32."""
    out = {}
    for R in TARGETS:
        for k in K_CANDIDATES:
            if k <= R:
                key = (2, R + k if R > k else 1)
            elif k == R + 1:
                key = (1, 1)
            else:
                continue
            assert r_min(k, *key) == R
            out.setdefault(key, []).append(k)
    return {key: sorted(set(ks)) for key, ks in out.items()}


def sweep_sequence(mr, span, ks, variant, seed):
    """Per k of the setting: runs of r_min and r_min - 1 matches at all 32 phases (positions in turn); with
    min_repeats == 1, also runs of k - 1 matches with an N at S[st+k-1] (dropped)."""
    p = Planter(seed, n_every=3000 if variant == "n" else 0, exotic=variant == "exotic")
    rng = random.Random(seed)
    for k in ks:
        R = r_min(k, mr, span)
        hflank = filter_of(R) in ("WORD", "HALF")
        for phase in range(32):
            u = primitive_unit(rng, k)
            for i, r in enumerate((R, R - 1)):
                if r < 1:
                    continue
                wm, wr = POSITIONS[(phase + i) % len(POSITIONS)]
                p.plant(u, r, phase, wm, wr, hflank=hflank or rng.random() < 0.5, present=r == R)
            if mr == 1 and R == k - 1 and k >= 2:
                p.plant(u, R, phase, hflank=hflank, present=False, n_last=True)
    return p.seq(), p.plants


def _kmin(mr):
    """kmin of a sweep scan: 1, or 2 with min_repeats == 1 (where kmin 1 and min_span 1 is refused: every base a row)."""
    return 1 if mr > 1 else 2


def _oracle_rows(seq, kmin, kmax, mr, span):
    fs = ns(min_motif_size=kmin, max_motif_size=kmax, min_repeats=mr, min_span=span)
    if mr == 1:
        return [(s, e, len(m)) for s, e, m in oracle.detect_repeats(seq, fs)]
    s, e, m, _ = oracle.detect_repeats_by_k(seq, fs, arrays=True)
    return list(zip(s.tolist(), e.tolist(), m.tolist()))


def _gpu_rows(ctx, seq, kmin, kmax, mr, span, knobs):
    if mr == 1:       # the host adds position 0's wrap-around candidates: compare what detect_repeats returns
        fs = ns(min_motif_size=kmin, max_motif_size=kmax, min_repeats=mr, min_span=span)
        return [(s, e, len(m)) for s, e, m in api.detect_repeats(seq, fs, device=0, **knobs)]
    with ctx.load(seq, max_motif_cap=kmax) as sq:
        n = sq.scan(kmin, kmax, mr, span, **knobs)
        _, s, e, k = sq.fetch(n)
    return list(zip(s.tolist(), e.tolist(), k.tolist()))


def _check_plants(rows, plants, what):
    have = set((s, e, k) for s, e, k in rows)
    lost = [p for p in plants if p[3] and p[:3] not in have]
    extra = [p for p in plants if not p[3] and p[:3] in have]
    assert not lost and not extra, (what, lost[:5], extra[:5])
    return sum(p[3] for p in plants), sum(not p[3] for p in plants)


def test_sweep_settings_cover_every_boundary():
    cover = {}
    for (mr, span), ks in sweep_settings().items():
        for k in ks:
            cover.setdefault(r_min(k, mr, span), set()).add(k)
    for R in TARGETS:
        ks = cover[R]
        assert 1 in ks and any(2 <= k <= 16 for k in ks), R
        if R >= 31:
            assert any(k >= 32 for k in ks) and any(k % 32 == 0 for k in ks), R


@pytest.mark.parametrize("variant", ["clean", "n", "exotic"])
def test_planted_rows_are_what_the_oracle_reports(variant):
    """CPU: the generator's intended rows -- present at r_min, absent at r_min - 1 -- agree with the C oracle."""
    n_in = n_out = 0
    for i, ((mr, span), ks) in enumerate(sorted(sweep_settings().items())):
        seq, plants = sweep_sequence(mr, span, ks, variant, seed=1000 + i)
        a, b = _check_plants(_oracle_rows(seq, _kmin(mr), max(ks), mr, span), plants, (mr, span))
        n_in, n_out = n_in + a, n_out + b
        assert (b"N" in seq) == (variant == "n" or mr == 1) and (b"R" in seq) == (variant == "exotic")
    assert n_in > 2000 and n_out > 2000


@gpu
@pytest.mark.parametrize("variant", ["clean", "n", "exotic"])
def test_threshold_sweep(variant):
    """Runs of exactly r_min and r_min - 1 matches at every bit phase, every filter boundary, every kernel shape: the
    rows equal the oracle's, and the planted rows are there (r_min) or not (r_min - 1)."""
    ctx = api.get_context(0)
    n_in = 0
    for i, ((mr, span), ks) in enumerate(sorted(sweep_settings().items())):
        seq, plants = sweep_sequence(mr, span, ks, variant, seed=1000 + i)
        kmin, kmax = _kmin(mr), max(ks)
        want = _oracle_rows(seq, kmin, kmax, mr, span)
        for knobs in SHAPES:
            got = _gpu_rows(ctx, seq, kmin, kmax, mr, span, knobs)
            assert got == want, (variant, mr, span, knobs, sorted(set(got) ^ set(want))[:5])
            n_in += _check_plants(got, plants, (mr, span, knobs))[0]
    assert n_in > 10000


@gpu
def test_threshold_runs_in_the_last_strip_of_a_tile():
    """Runs that start in the last word of a tile of every shape (w = 2047 mod 2048 ends the T <= 8 tiles; for T = 16 it is
    the last word of a strip), so their last matches fall into the look-ahead word and the halo."""
    ctx = api.get_context(0)
    n_in = 0
    for R in (14, 15, 30, 31, 62, 63):
        for k in (1, 5):
            span = R + k
            p = Planter(R * 100 + k, n_every=50_000)
            rng = random.Random(R + k)
            for phase in range(0, 32, 3):
                u = primitive_unit(rng, k)
                p.plant(u, R, phase, 2048, 2047, present=True)
                p.plant(u, R - 1, (phase + 1) % 32, 2048, 2047, present=False)
            seq = p.seq()
            want = _oracle_rows(seq, 1, k, 2, span)
            for knobs in SHAPES:
                got = _gpu_rows(ctx, seq, 1, k, 2, span, knobs)
                assert got == want, (R, k, knobs)
                n_in += _check_plants(got, p.plants, (R, k, knobs))[0]
    assert n_in > 800


def homopolymer_sequence(seed, span):
    """Motifs A^(k-1)C, k = 2..20, runs of r_min - 1 .. r_min + k matches; A stretches of 8, 9, 16 and 17 bases (with
    the motif's own k-1) end at the run's start, and begin at its end where the run stops before a C."""
    p = Planter(seed)
    rng = random.Random(seed)
    stretches = [8, 9, 16, 17]
    for k in range(2, 21):
        u = b"A" * (k - 1) + b"C"
        R = r_min(k, 2, span)
        for r in range(R - 1, R + k + 1):
            phases = range(32) if r in (R - 1, R) else [rng.randrange(32)]
            for phase in phases:
                la = [x - (k - 1) for x in stretches if x - (k - 1) >= 1]
                left_a = la[phase % len(la)] if la and phase % 3 else 0
                right_a = 0
                if u[r % k] != ord("A") and phase % 2:
                    ra = [x - (k - 1) for x in stretches if x - (k - 1) >= 1]
                    right_a = ra[phase % len(ra)] if ra else 1
                wm, wr = POSITIONS[phase % len(POSITIONS)]
                p.plant(u, r, phase, wm, wr, hflank=False, present=r >= R, left_a=left_a, right_a=right_a)
    return p.seq(), p.plants


@pytest.mark.parametrize("span", [1, 30])
def test_homopolymer_plants_are_what_the_oracle_reports(span):
    seq, plants = homopolymer_sequence(7 + span, span)
    _check_plants(_oracle_rows(seq, 1, 20, 2, span), plants, span)


@gpu
@pytest.mark.parametrize("span", [1, 30])
def test_homopolymer_suppression_edges(span):
    """k 2-16 count positions that start more than 8 (k <= 8) or 16 equal bases as mismatches in the fast phase; a
    primitive motif never has a run position there, so A^(k-1)C runs must all survive, at every phase."""
    ctx = api.get_context(0)
    seq, plants = homopolymer_sequence(7 + span, span)
    want = _oracle_rows(seq, 1, 20, 2, span)
    for knobs in SHAPES:
        got = _gpu_rows(ctx, seq, 1, 20, 2, span, knobs)
        assert got == want, (span, knobs, sorted(set(got) ^ set(want))[:5])
        _check_plants(got, plants, (span, knobs))


# ---- B. large motif sizes --------------------------------------------------------------------------------------------

def _random_acgt(rng, n):
    return rng.choice(np.frombuffer(ACGT, np.uint8), n).tobytes()


def large_unit_sequence(seed, kmax):
    """~20-60 kbp: units of 1023 ... 4096 bases (those <= kmax) in 2-5 copies (5 copies of 1024: a run past walk_limit),
    small units, spacers."""
    rng = np.random.default_rng(seed)
    r = random.Random(seed)
    parts = [_random_acgt(rng, 500)]
    for size in (1023, 1024, 1025, 2047, 2048, 4096):
        if size > kmax:
            continue
        u = primitive_unit(r, size)
        copies = 5 if size == 1024 else r.randint(2, 3)
        parts += [u * copies + u[:r.randint(0, size - 1)], _random_acgt(rng, r.randint(100, 900))]
    for _ in range(20):
        u = primitive_unit(r, r.randint(1, 300))
        parts += [u * r.randint(2, 6), _random_acgt(rng, r.randint(20, 400))]
    return b"".join(parts)


@gpu
@pytest.mark.parametrize("kmax", [257, 1000, 1024, 1025, 2048, 4097, 65535])
def test_large_motif_sizes_full_mode(kmax):
    ctx = api.get_context(0)
    seq = large_unit_sequence(kmax, kmax)
    shapes = [{}, {"words_per_thread": 1, "walk_limit_words": 2}] + ([{"flags": _cabi.SCAN_WARP_TILES}] if kmax <= 1024 else [])
    for mr in (2, 3):
        want = _oracle_rows(seq, 1, kmax, mr, 9)
        if kmax >= 1024:                                             # a 1024-base unit in 5 copies: past walk_limit
            assert any(k >= 1000 for _, _, k in want) and any(e - s - k > 64 * 32 for s, e, k in want)
        for knobs in shapes:
            assert _gpu_rows(ctx, seq, 1, kmax, mr, 9, knobs) == want, (kmax, mr, knobs)


@gpu
@pytest.mark.parametrize("k,p", [(30030, 13), (39270, 17)])
def test_six_prime_divisor_motif_sizes(k, p):
    """30030 = 2*3*5*7*11*13 and 39270 = 2*3*5*7*11*17 fill all six divisor slots of KEntry: a motif of period k/p (the
    last slot) is dropped, a primitive one of the same length kept."""
    ctx = api.get_context(0)
    r = random.Random(k)
    rng = np.random.default_rng(k)
    v = primitive_unit(r, k // p) * p
    u = primitive_unit(r, k)
    other = lambda b: bytes([next(x for x in ACGT if x != b)])      # noqa: E731 (a mismatch ends the run)
    seq = b"".join([_random_acgt(rng, 700), v * 2 + v[:50], other(v[50]), _random_acgt(rng, 899), other(u[-1]),
                    u * 2 + u[:77], other(u[77]), _random_acgt(rng, 600)])
    want = _oracle_rows(seq, k, k, 2, 1)
    st_u = 700 + len(v) * 2 + 50 + 1 + 900
    assert (st_u, st_u + 2 * k + 77, k) in want and not any(s < 700 + 5 for s, _, _ in want)
    for knobs in ({}, {"words_per_thread": 1}):
        assert _gpu_rows(ctx, seq, k, k, 2, 1, knobs) == want


def hail_sequence(seed, n):
    """~n bases with satellites of period 171 and 997 straddling every 20 kb interval end."""
    rng = np.random.default_rng(seed)
    r = random.Random(seed)
    buf = bytearray(_random_acgt(rng, n))
    for pos in range(20_000, n - 6000, 20_000):
        u = primitive_unit(r, r.choice([171, 997]))
        sat = u * (4 if len(u) > 500 else 9)
        at = pos - r.randint(0, len(sat))
        buf[at:at + len(sat)] = sat
    for _ in range(n // 2000):
        u = primitive_unit(r, r.randint(1, 12))
        at = r.randrange(n - 100)
        s = (u * r.randint(3, 20))[:100]
        buf[at:at + len(s)] = s
    return bytes(buf)


@gpu
def test_interval_mode_at_the_hail_pipeline_setting(tmp_path, monkeypatch, capsys):
    """-min 1 -max 1000 over 20 kb intervals: detect_repeats per interval and detect_repeats_intervals against the
    oracle, --intervals against per-line -i runs."""
    fs = ns(min_motif_size=1, max_motif_size=1000, min_repeats=3, min_span=9)
    seqs = [hail_sequence(1, 200_000), hail_sequence(2, 300_000)]
    n_rows = 0
    for seq in seqs:
        ivs = [(a, min(a + 20_000, len(seq))) for a in range(0, len(seq), 20_000)] + [(19_000, 21_500), (150_123, 161_000)]
        want = []
        for a, b in ivs:
            try:
                want.append(oracle.detect_repeats(seq, intervals._settings_for(fs, a, b)))
            except AssertionError:                                  # prf:77-78 (the last interval may end mid-repeat)
                with pytest.raises(AssertionError):
                    api.detect_repeats(seq, intervals._settings_for(fs, a, b), device=0)
                want.append(None)
        ivs, want = [iv for iv, w in zip(ivs, want) if w is not None], [w for w in want if w is not None]
        assert len(ivs) >= 10 and intervals.detect_repeats_intervals(seq, ivs, fs, device=0) == want
        for (a, b), w in list(zip(ivs, want))[::3]:
            assert api.detect_repeats(seq, intervals._settings_for(fs, a, b), device=0) == w
        assert any(len(m) == 171 for w in want for _, _, m in w) and any(len(m) == 997 for w in want for _, _, m in w)
        n_rows += sum(len(w) for w in want)
    assert n_rows > 300
    monkeypatch.chdir(tmp_path)
    fa = tmp_path / "hail.fa"
    _write_fasta(fa, [("c1", seqs[0].decode()), ("c2", seqs[1].decode())])
    lines = [("c1", 0, 20_000), ("c1", 40_000, 60_000), ("c2", 260_000, 280_000), ("c2", 19_000, 21_500)]
    (tmp_path / "l.bed").write_text("".join(f"{c}\t{a}\t{b}\n" for c, a, b in lines))
    flags = ["-min", "1", "-max", "1000"]
    bed, out = b"", ""
    for c, a, b in lines:
        assert cli.main([str(fa), *flags, "-i", f"{c}:{a}-{b}", "-o", "one"]) == 0
        bed += (tmp_path / "one.bed").read_bytes()
        out += capsys.readouterr().out.replace("Wrote results to one.bed\n", "")
    assert cli.main([str(fa), *flags, "--intervals", str(tmp_path / "l.bed"), "-o", "many"]) == 0
    assert (tmp_path / "many.bed").read_bytes() == bed and bed.count(b"\n") > 20
    assert capsys.readouterr().out == out + "Wrote results to many.bed\n"


_P1, _P2, _B = 2147483647, 2147483629, 1_000_003


def _stop_numpy(s, end_position, kmin, kmax, full_len=None):
    """_stop_literal vectorised over k: tracker k is mid-repeat at t iff the k compares of M_k ending at j = min(t, L-k-1)
    are all ones, i.e. s[j-k+1 : j+1] == s[j+1 : j+k+1] without N (window equality by two polynomial hashes)."""
    W = len(s)
    L = W if full_len is None else full_len
    if end_position >= L - 1:
        return -1
    t_last = L - 1 if W == L else W - 1 - kmax
    a = np.frombuffer(s, np.uint8).astype(np.int64)
    hs = []
    for p in (_P1, _P2):
        h = np.zeros(W + 1, np.int64)
        pw = np.ones(W + 1, np.int64)
        hv, pv = 0, 1
        for i, c in enumerate(a.tolist()):
            hv = (hv * _B + c) % p
            pv = pv * _B % p
            h[i + 1], pw[i + 1] = hv, pv
        hs.append((h, pw, p))
    cn = np.concatenate([[0], np.cumsum(a == ord("N"))])
    ks = np.arange(kmin, kmax + 1, dtype=np.int64)
    for t in range(end_position + 1, t_last + 1):
        j = np.minimum(t, L - ks - 1)
        lo = j - ks + 1
        ok = lo >= 0
        lo, kk = lo[ok], ks[ok]
        mid = cn[lo + kk] == cn[lo]
        for h, pw, p in hs:
            w1 = (h[lo + kk] - h[lo] * pw[kk] % p) % p
            w2 = (h[lo + 2 * kk] - h[lo + kk] * pw[kk] % p) % p
            mid &= w1 == w2
        if not mid.any():
            return t
    return -1 if W == L else -2


def test_numpy_stop_loop_equals_the_literal_loop():
    rng = random.Random(5)
    n = 0
    for _ in range(300):
        kmin = rng.randint(1, 6)
        kmax = kmin + rng.randint(0, 40)
        f = rng.randint(1, 400)
        s = bytes(rng.choice(b"ACGTN" if rng.random() < 0.3 else b"AC") for _ in range(f))
        if rng.random() < 0.6:
            u = bytes(rng.choice(ACGT) for _ in range(rng.randint(1, kmax + 2)))
            p = rng.randint(0, f)
            s = (s[:p] + u * rng.randint(2, 30) + s[p:])[:max(f, 1)]
            f = len(s)
        e = rng.choice([rng.randint(0, f), max(0, f - rng.randint(0, 2 * kmax + 2))])
        w = f if rng.random() < 0.6 else rng.randint(0, f)
        want = _stop_literal(s[:w], e, kmin, kmax, f)
        assert _stop_numpy(s[:w], e, kmin, kmax, f) == want, (s, w, e, kmin, kmax)
        n += want >= 0
    assert n > 80


def _optin_nk():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin // 4


def stop_records(seed, kmax, count):
    """Records of kmax/2 .. 2.2 kmax bases with a satellite of a unit of kmax/2 .. kmax bases (2 copies + a tail) and small
    tandem repeats; the interval ends inside the satellite's mid-repeat range or near the record's end."""
    rng = np.random.default_rng(seed)
    r = random.Random(seed)
    recs, E, W = [], [], []
    for i in range(count):
        n = r.randint(max(kmax // 2, 64), int(2.2 * kmax) + 200)
        buf = bytearray(_random_acgt(rng, n))
        U = r.randint(max(1, kmax // 2), kmax)
        tail = r.randint(1, 150)
        st = r.randint(0, max(0, n - 2 * U - tail - 1))
        if st + 2 * U + tail <= n:
            u = _random_acgt(rng, U)
            buf[st:st + 2 * U + tail] = (u * 3)[:2 * U + tail]
            e = st + U - 1 + r.randint(-3, tail)
        else:
            e = r.randint(0, n)
        for _ in range(3):
            v = _random_acgt(rng, r.randint(1, 20))
            at = r.randrange(n)
            piece = v * r.randint(2, 10)
            buf[at:at + len(piece)] = piece[:n - at]
        if i % 5 == 4:
            e = max(0, n - r.randint(0, 2 * kmax))                   # a tracker that stopped before e + 1
        if i % 7 == 3:
            buf[max(0, e - 5):e + 5] = b"N" * len(buf[max(0, e - 5):e + 5])
        recs.append(bytes(buf))
        E.append(max(0, min(e, n)))
        W.append(n if i % 4 else r.randint(0, n))                   # every fourth: a truncated prefix
    return recs, E, W


@gpu
def test_interval_stop_kernel_at_every_launch_shape():
    """crf_interval_stop for nk = kmax - kmin + 1 at each change of its launch shape: 4 warps up to 3072 motif sizes, then
    2, then 1; above 12 288, more than 48 KB of shared memory; up to what the device gives one block -- against the
    literal loop (vectorised).  One more motif size is refused."""
    optin = _optin_nk()
    assert optin >= _cabi.STOP_MAX_MOTIF_SIZES, "the device gives a block less shared memory than crf_interval_stop assumes"
    ctx = api.get_context(0)
    n_dec = n_und = 0
    for nk in (1000, 3072, 3073, 6144, 6145, 12288, 12289, min(optin, _cabi.STOP_MAX_MOTIF_SIZES)):
        kmin = 1 if nk % 2 else 3
        kmax = kmin + nk - 1
        recs, E, W = stop_records(nk, kmax, 10)
        F = [len(x) for x in recs]
        starts = np.cumsum([0] + F[:-1])
        planes = _cabi.pack_ascii(b"".join(recs)).with_runs()
        want = [_stop_numpy(x[:w], e, kmin, kmax, f) for x, w, e, f in zip(recs, W, E, F)]
        with ctx.load_packed(planes, max_motif_cap=kmax, ranges=(starts, W, None, None)) as seq:
            got = seq.interval_stop(kmin, kmax, E, F)
        assert got.tolist() == want, (nk, got.tolist(), want)
        n_dec += sum(x >= 0 for x in want)
        n_und += sum(x == -2 for x in want)
    assert n_dec > 30 and n_und > 3
    nk = _cabi.STOP_MAX_MOTIF_SIZES + 1
    with ctx.load_packed(_cabi.pack_ascii(b"ACGT" * 100).with_runs(), max_motif_cap=nk,
                         ranges=([0], [400], None, None)) as seq:
        with pytest.raises(NotImplementedError):
            seq.interval_stop(1, nk, [10], [400])


def test_more_motif_sizes_than_the_stop_kernel_takes_go_to_the_single_interval_path(monkeypatch):
    """CPU: run_intervals hands every interval to single() when crf_interval_stop would refuse the motif range."""
    seen = []
    real = intervals.scan_intervals

    def spy(ctx, planes, src, *a, **kw):
        seen.append(len(src))
        return real(ctx, planes, src, *a, **kw)
    monkeypatch.setattr(intervals, "scan_intervals", spy)
    monkeypatch.setattr(api, "get_context", lambda device=None: None)
    planes = _cabi.pack_ascii(b"ACGT" * 50).with_runs()
    fs = ns(min_motif_size=2, max_motif_size=2 + _cabi.STOP_MAX_MOTIF_SIZES, min_repeats=3, min_span=9)
    outcome, *_ = intervals.run_intervals(planes, 0, 200, [0, 10, 50], [100, 20, 200], fs, single=lambda i: [("s", i)])
    assert outcome == [[("s", 0)], [("s", 1)], [("s", 2)]] and seen == [0]
    assert intervals.last_stats["fallback"] == 3


@gpu
def test_detect_repeats_intervals_beyond_the_stop_kernel(tmp_path, monkeypatch, capsys):
    """More motif sizes than crf_interval_stop takes (-min 1 -max 65535): detect_repeats_intervals equals per-interval
    detect_repeats, and --intervals the -i runs (both used to raise NotImplementedError)."""
    seq = hail_sequence(9, 70_000)
    fs = ns(min_motif_size=1, max_motif_size=65535, min_repeats=3, min_span=9)
    ivs = [(0, 20_000), (19_000, 21_500), (40_000, 60_000)]
    want = [api.detect_repeats(seq, intervals._settings_for(fs, a, b), device=0) for a, b in ivs]
    assert intervals.detect_repeats_intervals(seq, ivs, fs, device=0) == want and sum(map(len, want)) > 20
    monkeypatch.chdir(tmp_path)
    fa = tmp_path / "x.fa"
    _write_fasta(fa, [("c", seq.decode())])
    (tmp_path / "l.bed").write_text("".join(f"c\t{a}\t{b}\n" for a, b in ivs))
    flags = ["-min", "1", "-max", "65535"]
    bed = b""
    for a, b in ivs:
        assert cli.main([str(fa), *flags, "-i", f"c:{a}-{b}", "-o", "one"]) == 0
        bed += (tmp_path / "one.bed").read_bytes()
    capsys.readouterr()
    assert cli.main([str(fa), *flags, "--intervals", str(tmp_path / "l.bed"), "-o", "many"]) == 0
    assert (tmp_path / "many.bed").read_bytes() == bed


# ---- C. overflow paths -----------------------------------------------------------------------------------------------

def _oracle_cols(seq, kmin, kmax, mr, span):
    s, e, m, _ = oracle.detect_repeats_by_k(seq, ns(min_motif_size=kmin, max_motif_size=kmax, min_repeats=mr,
                                                       min_span=span), arrays=True)
    return s, e, m


def _same(got, want):
    return all(np.array_equal(np.asarray(a).astype(np.int64), np.asarray(b).astype(np.int64)) for a, b in zip(got, want))


@gpu
def test_spill_sort_and_result_reruns():
    """--min-repeats 2 --min-span 1 makes every AA a row: every tile spills, past SPILL_SMALL (global bitonic sort, gather
    again).  min_repeats == 1 adds the second single-copy filter pass.  result_cap = 1 forces reruns, once as a
    captured graph on a small input, then again on the grown buffers."""
    ctx = api.get_context(0)
    seq = _random_acgt(np.random.default_rng(3), 300_000)
    want = _oracle_cols(seq, 1, 8, 2, 1)
    with ctx.load(seq, max_motif_cap=8) as sq:
        for knobs in ({"result_cap": 1}, {}):
            n = sq.scan(1, 8, 2, 1, **knobs)
            st = sq.stats()
            assert st.n_spilled > 4096 and _same(sq.fetch(n)[1:], want)
            assert st.reruns >= 1 or knobs == {}
        n = sq.scan(2, 8, 1, 1)
        assert sq.stats().n_spilled > 4096
        assert _same(sq.fetch(n)[1:], _runs_single_copy(seq, 2, 8, 1))
    small = seq[:20_000]
    want = _oracle_cols(small, 1, 8, 3, 9)
    with ctx.load(small, max_motif_cap=8) as sq:
        for rep in range(2):
            n = sq.scan(1, 8, 3, 9, result_cap=1)
            assert (sq.stats().reruns >= 1) == (rep == 0) and _same(sq.fetch(n)[1:], want)
    fs = ns(min_motif_size=1, max_motif_size=8, min_repeats=2, min_span=1)
    ivs = [(0, 150_000), (100_000, 300_000), (299_000, 300_000)]
    assert intervals.detect_repeats_intervals(seq, ivs, fs, device=0) == \
        [oracle.detect_repeats(seq, intervals._settings_for(fs, a, b)) for a, b in ivs]
    fs1 = ns(min_motif_size=2, max_motif_size=8, min_repeats=1, min_span=1)
    assert api.detect_repeats(seq[:120_000], fs1, device=0) == oracle.detect_repeats(seq[:120_000], fs1)


@gpu
def test_long_run_queue_full():
    """One 8 kbp tile (T = 1) with 40 primitive runs longer than walk_limit_words = 1: the tile's queue for the block walker
    (LONGCAP = 32) fills, and handle_start walks the rest alone."""
    ctx = api.get_context(0)
    r = random.Random(4)
    rng = np.random.default_rng(4)
    parts = []
    for i in range(40):
        u = primitive_unit(r, r.randint(2, 5))
        parts += [_random_acgt(rng, 20), u * (130 // len(u)), b"N"]
    seq = b"".join(parts)
    assert len(seq) <= 8192
    want = _oracle_cols(seq, 1, 10, 3, 9)
    assert ((want[1] - want[2] - want[0]) > 96).sum() > 32
    with ctx.load(seq, max_motif_cap=10) as sq:
        n = sq.scan(1, 10, 3, 9, words_per_thread=1, walk_limit_words=1)
        st = sq.stats()
        assert st.n_tiles == 1 and st.n_long == 32 and _same(sq.fetch(n)[1:], want)


@gpu
def test_start_queue_full():
    """k 1-4 with r_min = k on AAC-like text at T = 16: more than two run starts per (strip, k) and more than STARTQ_CAP =
    512 beyond those per tile (counted from M_k here), so handle_start runs in the exact phase."""
    ctx = api.get_context(0)
    r = random.Random(6)
    seq = b"".join(r.choice([b"AAC", b"AAG", b"CCT", b"GGA", b"TTC", b"ACAC", b"AGAG"]) for _ in range(60_000))
    a = np.frombuffer(seq, np.uint8)
    over = np.zeros(len(seq) // 131072 + 1, np.int64)
    for k in range(1, 5):
        m = np.concatenate([[0], (a[:-k] == a[k:]).astype(np.int8), [0]])
        edge = np.diff(m)
        st, en = np.flatnonzero(edge == 1), np.flatnonzero(edge == -1)
        st = st[en - st >= min(k, 32)]
        per_strip = np.bincount(st // 512)
        assert per_strip.max() > 2
        tiles = np.arange(per_strip.size) * 512 // 131072
        np.add.at(over, tiles, np.maximum(per_strip - 2, 0))
    assert over.max() > 512
    want = _oracle_cols(seq, 1, 4, 2, 1)
    with ctx.load(seq, max_motif_cap=4) as sq:
        n = sq.scan(1, 4, 2, 1, words_per_thread=16)
        assert _same(sq.fetch(n)[1:], want)


@gpu
def test_open_row_list_grows():
    """300+ records loaded as ranges, all open-ended, each ending in a repeat: more than OPEN_CAP_INITIAL = 256 open rows;
    the list grows and fetch_open returns every one with its end."""
    ctx = api.get_context(0)
    r = random.Random(8)
    rng = np.random.default_rng(8)
    recs = []
    for _ in range(320):
        u = primitive_unit(r, r.randint(1, 6))
        recs.append(_random_acgt(rng, r.randint(30, 200)) + b"G" + u * r.randint(10, 14))
    src = b"".join(recs)
    starts = np.cumsum([0] + [len(x) for x in recs[:-1]])
    want = set()
    for i, x in enumerate(recs):
        s, e, m = _oracle_cols(x, 1, 8, 3, 9)
        want |= {(i, a, b, c) for a, b, c in zip(s.tolist(), e.tolist(), m.tolist()) if b == len(x)}
    assert len(want) > 256
    with ctx.load_ranges(src, starts, [len(x) for x in recs], max_motif_cap=8) as sq:
        sq.set_output_map(open_ended=np.ones(len(recs), np.uint8))
        n = sq.scan(1, 8, 3, 9)
        rows = sq.fetch(n)
        assert sq.stats().n_open == len(want)
        op = sq.fetch_open(cap=1024)
    assert {tuple(x) for x in op[:, 1:].tolist()} == want
    assert all(rows[2][i] == e for i, _, _, e, _ in op.tolist())


@gpu
def test_multi_rank_step_voided_by_a_long_spill_list():
    """Two loopback ranks whose spill lists exceed SPILL_SMALL: publish_kernel voids the asynchronous step and every rank
    repeats it through crf_scan; the gathered rows equal the single scan."""
    from crf_b200 import multi
    rng = np.random.default_rng(12)
    bases = np.frombuffer(_random_acgt(rng, 1_200_000), np.uint8).copy()
    offsets = np.array([0, 400_000, 1_200_000], np.uint64)
    ctx = api.get_context(0)
    with ctx.load(bases, offsets, max_motif_cap=8) as sq:
        n = sq.scan(1, 8, 2, 1)
        assert sq.stats().n_spilled > 2 * 4096
        want = sq.fetch(n)
    got = multi.scan_on_devices([0, 0], bases, offsets[:-1], np.diff(offsets.astype(np.int64)), 1, 8, 2, 1,
                                chunk=1 << 18, halo=1 << 12, timeout_s=60)
    assert _same(got, want)
