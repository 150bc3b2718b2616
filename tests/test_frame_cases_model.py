"""Crafted framing cases and a plain restatement of streaming framing (CPU).

Framing turns a capture's bit and quiet planes into its result: the first 1,0,0,0 terminator (afskmodem.py:362-366,
__scanTraining :386-390), the first quiet window at or after k0 (:372-378), then Hamming(7,4) over 14-window groups
(:145-163, :393-399).  It runs in k_frame<T,W> (three variants), frame_capture_warp (k_frame_warp and the fused
schedule's frame jobs), k_stream_frame (payload retention) and the bits-mode final framing.  Real transmissions almost
never reach the inputs where their masks and step loops go wrong, so this file builds them:

  * framed_capture turns any decision and quiet sequence into audio that demodulates to exactly that sequence: `lead`
    zero frames, the reference's training cycle as windows 0 and 1 (so the oracle's first strict minimum, its clock,
    is `lead`), then the mark tone for a 1 and the space tone for a 0, at full scale when loud and at +-600 when quiet
    (the limiter still sees the tone; mean |x| = 600 < amp_end), then 1 .. bf frames, so that K is exact.
  * frame_cases names case families: T terminator position, E end of capture, Q first quiet window, H payload (k0 and
    nbits residues, all 128 codewords at every codeword slot of a 56-bit quad), L long captures; with the search-step
    edges of each framing path (STEPS).
  * stream_job restates one k_stream_frame job on packed plane words, reading the previous word only where the kernel
    does (c < 32 w + 3) and no word below those a channel keeps.  Chained over cuts of a sequence into increasing
    window limits it must give whole-sequence framing.

tests/test_gpu_framing.py compares every framing path with these references on the GPU."""
import functools

import numpy as np
import pytest

from oracle import oracle as O
from test_demod_planes_model import SYNC, bit_frames, frame, ref_planes
from test_frame_model import LUT, kernel_model
from test_stream_payload_model import ENDED, PAYLOAD, TRAIN, decode_bytes, frame_whole

AMP_END = 14000
QUIET = 600                                        # sample magnitude of a quiet window
BAUDS = (12000, 6000, 2400, 1200, 300)             # 4, 8, 20, 40 and 160 samples per bit
FAMILIES = ("T", "E", "Q", "H", "L")
# plane words per search step, as windows: frame_capture_warp 32 lanes x 8 words, k_frame<128,4> and <512,8>,
# k_stream_frame 32 lanes x 1 word
STEPS = {"warp": 8192, "cta128": 16384, "cta512": 131072, "stream": 1024}
MAX_WINDOWS = {"warp": 262144, "cta128": None, "cta512": None, "stream": None}     # afsk_rx.cu kFrameWarpMaxWindows
BATCH_PATHS = ("warp", "cta128", "cta512")
# the bauds whose step edges are crafted (long steps only where the captures stay small)
STEP_BAUDS = {"warp": (12000, 6000, 2400), "cta128": (12000, 6000, 2400), "cta512": (12000,),
              "stream": BAUDS}
D = range(-3, 4)                                    # offsets around an edge


@functools.lru_cache(maxsize=None)
def _tones(baud):
    return O.tone("mark", baud).astype(np.int64), O.tone("space", baud).astype(np.int64)


def framed_capture(baud, bits, quiet, lead, tail, amp_end=AMP_END):
    """int16 audio whose windows at clock `lead` decide exactly (bits, quiet); see the module docstring"""
    bf = bit_frames(baud)
    bits, quiet = np.asarray(bits, bool), np.asarray(quiet, bool)
    K = len(bits)
    assert K >= 2 and bits[0] and not bits[1] and not quiet[:2].any(), "windows 0, 1 are the training cycle"
    assert 0 <= lead < SYNC - 2 * bf and 1 <= tail <= bf
    mark, space = _tones(baud)
    W = np.where(bits[:, None], mark, space)
    W = np.where(quiet[:, None], np.sign(W) * QUIET, W)
    x = np.concatenate([np.zeros(lead, np.int64), W.ravel(), np.zeros(tail, np.int64)]).astype(np.int16)
    assert len(x) >= SYNC, (baud, K, lead)
    o = O.rx_decode(x, baud, amp_end, want_bits=True)
    assert o["clock"] == lead, (baud, o["clock"], lead)
    rb, rq = ref_planes(x, baud, lead, amp_end)
    assert np.array_equal(rb, bits) and np.array_equal(rq, quiet), baud
    train_end, coded = frame(bits, quiet, lead, bf)
    assert o["train_end"] == train_end and np.array_equal(o["bits"], coded), baud
    assert (o["status"] == O.ST_NO_DATA) == (len(coded) == 0) and o["data"] == decode_bytes(coded), baud
    return x


# ---------------------------------------------------------------- sequences ---------------------------------------

TRAIN_KINDS = ("alt", "ones", "near", "rand")


def training(n, kind, rng):
    """n >= 1 decided windows starting 1,0 (the training cycle) without a terminator: alternating, a stuck 1, the
    near miss 1,0,0 repeated, or random with zero runs of at most two"""
    if kind == "alt":
        t = np.tile([1, 0], n // 2 + 1)
    elif kind == "ones":
        t = np.concatenate([[1, 0], np.ones(n, np.int64)])
    elif kind == "near":
        t = np.tile([1, 0, 0], n // 3 + 1)
    else:
        t = [1, 0]
        while len(t) < n:
            t += [1] + [0] * int(rng.integers(0, 3))
        t = np.array(t)
    return np.asarray(t[:n], np.uint8)


def sequence(K, k_t, rng, kind="alt", quiet=(), payload=None):
    """K windows: training, the terminator 1,0,0,0 ending at window k_t (None: none), then payload bits (random, or
    given and then random); quiet windows at `quiet`"""
    assert k_t is None or k_t == 3 or k_t >= 5, k_t              # windows 0, 1 are 1, 0: no terminator ends at 4
    if k_t is None:
        bits = training(K, kind, rng)
    else:
        head = training(k_t - 3, kind, rng) if k_t > 3 else np.zeros(0, np.uint8)
        body = rng.integers(0, 2, max(K - k_t - 1, 0)).astype(np.uint8)
        if payload is not None:
            body[:len(payload)] = payload[:len(body)]
        bits = np.concatenate([head, [1, 0, 0, 0], body]).astype(np.uint8)[:K]
    q = np.zeros(K, bool)
    q[[k for k in quiet if 2 <= k < K]] = True
    return bits.astype(bool), q


def codeword_payload(rot):
    """1024 codewords: every 7-bit codeword at every slot n0 .. n7 of a 56-bit quad (even slots a byte's high nibble,
    odd slots its low one); bit i of a codeword is received i-th"""
    j = np.arange(1024)
    cw = (j // 8 + 37 * (j % 8) + rot) % 128
    return ((cw[:, None] >> np.arange(7)) & 1).astype(np.uint8).ravel()


class Case:
    """one crafted capture: family, name, tags (what it was built to reach), decided windows and framing layout"""

    def __init__(self, family, name, baud, bits, quiet, rng, tags=(), lead=None, tail=None):
        self.family, self.name, self.baud = family, name, baud
        self.bits, self.quiet = np.asarray(bits, bool), np.asarray(quiet, bool)
        self.tags = frozenset(tags)
        bf = bit_frames(baud)
        K = len(self.bits)
        self.tail = int(rng.integers(1, bf + 1)) if tail is None else tail
        lo = max(0, SYNC - K * bf - self.tail)
        assert lo < SYNC - 2 * bf, (name, baud, K)
        self.lead = int(rng.integers(lo, SYNC - 2 * bf)) if lead is None else lead

    @property
    def K(self):
        return len(self.bits)

    @property
    def kmax(self):
        """the capture's windows at clock 0, by which a decode picks its framing kernel (afsk_rx.cu launch_frame)"""
        bf = bit_frames(self.baud)
        return -(-(self.lead + self.K * bf + self.tail - bf) // bf)

    def audio(self):
        return framed_capture(self.baud, self.bits, self.quiet, self.lead, self.tail)

    def reference(self):
        """(status, clock, train_end, nbits, nbytes, payload) by the reference's framing of the crafted windows"""
        r, data = frame_whole(self.bits, self.quiet, self.K, self.lead, bit_frames(self.baud))
        return r + (data,)

    def layout(self):
        k0, nbits, _ = kernel_model(self.bits.astype(np.uint8), self.quiet.astype(np.uint8))
        return k0, nbits


def frame_cases(baud, variant):
    """the named cases at this baud for framing path `variant` (STEPS): the families every path shares, and the T / Q
    cases at the path's search-step edges (where STEP_BAUDS crafts them)"""
    rng = np.random.default_rng([baud, list(STEPS).index(variant)])
    bi = BAUDS.index(baud)
    out = []

    def add(fam, name, bits, quiet, *tags, lead=None, tail=None):
        out.append(Case(fam, f"{fam}:{name}", baud, bits, quiet, rng, tags, lead, tail))

    kinds = TRAIN_KINDS
    # T: the terminator at k_t = 3, at every residue mod 32 (32 + r: the windows straddling a word among them), over
    # every kind of training
    add("T", "k3", *sequence(60, 3, rng), "k_t=3")
    for r in range(32):
        k_t = 32 * (1 + (r + bi) % 3) + r
        if k_t == 4:
            continue
        add("T", f"r{r}", *sequence(k_t + 40 + r, k_t, rng, kinds[r % 4]), f"kt%32={k_t % 32}", f"train={kinds[r % 4]}")
    # E: no terminator, the last windows ...1 / ...1,0 / ...1,0,0, K at every residue mod 32; terminators at K - 1,
    # K - 2, K - 4
    for r in range(32):
        K = 64 + 32 * (bi % 2) + r
        end = [[1], [1, 0], [1, 0, 0]][r % 3]
        bits = np.concatenate([training(K - len(end), kinds[r % 4], rng), end]).astype(bool)
        add("E", f"end{len(end)}K{r}", bits, np.zeros(K, bool), f"K%32={K % 32}", f"end={len(end)}")
    for e in (1, 2, 4):
        for K in (67, 96, 129):
            add("E", f"term@K-{e}:{K}", *sequence(K, K - e, rng), f"term@K-{e}")
    # Q: quiet windows only before k0 (earlier words, the word of k0, window k0 - 1); the first quiet window at k0 + r
    # for every r mod 14, at K - 1; none
    for k_t in (70, 77, 95, 100):
        k0 = k_t + 1
        before = [int(k) for k in rng.choice(np.arange(2, 32 * (k0 >> 5)), 4, replace=False)]
        inword = list(range(32 * (k0 >> 5), k0))
        add("Q", f"before{k_t}", *sequence(k_t + 90, k_t, rng, quiet=before + inword), "quiet<k0",
            *(["quiet in k0 word", "quiet@k0-1"] if inword else []))
    for r in range(28):
        k_t = 40 + 9 * r
        add("Q", f"at{r}", *sequence(k_t + r + 70, k_t, rng, quiet=[k_t + 1 + r, k_t + 5 + r]), f"q-k0%14={r % 14}")
    add("Q", "atK-1", *sequence(120, 50, rng, quiet=[119]), "q@K-1")
    add("Q", "none", *sequence(120, 50, rng), "no quiet")
    # H: k0 at every residue mod 32; nbits at every residue mod 56 (0 .. 3 tail bytes after the quads); nbits 1 .. 13;
    # every codeword at every quad slot
    for r in range(32):
        k_t = 64 + r - 1
        nbits = 56 * int(rng.integers(1, 6)) + (7 * r + bi) % 56
        end = "quiet" if r % 2 else "K"
        K = k_t + 1 + nbits + (6 if end == "quiet" else 0)
        add("H", f"k0r{r}", *sequence(K, k_t, rng, kinds[r % 4], quiet=[k_t + 1 + nbits] if end == "quiet" else []),
            f"k0%32={(k_t + 1) % 32}")
    for r in range(56):
        k_t = 40 + (5 * r + bi) % 32
        nbits = 56 * (r % 3) + r
        add("H", f"nb{r}", *sequence(k_t + 1 + nbits + 3, k_t, rng, quiet=[k_t + 1 + nbits]), f"nbits%56={r}")
    for n in range(1, 14):
        add("H", f"short{n}", *sequence(60 + n + 9, 60, rng, quiet=[61 + n]), f"nbits={n}")
    for rot in range(2 if bi < 3 else 1):
        k_t = 100 + 3 * bi + rot * 4
        pay = codeword_payload(37 * rot + bi)
        add("H", f"cw{rot}", *sequence(k_t + 1 + len(pay) + 8, k_t, rng, payload=pay, quiet=[k_t + 1 + len(pay)]), "codewords")
    # T / Q at this path's search-step edges (the quiet search starts at the word of k0)
    if baud in STEP_BAUDS[variant]:
        st = STEPS[variant]
        for m in (1, 2) if st <= 8192 else (1,):
            for d in D:
                add("T", f"step{st}x{m}{d:+d}", *sequence(m * st + d + 50, m * st + d, rng, kinds[d % 4]), f"kt=step{d:+d}")
                k_t = 37 + 5 * (d + 3)
                q = 32 * ((k_t + 1) >> 5) + m * st + d
                add("Q", f"step{st}x{m}{d:+d}", *sequence(q + 40, k_t, rng, quiet=[q]), f"q=step{d:+d}")
    # L: exactly 262,144 and 262,145 windows at 12000 baud, as the decode counts them to pick a kernel (at clock 0:
    # the clock is lead = 0, or 1 frame, which adds one); longer ones with the terminator and the first quiet window
    # near 131072-window steps (built once, with the longest path's cases)
    if baud == 12000 and variant == "cta512":
        for K, lead in ((262144, 0), (262145, 0), (262144, 1)):
            add("L", f"K{K}lead{lead}", *sequence(K, 1000 + K % 2, rng, quiet=[K - 2] if lead else []),
                f"K={K + lead}", lead=lead, tail=bit_frames(baud))
        for d in (-2, 0, 3):
            k_t = 131072 + d
            q = 32 * ((k_t + 1) >> 5) + 131072 - d
            add("L", f"long{d:+d}", *sequence(262144 + 700 + d, k_t, rng, quiet=[q]), "K>262144", f"kt=131072{d:+d}")
    return out


@functools.lru_cache(maxsize=1)
def batch_cases():
    """the cases of the batch paths at every baud: the shared families once, every path's step edges, L"""
    seen, out = set(), []
    for v in BATCH_PATHS:
        for b in BAUDS:
            for c in frame_cases(b, v):
                if (b, c.name) not in seen:
                    seen.add((b, c.name))
                    out.append(c)
    return out


@functools.lru_cache(maxsize=None)
def path_cases(variant):
    """every case that runs through path `variant`: for a batch path the batch's captures within its window limit,
    for k_stream_frame the stream cases of every baud"""
    if variant == "stream":
        return [c for b in BAUDS for c in frame_cases(b, "stream")]
    lim = MAX_WINDOWS[variant]
    return [c for c in batch_cases() if lim is None or c.kmax <= lim]


# ---------------------------------------------------------------- k_stream_frame restatement ----------------------

M32 = 0xFFFFFFFF


def pack_words(bits, n_words):
    """windows -> little-endian 32-bit plane words (window 32 j + t in bit t of word j), zero past the last window"""
    b = np.zeros(32 * n_words, np.uint8)
    b[:len(bits)] = bits
    return np.packbits(b.reshape(-1, 32), axis=1, bitorder="little").view("<u4").reshape(-1).astype(np.int64)


def term_masks(prev, cur):
    fl = lambda s: ((cur << s) | (prev >> (32 - s))) & M32        # noqa: E731  __funnelshift_l
    return fl(3) & ~fl(2) & ~fl(1) & ~cur & M32


def _first(M, w0):
    """the first set bit over words w0, w0 + 1, ... of masks M, as a window (None: none)"""
    nz = np.flatnonzero(M)
    if not len(nz):
        return None
    m = int(M[nz[0]])
    return 32 * (w0 + int(nz[0])) + (m & -m).bit_length() - 1


def stream_job(bw, qw, st, k_end, kept, reads=None):
    """One k_stream_frame job over plane words bw / qw (the words below `kept` are not the channel's: reading one is
    an error): FrameState st = dict(consumed, k0, k1, nbytes, phase) framed over windows [consumed, k_end).  -> (new
    state, {byte index: byte}).  reads (a list) receives what the job read, for the quota checks."""
    F = dict(st)
    c, K = F["consumed"], k_end
    got = {}
    if F["phase"] == TRAIN and c < K:
        w = np.arange(c >> 5, ((K - 1) >> 5) + 1)
        assert w[0] >= kept, (c, kept)
        cur = bw[w]
        use_prev = (w > 0) & (c < 32 * w + 3)                        # the predecessor only where its bits enter windows >= c
        assert (w[use_prev] - 1 >= kept).all(), (c, kept)
        prev = np.where(use_prev, bw[np.maximum(w - 1, 0)], 0)
        M = term_masks(prev, cur)
        M[0] &= ~((1 << (c & 31)) - 1) & M32
        rem = K - 32 * w
        M = np.where(rem < 32, M & ((1 << np.clip(rem, 0, 32)) - 1), M)
        kt = _first(M, int(w[0]))
        if kt is None:
            c = K
        else:
            F["phase"], F["k0"] = PAYLOAD, kt + 1
            if reads is not None:
                reads.append(("term", c, kt))
            c = F["k0"]
    if F["phase"] == PAYLOAD:
        kq = None
        if c < K:
            w = np.arange(c >> 5, ((K - 1) >> 5) + 1)
            assert w[0] >= kept, (c, kept)
            M = qw[w].copy()
            M[0] &= ~((1 << (c & 31)) - 1) & M32
            rem = K - 32 * w
            M = np.where(rem < 32, M & ((1 << np.clip(rem, 0, 32)) - 1), M)
            kq = _first(M, int(w[0]))
        if kq is not None:
            F["phase"], F["k1"] = ENDED, kq
            if reads is not None:
                reads.append(("quiet", c, kq, K))
        c = max(c, K)
        lim = kq if kq is not None else c
        nb = (lim - F["k0"]) // 14
        if nb > F["nbytes"]:
            i = np.arange(F["nbytes"], nb)
            pos = F["k0"] + 14 * i
            assert (pos >> 5).min() >= kept, (F, kept)
            v = (((bw[(pos >> 5) + 1] << 32) | bw[pos >> 5]) >> (pos & 31)) & 0x3FFF
            lut = np.array(LUT, np.int64)
            by = (lut[v & 0x7F] << 4) | lut[(v >> 7) & 0x7F]
            got = dict(zip(i.tolist(), by.tolist()))
        if reads is not None and kq is None and (lim - F["k0"]) % 14:
            reads.append(("cut byte", lim))
        F["nbytes"] = max(F["nbytes"], nb)
    F["consumed"] = max(F["consumed"], c)
    return F, got


def fresh_state():
    return dict(consumed=0, k0=0, k1=0, nbytes=0, phase=TRAIN)


def kept_word(F):
    """the first plane word a channel keeps for a recording in state F (streams_bits: the word of window consumed - 3
    in training, of the next incomplete byte in payload)"""
    return (F["k0"] + 14 * F["nbytes"]) // 32 if F["phase"] == PAYLOAD else max(F["consumed"] - 3, 0) // 32


def job_result(F, clk, bf, K):
    """the final job's AfskRxResult: (status, clock, train_end, nbits, nbytes)"""
    k0 = F["k0"] if F["phase"] >= PAYLOAD else K
    k1 = F["k1"] if F["phase"] == ENDED else K
    nbits = k1 - k0
    return (O.ST_OK if nbits > 0 else O.ST_NO_DATA, clk, clk + k0 * bf, nbits, F["nbytes"] if nbits > 0 else 0)


def pending_of(F, clk, bf):
    """afsk_rx_streams_pending_payload without the bytes: (train_end, nbits, ended)"""
    if F["phase"] == TRAIN:
        return -1, 0, False
    return clk + F["k0"] * bf, (F["k1"] if F["phase"] == ENDED else F["consumed"]) - F["k0"], F["phase"] == ENDED


class StreamFramer:
    """a recording's plane words (decided windows past the limits among them: `extra` random windows after the
    recording's K) framed job by job; words below the kept one are overwritten with garbage before each job"""

    def __init__(self, bits, quiet, extra_bits=None, extra_quiet=None, seed=0):
        b = np.concatenate([bits, extra_bits if extra_bits is not None else []]).astype(np.uint8)
        q = np.concatenate([quiet, extra_quiet if extra_quiet is not None else []]).astype(np.uint8)
        n = (len(b) + 31) // 32 + 2
        self.bw, self.qw = pack_words(b, n), pack_words(q, n)
        self.F, self.data, self.reads = fresh_state(), bytearray(), []
        self.rng = np.random.default_rng(seed)

    def advance(self, k_end):
        if k_end <= self.F["consumed"] or self.F["phase"] == ENDED:
            return
        kept = kept_word(self.F)
        bw, qw = self.bw.copy(), self.qw.copy()
        bw[:kept] = self.rng.integers(0, 1 << 32, kept)
        qw[:kept] = self.rng.integers(0, 1 << 32, kept)
        self.F, got = stream_job(bw, qw, self.F, k_end, kept, self.reads)
        for i in sorted(got):
            assert i == len(self.data), (i, len(self.data))
            self.data.append(got[i])

    def final(self, K, clk, bf):
        self.advance(K)
        return job_result(self.F, clk, bf, K), bytes(self.data)


def stream_tags(reads):
    """what a chain of jobs met: a terminator whose 1 lay below the job's first window and in the previous plane
    word; a first quiet window at a job's first window or at the window before its limit; a byte group cut by a
    limit; a search past a job's first 1024-window step"""
    tags = set()
    for r in reads:
        if r[0] == "term":
            _, c, kt = r
            if kt - 3 < c and (kt - 3) >> 5 < c >> 5:
                tags.add("term 1 in previous push and word")
            if kt - 32 * (c >> 5) >= STEPS["stream"]:
                tags.add("term past step")
        elif r[0] == "quiet":
            _, c, kq, K = r
            if kq == c:
                tags.add("quiet at job start")
            if kq == K - 1:
                tags.add("quiet at limit")
            if kq - 32 * (c >> 5) >= STEPS["stream"]:
                tags.add("quiet past step")
        else:
            tags.add("byte cut by limit")
    return tags


# ---------------------------------------------------------------- self-checks ------------------------------------

@pytest.mark.parametrize("baud", BAUDS)
def test_crafted_captures_decode_to_their_sequences(baud):
    """every case of every path: framed_capture's asserts (the oracle's clock, ref_planes and the oracle's framing
    of the crafted windows), and the packed-word model of k_frame / k_frame_warp equals the reference"""
    for c in [c for c in batch_cases() if c.baud == baud] + frame_cases(baud, "stream"):
        c.audio()
        k0, nbits, by = kernel_model(c.bits.astype(np.uint8), c.quiet.astype(np.uint8))
        ref = c.reference()
        assert (c.lead + k0 * bit_frames(baud), nbits, by) == (ref[2], ref[3], ref[5]), (baud, c.name)


def _cut_check(bits, quiet, cuts, clk, bf, extra, seed, want):
    """chained jobs at the increasing limits `cuts`, then the final job with K = len(bits): whole-sequence framing
    (want); the bytes after every cut a prefix of the final bytes"""
    K = len(bits)
    fr = StreamFramer(bits, quiet, extra[0], extra[1], seed)
    snaps = []
    for c in cuts:
        fr.advance(c)
        snaps.append(bytes(fr.data))
    got = fr.final(K, clk, bf)
    assert got == want, (cuts, got[0], want[0])
    assert all(want[1].startswith(s) for s in snaps), cuts
    return fr.reads


@pytest.mark.parametrize("baud", BAUDS)
def test_stream_jobs_over_every_cut_equal_whole_sequence_framing(baud):
    """the stream path's cases (those within 1200 windows) cut once at every window, and in random schedules of
    several increasing limits; decided windows past K sit in the planes beyond the final limit"""
    rng = np.random.default_rng(baud)
    bf = bit_frames(baud)
    tags, n = set(), 0
    for c in frame_cases(baud, "stream"):
        extra = (rng.integers(0, 2, 40).astype(bool), rng.random(40) < 0.2)
        want = frame_whole(c.bits, c.quiet, c.K, c.lead, bf)
        single = range(0, c.K + 1) if c.K <= 1200 else sorted(set(rng.integers(0, c.K, 200).tolist()))
        for cut in single:
            tags |= stream_tags(_cut_check(c.bits, c.quiet, [cut], c.lead, bf, extra, cut, want))
        for _ in range(6):
            m = int(rng.integers(2, 12))
            cuts = sorted(rng.integers(0, c.K + 1, m).tolist())
            tags |= stream_tags(_cut_check(c.bits, c.quiet, cuts, c.lead, bf, extra, m, want))
        n += 1
    assert n > 150
    assert {"term 1 in previous push and word", "quiet at job start", "quiet at limit", "byte cut by limit",
            "term past step", "quiet past step"} <= tags, tags


def test_stream_job_reads_the_previous_word_only_where_it_must():
    """a terminator whose 1 is in the word before the job's first window: found with c % 32 in 0 .. 2; the same
    sequence with the previous word read as zero misses it (the restatement is not vacuous there)"""
    bits = training(200, "alt", None).astype(bool)
    bits[63:67] = [1, 0, 0, 0]                                       # the terminator ends at 66; its 1 in word 1
    quiet = np.zeros(200, bool)
    for c in (64, 65, 66):
        fr = StreamFramer(bits, quiet)
        fr.advance(c)
        assert fr.F["phase"] == TRAIN and kept_word(fr.F) == 1, c
        fr.advance(200)
        assert fr.F["phase"] == PAYLOAD and fr.F["k0"] == 67, c
        assert "term 1 in previous push and word" in stream_tags(fr.reads)
        bw = fr.bw.copy()
        bw[1] = 0
        F, _ = stream_job(bw, fr.qw, dict(consumed=c, k0=0, k1=0, nbytes=0, phase=TRAIN), 200, 1)
        assert F["phase"] == TRAIN, c


def _quads(c):
    k0, nbits = c.layout()
    nbytes = nbits // 14
    return k0, nbits, nbytes


def test_quotas_every_family_and_residue_reaches_every_path():
    """per path: every family; terminators at k_t = 3 and every residue mod 32, each training kind; K at every
    residue mod 32 with each ending; terminators at K - 1 / K - 2 / K - 4; quiet windows before k0, at k0 + every
    residue mod 14, at K - 1, none; k0 at every residue mod 32; nbits at every residue mod 56 and 1 .. 13; every
    codeword at every quad slot, quads at every bit offset of a word, tail bytes at every offset; the path's step
    edges at +-0..3; the 262,144 / 262,145 window captures (the CTA paths: 262,145 and longer ones too)"""
    for v in STEPS:
        cases = path_cases(v)
        tags = set().union(*(c.tags for c in cases))
        assert {c.family for c in cases} == set(FAMILIES) or (v == "stream" and {c.family for c in cases} == set("TEQH")), v
        want = ({"k_t=3"} | {f"kt%32={r}" for r in range(32)} | {f"train={k}" for k in TRAIN_KINDS}
                | {f"K%32={r}" for r in range(32)} | {f"end={e}" for e in (1, 2, 3)} | {f"term@K-{e}" for e in (1, 2, 4)}
                | {"quiet<k0", "quiet in k0 word", "quiet@k0-1", "q@K-1", "no quiet"} | {f"q-k0%14={r}" for r in range(14)}
                | {f"k0%32={r}" for r in range(32)} | {f"nbits%56={r}" for r in range(56)} | {f"nbits={n}" for n in range(1, 14)}
                | {"codewords"} | {f"kt=step{d:+d}" for d in D} | {f"q=step{d:+d}" for d in D})
        if v != "stream":
            want |= {"K=262144"} | ({"K=262145", "K>262144"} if v != "warp" else set())
            assert {c.kmax for c in cases if c.family == "L" and "K>262144" not in c.tags} == (
                {262144} if v == "warp" else {262144, 262145}), v
        assert want <= tags, (v, sorted(want - tags))
        shifts, tails, slots = set(), set(), set()
        for c in cases:
            k0, nbits, nbytes = _quads(c)
            q = nbytes // 4
            shifts |= {(k0 + 56 * i) & 31 for i in range(min(q, 64))}
            tails |= {(k0 + 14 * i) & 31 for i in range(4 * q, nbytes)}
            if "codewords" in c.tags:
                b = c.bits[k0:k0 + 56 * q].astype(np.int64).reshape(-1, 7) @ (1 << np.arange(7))
                slots |= set(zip(b.tolist(), (np.arange(len(b)) % 8).tolist()))
        assert shifts == set(range(32)) and tails == set(range(32)), (v, sorted(set(range(32)) - shifts), sorted(set(range(32)) - tails))
        assert len(slots) == 128 * 8, (v, len(slots))
        st = STEPS[v]
        edges = {(c.layout()[0] - 1) % st for c in cases if c.name.startswith(f"T:step{st}x")}
        qedges = {(c.layout()[0] + c.layout()[1] - 32 * (c.layout()[0] >> 5)) % st for c in cases
                  if c.name.startswith(f"Q:step{st}x")}
        assert edges == qedges == {d % st for d in D}, (v, edges, qedges)
