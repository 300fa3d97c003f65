"""The per-frame callers at their edges: Frame::ComputeStereoMatches (lld_stereo_matches), Tracking::AddLinesFrom
(lld_line_associate) and Map{Point,Line}::ComputeDistinctiveDescriptors (lld_medoid_orb / lld_medoid_float).

Small hand-built problems pin each rule: every case states which keypoint / line gets what and which get nothing, and on the
CPU the oracle and the numpy transcriptions of test_cpu_oracle.py must both give exactly that.  On the GPU every case, and
larger generated batches (720p / 1080p frames, a bordered pyramid whose row stride is not its width, ragged batches, frames
of more than 1024 lines, landmarks of up to 256 observations), must be bit- / index-exact against the oracle.  The argument
checks reject out-of-range octaves and indices before anything is allocated or launched."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_cpu_oracle import _add_lines_from_numpy, _medoid_landmarks, _medoid_numpy, _stereo_matches_numpy  # noqa: E402

from lld_slam_b200 import api, synth  # noqa: E402

f32 = np.float32
LLD_ERR_ARG, LLD_ERR_UNSUPPORTED = -2, -4


def _flip(d, n, first=0):
    """d with bits [first, first + n) flipped: Hamming distance n to d"""
    bits = np.unpackbits(d.copy())
    bits[first:first + n] ^= 1
    return np.packbits(bits)


# ------------------------------------------------------------------------------------------------------------------
# stereo matching: hand-built frames
# ------------------------------------------------------------------------------------------------------------------
SAD_STEP = 10   # a pasted right patch differs from its left patch by SAD_STEP on sad_px pixels: its SAD is SAD_STEP * sad_px


class _StereoFrame:
    """A frame of 96 x 160 pixels, pyramid scale factor 2 (level l is (96 >> l) x (160 >> l)), mb = 0.5, mbf = 32: maxD = 64.
    Left and right levels are independent noise in [40, 216), so a right patch resembles a left one only where a case pastes
    it; there the SAD is exactly SAD_STEP * sad_px, everywhere else it is thousands.  Keypoints are given in level pixels."""

    def __init__(self, seed, n_levels=3, rows=96, cols=160):
        self.rng = np.random.default_rng(seed)
        self.scale = (2.0 ** np.arange(n_levels)).astype(f32)
        self.L = [self.rng.integers(40, 216, (rows >> l, cols >> l), dtype=np.uint8) for l in range(n_levels)]
        self.R = [self.rng.integers(40, 216, (rows >> l, cols >> l), dtype=np.uint8) for l in range(n_levels)]
        self.used = [np.zeros((rows >> l, cols >> l), bool) for l in range(n_levels)]
        self.kpL, self.octL, self.descL, self.kpR, self.octR, self.descR = [], [], [], [], [], []
        self.expect = []   # per left keypoint: None (no match) or (level-0 uright expected, tolerance)

    def desc(self):
        return self.rng.integers(0, 256, 32, dtype=np.uint8)

    def left(self, uL, vL, lvl, desc, expect_col=None):
        """expect_col: level column of the right patch the match must land on (None: no match)"""
        self.kpL.append((uL, vL)); self.octL.append(lvl); self.descL.append(desc)
        s = float(self.scale[lvl])
        self.expect.append(None if expect_col is None else (s * expect_col, 0.5 * s))   # |parabola offset| <= 1/2

    def right(self, uR, vR, lvl, desc):
        self.kpR.append((uR, vR)); self.octR.append(lvl); self.descR.append(desc)

    def paste(self, lvl, su, sv, col, sad_px=20):
        """right patch centred (sv, col) := left patch centred (sv, su), + SAD_STEP on sad_px pixels other than the centre"""
        blk = self.L[lvl][sv - 5:sv + 6, su - 5:su + 6].astype(np.int32).reshape(-1)
        assert blk.size == 121
        add = np.zeros(121, np.int32)
        add[[i for i in range(121) if i != 60][:sad_px]] = SAD_STEP
        m = self.used[lvl][sv - 5:sv + 6, col - 5:col + 6]
        assert m.shape == (11, 11) and not m.any(), "pasted patches overlap"
        m[:] = True
        self.R[lvl][sv - 5:sv + 6, col - 5:col + 6] = (blk + add).reshape(11, 11).astype(np.uint8)

    def pair(self, su, sv, lvl, disp, inc=0, flips=0, sad_px=20, match=True, uR=None, vR=None, octR=None, paste=True):
        """left keypoint at level pixel (su, sv), its right keypoint disp level pixels to the left (or at uR), the right patch
        pasted inc pixels from the right keypoint; match: whether the case expects the pair to be accepted"""
        s = float(self.scale[lvl])
        sr = su - disp
        d = self.desc()
        self.left(f32(su * s), f32(sv * s), lvl, d, sr + inc if match else None)
        self.right(f32(sr * s) if uR is None else f32(uR), f32(sv * s) if vR is None else f32(vR), lvl if octR is None else octR,
                   _flip(d, flips))
        if paste:
            self.paste(lvl, su, sv, sr + inc, sad_px)
        return d

    def frame(self):
        a2 = lambda v: np.ascontiguousarray(np.array(v, f32).reshape(-1, 2))                # noqa: E731
        d32 = lambda v: np.ascontiguousarray(np.array(v, np.uint8).reshape(-1, 32))         # noqa: E731
        return dict(kpL=a2(self.kpL), octL=np.array(self.octL, np.int32), descL=d32(self.descL),
                    kpR=a2(self.kpR), octR=np.array(self.octR, np.int32), descR=d32(self.descR),
                    scale=self.scale, inv=(f32(1) / self.scale).astype(f32), pyrL=self.L, pyrR=self.R,
                    mb=f32(0.5), mbf=f32(32.0))


def _st_left_patch_edges():
    """the left 11x11 patch leaves the level image on each side, at level 0 and at the top level, next to its in-bounds twin"""
    F = _StereoFrame(1)
    for lvl, (rows, cols), disp, su in ((0, (96, 160), 12, 30), (2, (24, 40), 6, 20)):
        F.pair(su, 4, lvl, disp, match=False, paste=False)                     # top: first row -1
        F.pair(su, 5, lvl, disp)                                               # first row 0
        F.pair(su, rows - 5, lvl, disp, match=False, paste=False)              # bottom: one row past the image
        F.pair(su, rows - 6, lvl, disp)                                        # last row inside
        F.pair(cols - 5, 11, lvl, disp, match=False, paste=False)              # right: one column past the image
        F.pair(cols - 6, 11 if lvl else 40, lvl, disp)                         # last column inside
        # left: first column -1.  Its twin (first column 0) meets the strip carve-out instead: its right keypoint lies left of it
        F.pair(4, 11, lvl, 0, uR=0.0, match=False, paste=False)
        F.pair(5, 11 if lvl else 60, lvl, 0, uR=0.0, match=False, paste=False)
    return [F]


def _st_right_strip_edges():
    """the slide strip of the right patch leaves the image on the left (first column -1) and on the right (endu = cols), each
    next to its twin one pixel further in"""
    F = _StereoFrame(2)
    F.pair(21, 20, 0, 12, match=False, paste=False)   # scaleduR0 = 9: strip starts at column -1
    F.pair(22, 40, 0, 12)                             # 10: column 0
    F.pair(154, 60, 0, 5, match=False, paste=False)   # 149: endu = 160 = cols
    F.pair(153, 80, 0, 5)                             # 148: endu = 159
    return [F]


def _st_row_range():
    """vL < 0, vL in (-1, 0), vL = nRows - 0.5 and vL >= nRows get nothing; right keypoints whose row band starts above row 0
    (y = 1.5, octave 1: rows -3 .. 6) or ends below the last row (y = 93.5: rows 89 .. 98) match inside the image"""
    F = _StereoFrame(3)
    dA = F.desc(); dB = F.desc()
    F.right(f32(40), f32(1.5), 1, dA)
    F.right(f32(100), f32(93.5), 1, dB)
    F.left(f32(52), f32(5.5), 0, dA, 40); F.paste(0, 52, 6, 40)        # row 5, patch centred on row round(5.5) = 6
    F.left(f32(112), f32(89.5), 0, dB, 100); F.paste(0, 112, 90, 100)
    for v in (-3.0, -0.5):
        F.left(f32(52), f32(v), 0, dA)
    for v in (95.5, 96.0, 200.0):
        F.left(f32(112), f32(v), 0, dB)
    return [F]


def _st_hamming_edges():
    """Hamming distance 74 is accepted, 75 rejected; an identical descriptor two octaves away is not a candidate"""
    F = _StereoFrame(4)
    F.pair(60, 20, 0, 10, flips=74)
    F.pair(60, 40, 0, 10, flips=75, match=False)
    F.pair(60, 60, 0, 10, octR=2, match=False)
    F.pair(60, 80, 0, 10, octR=1)                     # one octave away: a candidate
    return [F]


def _st_tie(swap):
    F = _StereoFrame(5)
    d = F.desc()
    a, b = (f32(56), f32(30)), (f32(70), f32(30))
    first, second = (b, a) if swap else (a, b)
    F.right(*first, 0, d); F.right(*second, 0, d)      # identical descriptors, both in row 30's band and in the window
    F.left(f32(80), f32(30), 0, d, int(first[0]))      # the lower index wins, wherever it lies
    F.paste(0, 80, 30, 56); F.paste(0, 80, 30, 70)
    return [F]


def _st_window_edges():
    """uR = uL and uR = uL - maxD are inside the disparity window; one ulp outside either is not"""
    F = _StereoFrame(6)
    F.pair(100, 20, 0, 0, inc=-1, uR=100.0)
    F.pair(100, 40, 0, 0, inc=-1, uR=np.nextafter(f32(100), f32(200)), match=False)
    F.pair(100, 60, 0, 64, inc=1, uR=36.0)
    F.pair(100, 80, 0, 64, inc=1, uR=np.nextafter(f32(36), f32(0)), match=False)
    return [F]


def _st_slide_ends():
    """the best SAD at incR = -5 / +5 rejects the point (no parabola), at -4 / +4 it is refined"""
    F = _StereoFrame(7)
    F.pair(100, 20, 0, 20, inc=-5, match=False)
    F.pair(100, 40, 0, 20, inc=-4)
    F.pair(100, 60, 0, 20, inc=5, match=False)
    F.pair(100, 80, 0, 20, inc=4)
    return [F]


def _st_disparity_range():
    """after refinement the disparity must lie in [0, maxD): the keypoints are inside the window, the patches outside it"""
    F = _StereoFrame(8)
    F.pair(110, 20, 0, 64, inc=-1, match=False)       # disparity about 65
    F.pair(110, 40, 0, 64, inc=1)                     # about 63
    F.pair(110, 60, 0, 0, inc=1, match=False)         # about -1
    return [F]


def _st_median_counts():
    """frames where 1, 2 and 3 points survive the SAD stage: the median is element count / 2 of the sorted SADs, and a SAD at
    or above 1.5 * 1.4 * median is dropped (SADs of 2 and 3 points: 100, 300 -> both stay; 100, 300, 1000 -> 1000 goes)"""
    one = _StereoFrame(9); one.pair(60, 20, 0, 10, sad_px=20)
    two = _StereoFrame(10); two.pair(60, 20, 0, 10, sad_px=10); two.pair(60, 50, 0, 10, sad_px=30)
    three = _StereoFrame(11)
    three.pair(60, 20, 0, 10, sad_px=10); three.pair(60, 50, 0, 10, sad_px=30); three.pair(60, 80, 0, 10, sad_px=100, match=False)
    return [one, two, three]


def _st_median_zero():
    """identical patches: every SAD and the median are 0, so thDist = 0 and every survivor is dropped"""
    F = _StereoFrame(12)
    for sv in (20, 50, 80):
        F.pair(60, sv, 0, 10, sad_px=0, match=False)
    return [F]


def _st_single_level():
    F = _StereoFrame(13, n_levels=1)
    F.pair(60, 20, 0, 10)
    F.pair(60, 50, 0, 10, flips=75, match=False)
    F.pair(120, 80, 0, 30, sad_px=15)
    return [F]


def _st_empty_sides():
    """a frame without left keypoints, one without right keypoints (its left keypoints get nothing) and a normal one"""
    a = _StereoFrame(14)
    a.right(f32(50), f32(30), 0, a.desc())
    b = _StereoFrame(15)
    for sv in (20, 40):
        b.left(f32(60), f32(sv), 0, b.desc())
    c = _StereoFrame(16)
    c.pair(60, 20, 0, 10)
    return [a, b, c]


STEREO_CASES = {
    "left_patch_edges": _st_left_patch_edges, "right_strip_edges": _st_right_strip_edges, "row_range": _st_row_range,
    "hamming_edges": _st_hamming_edges, "tie_lower_index": lambda: _st_tie(False), "tie_swapped": lambda: _st_tie(True),
    "window_edges": _st_window_edges, "slide_ends": _st_slide_ends, "disparity_range": _st_disparity_range,
    "median_counts": _st_median_counts, "median_zero": _st_median_zero, "single_level": _st_single_level,
    "empty_sides": _st_empty_sides,
}


def _stereo_case(name):
    builders = STEREO_CASES[name]()
    return [b.frame() for b in builders], [b.expect for b in builders]


def _check_stereo_expect(frames, expects, uright, n_matched):
    off = 0
    for f, (fr, exp) in enumerate(zip(frames, expects)):
        u = uright[off:off + len(exp)]
        off += len(exp)
        for i, e in enumerate(exp):
            if e is None:
                assert u[i] == -1, (f, i, u[i])
            else:
                assert u[i] != -1 and abs(float(u[i]) - e[0]) <= e[1], (f, i, u[i], e)
        assert n_matched[f] == sum(e is not None for e in exp), (f, n_matched[f])
    assert off == len(uright)


# ------------------------------------------------------------------------------------------------------------------
# stereo matching: CPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(STEREO_CASES))
def test_stereo_case_oracle_and_numpy(built, name):
    frames, expects = _stereo_case(name)
    o = api.stereo_matches(synth.batch_stereo(frames), impl="oracle")
    off = 0
    for fr in frames:
        n = len(fr["kpL"])
        uR, dep = _stereo_matches_numpy(fr)
        assert np.array_equal(o["uright"][off:off + n], uR) and np.array_equal(o["depth"][off:off + n], dep)
        off += n
    _check_stereo_expect(frames, expects, o["uright"], o["n_matched"])


def test_stereo_padded_pyramid_on_the_oracle(built):
    """a bordered pyramid (row stride cols + 38, the image a region inside it) gives what the packed one gives"""
    frames = [synth.make_stereo_frame(s, n_kp=300) for s in (21, 22)]
    a = api.stereo_matches(synth.batch_stereo(frames), impl="oracle")
    p = synth.batch_stereo(frames, pad=38)
    assert (p["pyr_stride"] == p["pyr_cols"] + 38).all()
    b = api.stereo_matches(p, impl="oracle")
    for k in ("uright", "depth", "n_matched"):
        assert np.array_equal(a[k], b[k])
    assert a["n_matched"].min() > 100


# ------------------------------------------------------------------------------------------------------------------
# temporal line association: hand-built frames
# ------------------------------------------------------------------------------------------------------------------
K_ASSOC = np.array([[500.0, 0, 320], [0, 500.0, 240], [0, 0, 1]])
BASE = 0.5    # stereo baseline in metres
D_ASSOC = 8


class _AssocBatch:
    """Frames seen by an identity camera (the right camera BASE to its right).  Map line j of a frame is the horizontal 3D line
    y = y_j, z = z_j with a zero descriptor unless given; a current line lies on its projection, shifted down by `off` pixels at
    both ends (reprojection error 2 * off), and its descriptor is the map line's plus `dist` in the first component
    (descriptor distance `dist`)."""

    def __init__(self, monocular=0, md_thr=2.0, thr=3.0):
        self.monocular, self.md_thr, self.thr = monocular, md_thr, thr
        self.frames = []

    def frame(self):
        self.frames.append(dict(ml=[], cur=[], right=[]))
        return self

    def map_line(self, y, z=5.0, valid=1, behind=False, desc=None):
        f = self.frames[-1]
        X1, X2 = np.array([-0.5, y, z]), np.array([0.5, y, z])
        if behind:
            X1 = np.array([-0.5, y, -1.0])
        d = (X2 - X1) / np.linalg.norm(X2 - X1)
        X0 = X1 - X1.dot(d) * d
        dsc = np.zeros(D_ASSOC, f32) if desc is None else np.array(desc, f32)
        f["ml"].append(dict(valid=valid, x0d=np.concatenate([X0, d]), x12=np.concatenate([X1, X2]), desc=dsc, y=y, z=z, cand=[]))
        return len(f["ml"]) - 1

    @staticmethod
    def _seg(y, z, shift_x, off):
        u = lambda X: 500.0 * (X - shift_x) / z + 320.0                 # noqa: E731
        v = 500.0 * y / z + 240.0 + off
        return [u(-0.5), v, u(0.5), v]

    def cur_line(self, ml, dist=0.5, off=0.0, octave=0, right=True, right_off=0.0, taken=0, desc=None):
        f = self.frames[-1]
        m = f["ml"][ml]
        dsc = m["desc"].copy() if desc is None else np.asarray(desc, f32)
        if desc is None:
            dsc[0] = f32(dsc[0] + f32(dist))
        rm = -1
        if right:
            f["right"].append(self._seg(m["y"], m["z"], BASE, right_off))
            rm = len(f["right"]) - 1
        f["cur"].append(dict(seg=self._seg(m["y"], m["z"], 0.0, off), octave=octave, lm=rm, taken=taken, desc=dsc))
        return len(f["cur"]) - 1

    def stray(self, y):
        """a current line in a frame without map lines"""
        self.frames[-1]["cur"].append(dict(seg=self._seg(y, 5.0, 0.0, 0.0), octave=0, lm=-1, taken=0, desc=np.zeros(D_ASSOC, f32)))

    def cand(self, ml, *idx):
        self.frames[-1]["ml"][ml]["cand"] += list(idx)

    def filler(self, n, ml):
        """n current lines nobody lists as a candidate"""
        for _ in range(n):
            self.cur_line(ml, dist=3.0)

    def problem(self):
        ml = [m for f in self.frames for m in f["ml"]]
        cur = [c for f in self.frames for c in f["cur"]]
        right = [r for f in self.frames for r in f["right"]]
        csr = lambda n: np.concatenate([[0], np.cumsum(n)]).astype(np.int32)   # noqa: E731
        T = np.eye(4); Tr = np.eye(4); Tr[0, 3] = BASE
        F = len(self.frames)
        return dict(
            n_frames=F, desc_dim=D_ASSOC, K=K_ASSOC.reshape(-1), thr_reproj_base=self.thr, md_thr=self.md_thr, monocular=self.monocular,
            ml_off=csr([len(f["ml"]) for f in self.frames]), ml_valid=np.array([m["valid"] for m in ml], np.uint8),
            ml_x0_dir=np.ascontiguousarray(np.array([m["x0d"] for m in ml], np.float64).reshape(-1, 6)),
            ml_x1x2=np.ascontiguousarray(np.array([m["x12"] for m in ml], np.float64).reshape(-1, 6)),
            ml_desc=np.ascontiguousarray(np.array([m["desc"] for m in ml], f32).reshape(-1, D_ASSOC)),
            cand_off=csr([len(m["cand"]) for m in ml]), cand_idx=np.array([i for m in ml for i in m["cand"]], np.int32),
            cur_off=csr([len(f["cur"]) for f in self.frames]),
            cur_left=np.ascontiguousarray(np.array([c["seg"] for c in cur], f32).reshape(-1, 4)),
            cur_octave=np.array([c["octave"] for c in cur], np.int32), cur_line_match=np.array([c["lm"] for c in cur], np.int32),
            cur_taken=np.array([c["taken"] for c in cur], np.uint8),
            cur_desc=np.ascontiguousarray(np.array([c["desc"] for c in cur], f32).reshape(-1, D_ASSOC)),
            right_off=csr([len(f["right"]) for f in self.frames]),
            cur_right=np.ascontiguousarray(np.array(right, f32).reshape(-1, 4)),
            T_curr=np.ascontiguousarray(np.tile(T.reshape(-1), (F, 1))), T_right=np.ascontiguousarray(np.tile(Tr.reshape(-1), (F, 1))))


def _la_gates(monocular):
    """a line without a right match and a line whose right segment is 10 px off: the stereo arm rejects both (no right match /
    right-image gate), the monocular arm checks the left image only and takes both"""
    B = _AssocBatch(monocular=monocular).frame()
    m = [B.map_line(y) for y in (-0.6, -0.2, 0.2)]
    a = B.cur_line(m[0], right=False)
    b = B.cur_line(m[1], right_off=5.0)
    c = B.cur_line(m[2])
    for j, i in zip(m, (a, b, c)):
        B.cand(j, i)
    return B, [[0, 1, 2] if monocular else [-1, -1, 2]]


def _la_ties():
    """equal distances at list positions 3 and 35 (two chunks of the warp argmin) and at 40 and 41: the earlier position wins,
    also when it holds the higher line index; a line claimed by an earlier map line is skipped"""
    B = _AssocBatch().frame()
    m0, m1 = B.map_line(0.1), B.map_line(0.1)
    fill = [B.cur_line(m0, dist=1.5) for _ in range(4)]
    t2 = B.cur_line(m0, dist=0.25); t1 = B.cur_line(m0, dist=0.25)        # identical segments and descriptors
    t4 = B.cur_line(m0, dist=0.25); t3 = B.cur_line(m0, dist=0.25)
    lst = [fill[i % 4] for i in range(45)]
    lst[3], lst[35] = t1, t2
    B.cand(m0, *lst)
    lst = [fill[i % 4] for i in range(45)]
    lst[3], lst[40], lst[41] = t1, t3, t4
    B.cand(m1, *lst)
    exp = [-1] * 8
    exp[t1], exp[t3] = m0, m1
    return B, [exp]


def _la_duplicates():
    """the same current line twice in one list; a second map line then finds it claimed and takes the next best"""
    B = _AssocBatch().frame()
    m0, m1 = B.map_line(0.0), B.map_line(0.0)
    a = B.cur_line(m0, dist=0.5); b = B.cur_line(m0, dist=1.0)
    B.cand(m0, a, a, b)
    B.cand(m1, a, b, a)
    exp = [-1, -1]
    exp[a], exp[b] = m0, m1
    return B, [exp]


def _la_taken_above_1024():
    """1500 current lines: lines taken on entry (1030, 1100) and claimed during the loop (1300) at bits beyond the first 32 words"""
    B = _AssocBatch().frame()
    P, Q, R = B.map_line(0.3), B.map_line(0.3), B.map_line(0.3)
    B.filler(1500, P)
    f = B.frames[-1]
    for i, dist, taken in ((1100, 0.1, 1), (1200, 0.5, 0), (1300, 0.3, 0), (1030, 0.1, 1), (40, 0.9, 0)):
        f["cur"][i]["desc"] = f["ml"][P]["desc"].copy(); f["cur"][i]["desc"][0] += f32(dist); f["cur"][i]["taken"] = taken
    B.cand(P, 1100, 1200, 1300)
    B.cand(Q, 1300, 1200)
    B.cand(R, 1030, 40)
    exp = [-1] * 1500
    exp[1300], exp[1200], exp[40] = P, Q, R
    return B, [exp]


def _la_empty_and_rejected():
    """a frame without map lines, one without current lines, and one with a map line behind the camera, an invalid map line and
    a map line with an empty candidate list, each next to a perfect candidate; the last map line matches"""
    B = _AssocBatch()
    B.frame(); B.stray(0.0); B.stray(0.2)
    B.frame(); B.map_line(0.0); B.map_line(0.2)
    B.frame()
    back = B.map_line(-0.3, behind=True); inval = B.map_line(0.0, valid=0); empty = B.map_line(0.3); ok = B.map_line(0.6)
    a = B.cur_line(back, dist=0.0); b = B.cur_line(inval, dist=0.0); B.cur_line(empty, dist=0.0); d = B.cur_line(ok, dist=0.0)
    B.cand(back, a); B.cand(inval, b); B.cand(ok, d)
    return B, [[-1, -1], [], [-1, -1, -1, ok]]


def _la_md_thr_edge():
    """a descriptor distance equal to md_thr (2) is accepted, the next float above it is not"""
    B = _AssocBatch().frame()
    m0, m1 = B.map_line(-0.2, desc=np.zeros(D_ASSOC)), B.map_line(0.2, desc=np.zeros(D_ASSOC))
    a = B.cur_line(m0, dist=2.0)
    b = B.cur_line(m1, dist=float(np.nextafter(f32(2.0), f32(3.0))))
    B.cand(m0, a); B.cand(m1, b)
    return B, [[m0, -1]]


def _la_octave_threshold():
    """reprojection error 8.5 (both ends 4.25 px off): inside 3 * 1.44^3 at octave 3, outside 3 * 1.44^2 at octave 2; 9.2 is
    outside at octave 3"""
    B = _AssocBatch().frame()
    m = [B.map_line(y) for y in (-0.6, -0.2, 0.2)]
    a = B.cur_line(m[0], off=4.25, right_off=4.25, octave=3)
    b = B.cur_line(m[1], off=4.25, right_off=4.25, octave=2)
    c = B.cur_line(m[2], off=4.6, right_off=4.6, octave=3)
    for j, i in zip(m, (a, b, c)):
        B.cand(j, i)
    return B, [[m[0], -1, -1]]


def _la_huge_distance():
    """finite descriptors at distance 1e10 and more: the reference keeps md = 1e10 and matches nothing (md_thr is no limit here)"""
    B = _AssocBatch(md_thr=1e30).frame()
    m0 = B.map_line(0.0, desc=np.zeros(D_ASSOC))
    a = B.cur_line(m0, dist=1e10); b = B.cur_line(m0, dist=5e10)
    B.cand(m0, a, b)
    return B, [[-1, -1]]


def _la_nan_descriptor():
    """a NaN in a current line's descriptor: that candidate is never chosen, whether before or after a finite one in its chunk;
    a NaN in the map line's descriptor matches nothing"""
    B = _AssocBatch().frame()
    m0, m1, m2 = B.map_line(-0.4), B.map_line(0.0), B.map_line(0.4)
    n0 = B.cur_line(m0, dist=np.nan); g0 = B.cur_line(m0, dist=0.5)
    g1 = B.cur_line(m1, dist=0.5); n1 = B.cur_line(m1, dist=np.nan)
    g2 = B.cur_line(m2, dist=0.5)
    B.frames[-1]["ml"][m2]["desc"][3] = np.nan
    B.cand(m0, n0, g0); B.cand(m1, g1, n1); B.cand(m2, g2)
    exp = [-1] * 5
    exp[g0], exp[g1] = m0, m1
    return B, [exp]


ASSOC_CASES = {
    "stereo_gates": lambda: _la_gates(0), "monocular_arm": lambda: _la_gates(1), "ties": _la_ties, "duplicates": _la_duplicates,
    "taken_above_1024": _la_taken_above_1024, "empty_and_rejected": _la_empty_and_rejected, "md_thr_edge": _la_md_thr_edge,
    "octave_threshold": _la_octave_threshold, "huge_distance": _la_huge_distance, "nan_descriptor": _la_nan_descriptor,
}


def _assoc_case(name):
    B, exp = ASSOC_CASES[name]()
    return B.problem(), exp


def _check_assoc_expect(p, exp, out):
    for f, e in enumerate(exp):
        a, b = int(p["cur_off"][f]), int(p["cur_off"][f + 1])
        assert out["cur_assoc"][a:b].tolist() == e, f
        assert out["n_added"][f] == sum(x >= 0 for x in e)


@pytest.mark.parametrize("name", sorted(ASSOC_CASES))
def test_line_assoc_case_oracle_and_numpy(built, name):
    p, exp = _assoc_case(name)
    o = api.line_associate(p, impl="oracle")
    ref, added = _add_lines_from_numpy(p)
    assert np.array_equal(o["cur_assoc"], ref) and np.array_equal(o["n_added"], added)
    _check_assoc_expect(p, exp, o)


def test_line_assoc_monocular_batch_on_the_oracle(built):
    """the generated batch in the monocular arm: lines without a right match take part"""
    p = synth.make_line_assoc_batch(4, 150, 120, 32, 31)
    p["monocular"] = 1
    o = api.line_associate(p, impl="oracle")
    ref, added = _add_lines_from_numpy(p)
    assert np.array_equal(o["cur_assoc"], ref) and np.array_equal(o["n_added"], added)
    assert ((o["cur_assoc"] >= 0) & (p["cur_line_match"] < 0)).sum() > 10


# ------------------------------------------------------------------------------------------------------------------
# distinctive descriptors
# ------------------------------------------------------------------------------------------------------------------
def _md_truncation():
    """1-D descriptors 0, 3 - 2^-22, 5.5: nearest-neighbour distances 2.9999998, 2.5000002, 2.5000002 all truncate to 2, so the
    first index wins (compared as floats, index 1 would)"""
    return [np.array([[0.0], [np.nextafter(f32(3), f32(0))], [5.5]], f32)], [0]


def _md_exact_integers():
    """2-D integer points at exact integer distances (3-4-5 triangles): medians sit exactly on integers"""
    pts = np.array([[0, 0], [3, 4], [6, 8], [6, 0], [0, 8]], f32)
    # N = 5, k = 2: third smallest of each row (itself included).  (3, 4) is 5 from every other point: median 5; the corners
    # have 6 or 8
    return [pts], [1]


def _md_first_of_equal_medians():
    """nearest-neighbour distances 10, 1, 1, 9: indices 1 and 2 tie, the first of them wins"""
    return [np.array([[0], [10], [11], [20]], f32)], [1]


def _md_all_identical():
    return [np.full((7, 5), 3.0, f32), np.full((40, 5), -1.0, f32)], [0, 0]


MEDOID_CASES = {"truncation": _md_truncation, "exact_integers": _md_exact_integers, "first_of_equal_medians": _md_first_of_equal_medians,
                "all_identical": _md_all_identical}


def _medoid_case(name):
    lms, exp = MEDOID_CASES[name]()
    D = lms[0].shape[1]
    assert all(x.shape[1] == D for x in lms)
    off = np.concatenate([[0], np.cumsum([len(x) for x in lms])]).astype(np.int32)
    return off, np.ascontiguousarray(np.concatenate(lms)), exp


def _small_integer_landmarks(N, D, seed, n_lm=3):
    """n_lm landmarks of N descriptors with entries in {0, 1, 2}: many exact and many tied distances"""
    rng = np.random.default_rng(seed)
    off = np.arange(n_lm + 1, dtype=np.int32) * N
    return off, rng.integers(0, 3, (n_lm * N, D)).astype(f32)


@pytest.mark.parametrize("name", sorted(MEDOID_CASES))
def test_medoid_case_oracle_and_numpy(built, name):
    off, desc, exp = _medoid_case(name)
    o = api.medoid_float(off, desc, impl="oracle")
    assert np.array_equal(o, _medoid_numpy(off, desc, False))
    assert o.tolist() == exp


def test_medoid_small_integers_oracle_and_numpy(built):
    for N, D in ((31, 1), (33, 32), (64, 72)):
        off, desc = _small_integer_landmarks(N, D, N + D)
        assert np.array_equal(api.medoid_float(off, desc, impl="oracle"), _medoid_numpy(off, desc, False))


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _stereo_gpu_vs_oracle(p, ctx):
    g = api.stereo_matches(p, impl="gpu", ctx=ctx)
    o = api.stereo_matches(p, impl="oracle")
    for k in ("uright", "depth", "n_matched"):
        assert np.array_equal(g[k], o[k]), k
    return o


@pytest.mark.gpu
@pytest.mark.parametrize("pad", [0, 38])
@pytest.mark.parametrize("name", sorted(STEREO_CASES))
def test_gpu_stereo_case(gpu_ctx, name, pad):
    frames, expects = _stereo_case(name)
    g = _stereo_gpu_vs_oracle(synth.batch_stereo(frames, pad=pad), gpu_ctx)
    _check_stereo_expect(frames, expects, g["uright"], g["n_matched"])


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", [(720, 1280), (1080, 1920)])
def test_gpu_stereo_tall_frames(gpu_ctx, rows, cols):
    """more rows than threads: the row-band pass takes a second (and third) turn; matches below row 512 must exist"""
    frames = [synth.make_stereo_frame(60 + rows + s, n_kp=2000, rows=rows, cols=cols, n_levels=8) for s in range(2)]
    for f in frames:
        f["mbf"] = f32(0.54 * 100.0)      # maxD = 100 px: the generator's disparity grows to 82 px at row 1080
    p = synth.batch_stereo(frames)
    o = _stereo_gpu_vs_oracle(p, gpu_ctx)
    low = (p["left_xy"][:, 1] >= 512) & (o["uright"] >= 0)
    assert low.sum() > 20 and o["n_matched"].min() > 200


@pytest.mark.gpu
def test_gpu_stereo_bordered_pyramid(gpu_ctx):
    """ORB-SLAM's pyramid levels are regions of a bordered image: row stride = cols + 38"""
    frames = [synth.make_stereo_frame(70 + s, n_kp=2000, rows=376, cols=1241, n_levels=8) for s in range(3)]
    p = synth.batch_stereo(frames, pad=38)
    o = _stereo_gpu_vs_oracle(p, gpu_ctx)
    assert o["n_matched"].min() > 500
    packed = api.stereo_matches(synth.batch_stereo(frames), impl="gpu", ctx=gpu_ctx)
    assert np.array_equal(packed["uright"], o["uright"])


@pytest.mark.gpu
def test_gpu_stereo_ragged_batch(gpu_ctx):
    """frames without left keypoints, without right keypoints, and of 1, 511, 512, 513 and 2000 keypoints in one batch"""
    frames = []
    for s, n in enumerate([400, 400, 1, 511, 512, 513, 2000]):
        frames.append(synth.make_stereo_frame(80 + s, n_kp=n))
    frames[0]["kpL"], frames[0]["octL"], frames[0]["descL"] = frames[0]["kpL"][:0], frames[0]["octL"][:0], frames[0]["descL"][:0]
    frames[1]["kpR"], frames[1]["octR"], frames[1]["descR"] = frames[1]["kpR"][:0], frames[1]["octR"][:0], frames[1]["descR"][:0]
    o = _stereo_gpu_vs_oracle(synth.batch_stereo(frames), gpu_ctx)
    assert o["n_matched"][0] == 0 and o["n_matched"][1] == 0 and o["n_matched"][3:].min() > 100


def _expect_rejected(ctx, call, code, *words):
    """the call fails with `code`, names the problem, and launches nothing"""
    with pytest.raises(RuntimeError) as ei:
        call()
    msg = str(ei.value)
    assert f"failed with {code}" in msg, msg
    for w in words:
        assert w in msg, msg
    assert ctx.launch_count() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("side", ["left_octave", "right_octave"])
def test_gpu_stereo_rejects_octave_out_of_range(gpu_ctx, side):
    frames, _ = _stereo_case("hamming_edges")
    p = synth.batch_stereo(frames)
    _stereo_gpu_vs_oracle(p, gpu_ctx)
    assert gpu_ctx.launch_count() > 0
    q = dict(p)
    q[side] = p[side].copy()
    q[side][-1] = p["n_levels"]
    _expect_rejected(gpu_ctx, lambda: api.stereo_matches(q, impl="gpu", ctx=gpu_ctx), LLD_ERR_ARG, side)


def _assoc_gpu_vs_oracle(p, ctx):
    g = api.line_associate(p, impl="gpu", ctx=ctx)
    o = api.line_associate(p, impl="oracle")
    assert np.array_equal(g["cur_assoc"], o["cur_assoc"]) and np.array_equal(g["n_added"], o["n_added"])
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ASSOC_CASES))
def test_gpu_line_assoc_case(gpu_ctx, name):
    p, exp = _assoc_case(name)
    _check_assoc_expect(p, exp, _assoc_gpu_vs_oracle(p, gpu_ctx))


@pytest.mark.gpu
def test_gpu_line_assoc_monocular_batch(gpu_ctx):
    p = synth.make_line_assoc_batch(32, 300, 250, 64, 33, n_cand=40)
    p["monocular"] = 1
    g = _assoc_gpu_vs_oracle(p, gpu_ctx)
    assert ((g["cur_assoc"] >= 0) & (p["cur_line_match"] < 0)).sum() > 100


@pytest.mark.gpu
def test_gpu_line_assoc_large_frames(gpu_ctx):
    """frames of 1500 and 3000 current lines: the taken bitset spans more than one word per lane"""
    p = synth.make_line_assoc_batch(4, 1200, 1500, 32, 35, n_cand=40)
    assert _assoc_gpu_vs_oracle(p, gpu_ctx)["n_added"].min() > 300
    p = synth.make_line_assoc_batch(2, 2000, 3000, 32, 36, n_cand=40)
    _assoc_gpu_vs_oracle(p, gpu_ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["cand_negative", "cand_past_frame", "right_match_past_frame"])
def test_gpu_line_assoc_rejects_bad_indices(gpu_ctx, bad):
    p = synth.make_line_assoc_batch(3, 40, 30, 16, 37, n_cand=5)
    _assoc_gpu_vs_oracle(p, gpu_ctx)
    assert gpu_ctx.launch_count() > 0
    q = dict(p)
    if bad == "right_match_past_frame":
        q["cur_line_match"] = p["cur_line_match"].copy()
        q["cur_line_match"][int(p["cur_off"][1])] = int(p["right_off"][2] - p["right_off"][1])   # frame 1's right-line count
        key = "cur_line_match"
    else:
        q["cand_idx"] = p["cand_idx"].copy()
        q["cand_idx"][int(p["cand_off"][p["ml_off"][1]])] = -1 if bad == "cand_negative" else 30   # frame 1 has 30 lines
        key = "cand_idx"
    _expect_rejected(gpu_ctx, lambda: api.line_associate(q, impl="gpu", ctx=gpu_ctx), LLD_ERR_ARG, key)


@pytest.mark.gpu
def test_gpu_line_assoc_monocular_ignores_right_match(gpu_ctx):
    """the monocular arm reads no right line, so it accepts any right-match value"""
    p = synth.make_line_assoc_batch(2, 40, 30, 16, 38, n_cand=5)
    p["monocular"] = 1
    p["cur_line_match"] = np.full_like(p["cur_line_match"], 10 ** 6)
    _assoc_gpu_vs_oracle(p, gpu_ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MEDOID_CASES))
def test_gpu_medoid_case(gpu_ctx, name):
    off, desc, exp = _medoid_case(name)
    assert api.medoid_float(off, desc, impl="gpu", ctx=gpu_ctx).tolist() == exp


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 32, 72])
@pytest.mark.parametrize("N", [1, 2, 31, 32, 33, 64, 255, 256])
def test_gpu_medoid_float_sizes(gpu_ctx, N, D):
    """every lane slot of k_medoid_float (up to 8 descriptors per lane) on small-integer descriptors, and real-valued ones"""
    off, desc = _small_integer_landmarks(N, D, 1000 * N + D)
    assert np.array_equal(api.medoid_float(off, desc, impl="gpu", ctx=gpu_ctx), api.medoid_float(off, desc, impl="oracle"))
    desc = np.random.default_rng(N + D).normal(0, 2.0, desc.shape).astype(f32)
    assert np.array_equal(api.medoid_float(off, desc, impl="gpu", ctx=gpu_ctx), api.medoid_float(off, desc, impl="oracle"))


@pytest.mark.gpu
@pytest.mark.parametrize("N", [255, 256])
def test_gpu_medoid_orb_capacity(gpu_ctx, N):
    rng = np.random.default_rng(N)
    off = np.array([0, N, 2 * N], np.int32)
    base = rng.integers(0, 256, 32, dtype=np.uint8)
    desc = np.stack([_flip(base, int(k), int(s)) for k, s in zip(rng.integers(0, 40, 2 * N), rng.integers(0, 200, 2 * N))])
    assert np.array_equal(api.medoid_orb(off, desc, impl="gpu", ctx=gpu_ctx), api.medoid_orb(off, desc, impl="oracle"))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["orb", "float"])
def test_gpu_medoid_rejects_257_observations(gpu_ctx, kind):
    off = np.array([0, 3, 3 + 257], np.int32)
    if kind == "orb":
        desc = np.zeros((260, 32), np.uint8)
        call = lambda: api.medoid_orb(off, desc, impl="gpu", ctx=gpu_ctx)      # noqa: E731
    else:
        desc = np.zeros((260, 4), f32)
        call = lambda: api.medoid_float(off, desc, impl="gpu", ctx=gpu_ctx)    # noqa: E731
    _expect_rejected(gpu_ctx, call, LLD_ERR_UNSUPPORTED, "257 observations", "at most 256")


@pytest.mark.gpu
def test_gpu_medoid_twenty_thousand_landmarks(gpu_ctx):
    off, desc = _medoid_landmarks(41, n_lm=20000, max_obs=24)
    assert np.array_equal(api.medoid_orb(off, desc, impl="gpu", ctx=gpu_ctx), api.medoid_orb(off, desc, impl="oracle"))
    off, desc = _medoid_landmarks(42, n_lm=20000, max_obs=24, dim=32)
    assert np.array_equal(api.medoid_float(off, desc, impl="gpu", ctx=gpu_ctx), api.medoid_float(off, desc, impl="oracle"))
