"""The observation pipeline's kernels (csrc/hlynr_post.cu, C ABI include/hlynr_post.h) driven directly with synthetic frames
and done lists, against a float64 numpy reference of the same algorithm (oracle/sb3_post.py fed the exact float32 frames).
No simulator: every frame, reward and done record is made here, so the sizes, stack depths and episode patterns can be
chosen where the kernels go wrong.

What is pinned, per step:
  (a) the un-normalised stack (hlynr_post_original), the per-env ages and discounted returns: bit for bit;
  (b) the normalised output against f32(clip((x - mean) / sqrt(var + eps))) in float64 with the DEVICE's mean / var (so the
      bound does not depend on how the statistics were summed): <= ULP_TOL float ulps, an absolute floor only where the
      reference is within 2^-40 |mean| inv_std of 0, clipped values exactly +-clip; and bit for bit against the float32
      emulation of normalize_kernel's op sequence (emulate_normalize);
  (c) terminal rows and hlynr_post_normalize rows (float64 arithmetic) within 1 ulp of the reference; the rows that differ
      (rounding ties of the product against the quotient) are counted;
  (d) obs_rms / ret_rms against the reference: bit for bit with dyadic frames, else within STAT_C * 2^-52 times a second
      moment (check_stats); count exact; the incrementally maintained column sums within 1e-9 of their scale
      (hlynr_post_check_sums).
The grid-stride loops run more than one pass: sizes are derived from the SM count (loop_thresholds).
Also here: hlynr_bootstrap_timeouts and hlynr_gae, the two rollout kernels that read the same done list, bit for bit.
The worst observed ratio of each assertion class is printed as a `post_reference` line (run pytest with -s to see it)."""
import ctypes as C
import json

import numpy as np
import pytest

from hlynr_intercept_b200 import abi
from oracle import sb3_post

F32, F64 = np.float32, np.float64
CLIP, EPS, GAMMA = 10.0, 1e-8, 0.99
ULP_TOL = 3                 # normalize_kernel against the float64 reference (the bound stated in hlynr_post.cu)
NEAR0_ZONE = 2.0 ** -40     # |reference| <= NEAR0_ZONE |mean| inv_std: the float pair hi + lo misses the mean by up to 2^-49 |mean|
NEAR0_FLOOR = 2.0 ** -46    # ... so there the error may reach this floor (times |mean| inv_std) instead of ULP_TOL ulps
# |device - reference| of mean / var in units of 2^-52 times a second moment (check_stats): the summation orders differ
# (two-stage column sums and incremental lag sums against numpy's pairwise sums of the whole stack).  Worst observed on a B200
# (printed as obs_ratio / ret_ratio): 2420 for obs_rms (400 009 envs, 26-D/1), 2.0 for ret_rms; each bound is within 10x.
STAT_C, RET_C = 16384.0, 16.0
SUMS_RTOL = 1e-9            # hlynr_post_check_sums against the scale of the sums

WORST = {}                  # assertion class -> worst observed value, or a count (printed per test)


@pytest.fixture(autouse=True)
def _fresh_worst():
    WORST.clear()


def _note(key, value):
    WORST[key] = max(WORST.get(key, 0), value)


def _count(key, value):
    WORST[key] = WORST.get(key, 0) + value


def _report(name):
    print("post_reference", json.dumps({"test": name, **{k: (float(v) if isinstance(v, float) else int(v)) for k, v in WORST.items()}}))
    WORST.clear()


# ---------------------------------------------------------------------------------------------------------------------------
# float32 emulation of normalize_kernel / normalize1_kernel and the float64 reference
# ---------------------------------------------------------------------------------------------------------------------------
def emulate_normalize(x, mean, var, eps=EPS, clip=CLIP):
    """The kernels' op sequence in numpy float32: inv_std = 1 / sqrt(var + eps) in float64 (merge_kernel), the mean split
    into m_hi = f32(mean), m_lo = f32(mean - m_hi), then fminf(fmaxf(((x - m_hi) - m_lo) * f32(inv_std), -clip), clip)."""
    inv = 1.0 / np.sqrt(np.asarray(var, F64) + eps)
    mean = np.asarray(mean, F64)
    mh = mean.astype(F32)
    ml = (mean - mh.astype(F64)).astype(F32)
    w = ((np.asarray(x, F32) - mh) - ml) * inv.astype(F32)
    return np.minimum(np.maximum(w, F32(-clip)), F32(clip))


def reference64(x, mean, var, eps=EPS, clip=CLIP):
    """SB3's normalize_obs in float64, before its cast to float32."""
    return np.clip((np.asarray(x, F32).astype(F64) - mean) / np.sqrt(var + eps), -clip, clip)


def _ordered(a):
    i = np.asarray(a, F32).view(np.int32).astype(np.int64)
    return np.where(i < 0, -(i & 0x7FFFFFFF), i)


def ulp_dist(a, b):
    """Distance in float32 steps (+0 and -0 are the same point)."""
    return np.abs(_ordered(a) - _ordered(b))


def normalize_errors(got, x, mean, var):
    """(ulp distance to the reference, mask of the near-zero zone, |got - ref64| / floor) of kernel outputs `got`."""
    ref64 = reference64(x, mean, var)
    scale = np.abs(mean) / np.sqrt(var + EPS)
    u = ulp_dist(got, ref64.astype(F32))
    near0 = np.abs(ref64) <= NEAR0_ZONE * scale
    floor = np.where(near0, np.abs(got.astype(F64) - ref64) / np.maximum(NEAR0_FLOOR * scale, 1e-300), 0.0)
    return u, near0, floor, ref64


# ---------------------------------------------------------------------------------------------------------------------------
# CPU: the emulation and the 3-ulp bound
# ---------------------------------------------------------------------------------------------------------------------------
def test_normalize_emulation_bound_cpu():
    """The kernel's float op sequence (emulated) is within 3 ulp of the float64 reference on unit-scale and offset-dominant
    data, 3 ulp is reached (the example below: obs - m_hi rounds in the operands' binade and the result lies one binade lower),
    and without m_lo the error on an offset-dominant channel is far beyond it."""
    x = np.array([0.03819734], F32)
    mean, var = np.array([1.0878614730224259]), np.array([1.1116040115333286])
    got = emulate_normalize(x, mean, var)
    assert got[0] == F32(-0.9955779) and reference64(x, mean, var).astype(F32)[0] == F32(-0.99557805)
    assert ulp_dist(got, reference64(x, mean, var).astype(F32))[0] == 3
    rng = np.random.default_rng(11)
    worst, n3 = 0, 0
    for mean_lo, mean_hi, spread in ((-1.5, 1.5, 1.0), (9.95, 10.05, 0.05), (999.0, 1001.0, 1.0), (-2.0, -2.0, 1e-5)):
        m = rng.uniform(mean_lo, mean_hi, 4096)
        v = rng.uniform(0.25, 2.0, 4096) * spread ** 2
        xs = (m + rng.normal(0, 1, (256, 4096)) * np.sqrt(v)).astype(F32)
        u, near0, floor, _ = normalize_errors(emulate_normalize(xs, m, v), xs, m, v)
        assert (u[~near0] <= ULP_TOL).all(), int(u[~near0].max())
        assert (floor <= 1.0).all()
        worst, n3 = max(worst, int(u[~near0].max())), n3 + int((u[~near0] == 3).sum())
    assert worst == ULP_TOL and n3 > 0
    # offset-dominant channel: the float pair is what keeps the cancellation
    m, v = np.full(1, 1000.0 + 1.0 / 3.0), np.full(1, 1e-4)
    xs = (m + rng.normal(0, 1e-2, (4096, 1))).astype(F32)
    mh = m.astype(F32)
    no_lo = ((xs - mh) * (1.0 / np.sqrt(v + EPS)).astype(F32)).astype(F32)
    assert ulp_dist(no_lo, reference64(xs, m, v).astype(F32)).max() > 1000
    assert ulp_dist(emulate_normalize(xs, m, v), reference64(xs, m, v).astype(F32)).max() <= ULP_TOL


def test_vecnormalize_update_is_step_without_normalisation_cpu():
    """sb3_post.VecNormalize.update (the statistics half of step) leaves obs_rms, ret_rms and the returns as step does."""
    rng = np.random.default_rng(3)
    a, b = sb3_post.VecNormalize(5, (3,)), sb3_post.VecNormalize(5, (3,))
    for t in range(4):
        obs, rew, dones = rng.normal(size=(5, 3)), rng.normal(size=5).astype(F32), rng.uniform(size=5) < 0.4
        a.training = b.training = t != 2
        a.step(obs, rew, dones, {})
        b.update(obs, rew, dones)
        for x, y in ((a.obs_rms.mean, b.obs_rms.mean), (a.obs_rms.var, b.obs_rms.var), (a.returns, b.returns),
                     (a.ret_rms.mean, b.ret_rms.mean), (a.ret_rms.var, b.ret_rms.var)):
            assert np.array_equal(x, y)


# ---------------------------------------------------------------------------------------------------------------------------
# synthetic data
# ---------------------------------------------------------------------------------------------------------------------------
def make_frame(rng, n, F, kind):
    """float32 [n, F].  kind 'mixed': channel c % 4 picks the generator -- 0 realistic (values in [-2, 1], channels held at
    the -2.0 'no track' fill for 90 % of the envs, 5 % exactly +-1), 1 offset-dominant (10 +- 0.05 or 1e3 +- 1), 2 near-constant
    (variance below eps), 3 clip edges (unit normal with +-0.0 and 0.1 % outliers at +-1e5 that normalise beyond the clip).
    kind 'dyadic': small integers / 8, so every sum over a power-of-two batch is exact in float64."""
    if kind == "dyadic":
        return (rng.integers(-16, 17, (n, F)) / 8.0).astype(F32)
    x = np.empty((n, F), F32)
    for c in range(F):
        g = c % 4
        if g == 0:
            col = rng.uniform(-2.0, 1.0, n)
            if c % 8 == 0:
                col[rng.uniform(size=n) < 0.9] = -2.0
            pm = rng.uniform(size=n) < 0.05
            col[pm] = rng.choice([-1.0, 1.0], int(pm.sum()))
        elif g == 1:
            col = 10.0 + rng.uniform(-0.05, 0.05, n) if c % 8 == 1 else 1e3 + rng.uniform(-1.0, 1.0, n)
        elif g == 2:
            col = (0.5 if c % 8 == 2 else -2.0) + rng.uniform(-1e-5, 1e-5, n)
        else:
            col = rng.normal(0.0, 1.0, n)
            col[rng.uniform(size=n) < 0.05] = 0.0
            neg0 = rng.uniform(size=n) < 0.05
            col[neg0] = -0.0
            out = rng.uniform(size=n) < 0.001
            col[out] = rng.choice([-1e5, 1e5], int(out.sum()))
        x[:, c] = col
    return x


def clip_edge_frame(rng, n, F):
    """Frames for the statistics mean 0.25, var + eps = 4 (inv_std 0.5 exactly): 20.25 / -19.75 normalise to exactly +-clip,
    +-1/4 outwards beyond it, inwards inside it; +-0.0 and 0.25 give -0.125 and 0; +-30 far beyond.  Multiples of 1/4 below
    32, so numpy's two-pass variance over a dyadic batch of 4096 stays exact too."""
    vals = np.array([20.25, -19.75, 20.5, -20.0, 20.0, -19.5, 0.0, -0.0, 0.25, 30.0, -30.0], F32)
    return vals[rng.integers(0, len(vals), (n, F))]


def done_pattern(rng, n, p, prev_done):
    """(terminated, truncated) uint8 [n]: each env finishes with probability p, an env that finished on the previous step
    finishes again with probability 1/2 (an episode of one step); a finished env is terminated-only or truncated-only."""
    done = (rng.uniform(size=n) < p) | (prev_done & (rng.uniform(size=n) < 0.5))
    term = done & (rng.uniform(size=n) < 0.5)
    return term.astype(np.uint8), (done & ~term).astype(np.uint8)


# ---------------------------------------------------------------------------------------------------------------------------
# the device pipeline through its C ABI
# ---------------------------------------------------------------------------------------------------------------------------
def loop_thresholds(sm_count, F, k):
    """Smallest n at which each grid-stride / fold loop of hlynr_post.cu runs a second pass (grids are capped at 8 blocks
    per SM, blocks_for)."""
    cap = 8 * sm_count
    if F % 2 == 0:
        lanes = max(512 // (F * k // 2), 1)
    else:
        lanes = 512 // (F * k)
    return {"colsum": cap * 16, "fold_col": 256 * 16, "fold_ret": 256 * 256, "returns": cap * 256, "normalize": cap * lanes * 8}


class Post:
    def __init__(self, n, F, k, clip=CLIP, eps=EPS, gamma=GAMMA):
        import torch

        from hlynr_intercept_b200 import _lib

        self.torch, self._lib, self.L = torch, _lib, _lib.load()
        self.n, self.F, self.k, self.D = n, F, k, F * k
        h = C.c_void_p()
        _lib.check(self.L.hlynr_post_create_frames(n, 0, F, k, clip, eps, gamma, C.byref(h)))
        self.h = h
        self.dev = torch.device("cuda", 0)
        t, d = torch, self.dev
        self.out = t.empty((n, self.D), dtype=t.float32, device=d)
        self.orig = t.empty((n, self.D), dtype=t.float32, device=d)
        self.term_out = t.empty((n, self.D), dtype=t.float32, device=d)
        self.rec_dt = abi.done_record_numpy_dtype()
        self.recs = t.zeros(n * self.rec_dt.itemsize, dtype=t.uint8, device=d)
        self.counter = t.zeros(1, dtype=t.int32, device=d)

    def _p(self, x):
        return C.c_void_p(x.data_ptr())

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.dev).cuda_stream)

    def write_frame(self, frame):
        """Writes the frame into the ring slot of the next reset / step, through a zero-copy view (as the step kernel does)."""
        from hlynr_intercept_b200.sim import _tensor_from_ptr

        p = C.c_void_p()
        self._lib.check(self.L.hlynr_post_obs_target(self.h, C.byref(p)))
        _tensor_from_ptr(self.torch, p.value, (self.n, self.F), self.torch.float32, self.dev).copy_(self.torch.from_numpy(frame))

    def reset(self, frame, training):
        self.write_frame(frame)
        self._lib.check(self.L.hlynr_post_reset(self.h, self._p(self.out), int(training), self._stream()))
        return self.out.cpu().numpy()

    def step(self, frame, rew, term, trunc, recs, training):
        t = self.torch
        self.write_frame(frame)
        rew_d, te_d, tr_d = (t.from_numpy(np.ascontiguousarray(a)).to(self.dev) for a in (rew, term, trunc))
        if len(recs):
            self.recs[: len(recs) * self.rec_dt.itemsize].copy_(t.from_numpy(recs.view(np.uint8).reshape(-1)))
        self.counter.fill_(len(recs))
        self._lib.check(self.L.hlynr_post_step(self.h, self._p(rew_d), self._p(te_d), self._p(tr_d), self._p(self.recs), self._p(self.counter),
                                               self.n, self._p(self.out), self._p(self.term_out), int(training), self._stream()))
        return self.out.cpu().numpy(), self.term_out[: len(recs)].cpu().numpy()

    def original(self):
        self._lib.check(self.L.hlynr_post_original(self.h, self._p(self.orig), self._stream()))
        return self.orig.cpu().numpy()

    def normalize_rows(self, x):
        xd = self.torch.from_numpy(np.ascontiguousarray(x, F32)).to(self.dev)
        out = self.torch.empty_like(xd)
        self._lib.check(self.L.hlynr_post_normalize(self.h, self._p(xd), xd.shape[0], self._p(out), self._stream()))
        return out.cpu().numpy()

    def stats(self):
        mean, var = np.zeros(self.D), np.zeros(self.D)
        c, rm, rv, rc = C.c_double(), C.c_double(), C.c_double(), C.c_double()
        self._lib.check(self.L.hlynr_post_get_stats(self.h, mean.ctypes.data_as(C.c_void_p), var.ctypes.data_as(C.c_void_p), C.byref(c),
                                                    C.byref(rm), C.byref(rv), C.byref(rc), self._stream()))
        return dict(mean=mean, var=var, count=c.value, ret_mean=rm.value, ret_var=rv.value, ret_count=rc.value)

    def set_stats(self, mean, var, count, ret_mean, ret_var, ret_count):
        mean, var = np.ascontiguousarray(mean, F64), np.ascontiguousarray(var, F64)
        self._lib.check(self.L.hlynr_post_set_stats(self.h, mean.ctypes.data_as(C.c_void_p), var.ctypes.data_as(C.c_void_p), count, ret_mean,
                                                    ret_var, ret_count, self._stream()))

    def ages_returns(self):
        """Per-env ages and discounted returns: the AGE / RETURNS sections of a snapshot image."""
        info, nbytes = abi.HlynrPostSnapshotInfo(), C.c_size_t()
        self._lib.check(self.L.hlynr_post_snapshot_layout(self.h, C.byref(info), C.byref(nbytes)))
        img = self.torch.empty(nbytes.value, dtype=self.torch.uint8, device=self.dev)
        self._lib.check(self.L.hlynr_post_snapshot_save(self.h, self._p(img), C.byref(info), self._stream()))
        img = img.cpu().numpy()
        a, r = info.section_offset[1], info.section_offset[2]
        return img[a: a + self.n].copy(), img[r: r + 8 * self.n].view(F64).copy()

    def check_sums(self):
        d = C.c_double()
        self._lib.check(self.L.hlynr_post_check_sums(self.h, 0, C.byref(d), self._stream()))
        return d.value

    def close(self):
        if self.h:
            self.L.hlynr_post_destroy(self.h)
            self.h = None


class Reference:
    """sb3_post.StackedObservations + VecNormalize (statistics half) fed the same float32 frames, plus the per-env age."""

    def __init__(self, n, F, k):
        self.n, self.F, self.k = n, F, k
        self.stack = sb3_post.StackedObservations(n, k, F)
        self.vn = sb3_post.VecNormalize(n, (F * k,), clip_obs=CLIP, gamma=GAMMA, epsilon=EPS)
        self.age = np.zeros(n, np.uint8)

    def reset(self, frame, training):
        self.vn.training = training
        stacked = self.stack.reset(frame)
        self.vn.reset(stacked.astype(F64))
        self.age[:] = 0
        return stacked

    def step(self, frame, rew, dones, tobs, training):
        """dones bool [n]; tobs {env: terminal_obs[0:F]} -> (stacked float32 [n, F k], {env: stacked terminal observation})."""
        self.vn.training = training
        infos = {e: {"terminal_observation": o} for e, o in tobs.items()}
        stacked, infos = self.stack.update(frame, dones, infos)
        self.vn.update(stacked.astype(F64), rew.astype(F64), dones)
        self.age = np.where(dones, 0, np.minimum(self.age.astype(np.int64) + 1, self.k - 1)).astype(np.uint8)
        return stacked, {e: i["terminal_observation"] for e, i in infos.items()}


def make_records(rng, pd, term, trunc, tobs_frame):
    """The step's done list: one record per finished env (env, flags, terminal_obs[0:26]) in a shuffled order."""
    envs = np.nonzero(term | trunc)[0]
    rng.shuffle(envs)
    recs = np.zeros(len(envs), pd.rec_dt)
    recs["env"] = envs
    recs["flags"] = np.where(term[envs] != 0, abi.DONE_TERMINATED, abi.DONE_TRUNCATED)
    recs["terminal_obs"][:, : pd.F] = tobs_frame[envs]
    recs["terminal_obs"][:, pd.F:] = 7.0   # past the frame width: must not be read
    return recs


# ---------------------------------------------------------------------------------------------------------------------------
# per-step checks
# ---------------------------------------------------------------------------------------------------------------------------
CHUNK = 1 << 16


def check_normalized(got, stacked, mean, var, what):
    """(b): kernel output against the emulation (bits) and the float64 reference (ULP_TOL / floor / exact clip)."""
    for r0 in range(0, got.shape[0], CHUNK):
        g, x = got[r0: r0 + CHUNK], stacked[r0: r0 + CHUNK]
        emu = emulate_normalize(x, mean, var)
        diff = g.view(np.uint32) != emu.view(np.uint32)
        if diff.any():
            r, c = np.argwhere(diff)[0]
            pytest.fail(f"{what}: {int(diff.sum())} outputs differ from the float32 emulation of the kernel, first [{r0 + r}, {c}]: "
                        f"x {x[r, c]!r} mean {mean[c]!r} var {var[c]!r}: got {g[r, c]!r}, emulation {emu[r, c]!r}")
        u, near0, floor, ref64 = normalize_errors(g, x, mean, var)
        far = u[~near0]
        _note("norm_ulp", int(far.max(initial=0)))
        _count("norm_3ulp_outputs", int((far == 3).sum()))
        _note("norm_floor_ratio", float(floor.max(initial=0.0)))
        assert far.max(initial=0) <= ULP_TOL, f"{what}: {int(far.max())} ulp from the float64 reference"
        assert floor.max(initial=0.0) <= 1.0, f"{what}: near zero, {floor.max():.3g} x the floor from the reference"
        scale = 1.0 / np.sqrt(var + EPS)
        beyond = np.abs((x.astype(F64) - mean) * scale) >= CLIP * (1 + 2.0 ** -20)
        assert (g[beyond] == np.sign(ref64[beyond]).astype(F32) * F32(CLIP)).all(), f"{what}: a clipped output is not exactly +-clip"


def check_double_path(got, x, mean, var, what):
    """(c): rows normalised in float64 (terminal_kernel, normalize_rows_kernel): within 1 ulp, counting the rows that differ."""
    if got.size == 0:
        return
    ref = reference64(x, mean, var).astype(F32)
    u = ulp_dist(got, ref)
    _note("double_path_ulp", int(u.max()))
    _count("double_path_ties", int((u != 0).sum()))
    assert u.max() <= 1, f"{what}: {int(u.max())} ulp from the float64 reference"


def check_stats(s, vn, exact, frame_m2, what):
    """(d): obs_rms / ret_rms of the device against the reference's.  The scale of obs_rms errors is var + mean^2 of the
    feature plus frame_m2, the largest mean(x^2) of its channel over the frames written so far: the per-lag sums are kept
    incrementally (S[d] = S[d-1] - frames of the finished envs), so when a lag empties -- every env finished -- what is left of
    its sums is the rounding of that cancellation, which scales with the frames that left, not with the (near-zero) moments
    of the lag."""
    rms, ret = vn.obs_rms, vn.ret_rms
    assert s["count"] == rms.count and s["ret_count"] == ret.count, what
    if exact:
        assert np.array_equal(s["mean"], rms.mean) and np.array_equal(s["var"], rms.var), \
            f"{what}: obs_rms not bit for bit: mean off by {np.abs(s['mean'] - rms.mean).max():.3g}, var {np.abs(s['var'] - rms.var).max():.3g}"
    err = np.maximum(np.abs(s["mean"] - rms.mean), np.abs(s["var"] - rms.var))
    for name, e, scale, bound in (("obs_rms", err, rms.var + rms.mean ** 2 + np.tile(frame_m2, len(err) // len(frame_m2)), STAT_C),
                                  ("ret_rms", max(abs(s["ret_mean"] - ret.mean), abs(s["ret_var"] - ret.var)), ret.var + ret.mean ** 2,
                                   RET_C)):
        r = float(np.max(e / np.maximum(2.0 ** -52 * scale, 1e-300)))
        _note(name[:3] + "_ratio", r)
        assert r <= bound, f"{what}: {name} differs from the reference by {r:.3g} x 2^-52 x its scale"


def check_sums(pd, stacked, what):
    """(d): the incrementally maintained per-lag sums against a recomputation from the ring, relative to their scale."""
    d = pd.check_sums()
    x = stacked.astype(F64)
    scale = max(float(np.abs(x).sum(0).max()), float((x * x).sum(0).max()), 1.0)
    _note("sums_rel", d / scale)
    assert d <= SUMS_RTOL * scale, f"{what}: check_sums {d:.3g} against a scale of {scale:.3g}"


def check_state(pd, ref, stacked, what):
    """(a): stack, ages and returns bit for bit."""
    orig = pd.original()
    assert np.array_equal(orig.view(np.uint32), stacked.view(np.uint32)), \
        f"{what}: un-normalised stack differs in {int((orig.view(np.uint32) != stacked.view(np.uint32)).sum())} entries"
    age, ret = pd.ages_returns()
    assert np.array_equal(age, ref.age), f"{what}: per-env ages differ for {int((age != ref.age).sum())} envs"
    assert np.array_equal(ret.view(np.int64), ref.vn.returns.view(np.int64)), \
        f"{what}: discounted returns differ for {int((ret != ref.vn.returns).sum())} envs, by up to {np.abs(ret - ref.vn.returns).max():.3g}"


def run_case(n, F, k, p, kind="mixed", T=14, seed=0, events=True, sums_every=1):
    """Reset, T steps (every env finishes on step 3; training off on steps 6-7; a mid-run reset on step 9), then frozen
    statistics set by hand (var 0, var 1e20, and the exact-clip statistics), every output checked on every step."""
    rng = np.random.default_rng(seed + 1000 * k + F)
    pd, ref = Post(n, F, k), Reference(n, F, k)
    exact = kind == "dyadic"
    m2 = np.zeros(F)

    def written(frame):   # the largest mean(x^2) per channel of the frames written so far (check_stats)
        m2[:] = np.maximum(m2, (frame.astype(F64) ** 2).mean(0))
        return frame

    try:
        frame = written(make_frame(rng, n, F, kind))
        out = pd.reset(frame, True)
        stacked = ref.reset(frame, True)
        s = pd.stats()
        check_state(pd, ref, stacked, f"reset")
        check_normalized(out, stacked, s["mean"], s["var"], "reset")
        check_stats(s, ref.vn, exact, m2, "reset")
        prev = np.zeros(n, bool)
        training = True
        for t in range(1, T + 1):
            what = f"n {n} F {F} k {k} p {p} step {t}"
            if events and t == 9:   # hlynr_post_reset in the middle of a run: returns and stacks start again
                frame = written(make_frame(rng, n, F, kind))
                out = pd.reset(frame, training)
                stacked = ref.reset(frame, training)
                s = pd.stats()
                check_state(pd, ref, stacked, what)
                check_normalized(out, stacked, s["mean"], s["var"], what)
                check_stats(s, ref.vn, exact, m2, what)
                prev[:] = False
                continue
            if events:
                training = not (6 <= t <= 7)
            term, trunc = done_pattern(rng, n, 1.0 if (events and t == 3) else p, prev)
            dones = (term | trunc) != 0
            frame, tobs_frame = written(make_frame(rng, n, F, kind)), make_frame(rng, n, F, kind)
            rew = rng.normal(0, 1, n).astype(F32)
            recs = make_records(rng, pd, term, trunc, tobs_frame)
            out, term_rows = pd.step(frame, rew, term, trunc, recs, training)
            stacked, tobs = ref.step(frame, rew, dones, {int(e): tobs_frame[e].copy() for e in np.nonzero(dones)[0]}, training)
            s = pd.stats()
            check_state(pd, ref, stacked, what)
            check_normalized(out, stacked, s["mean"], s["var"], what)
            if len(recs):
                want = np.stack([tobs[int(e)] for e in recs["env"]])
                check_double_path(term_rows, want, s["mean"], s["var"], what + " terminal rows")
            check_stats(s, ref.vn, exact, m2, what)
            if t % sums_every == 0:
                check_sums(pd, stacked, what)
            prev = dones
        if events:
            # frozen statistics set by hand (VecNormalize.load): var 0, a very large var, and mean 0.25 / var + eps = 4
            s = pd.stats()
            D = F * k
            for mean, var, kind2 in ((s["mean"], np.zeros(D), kind), (s["mean"], np.full(D, 1e20), kind),
                                     (np.full(D, 0.25), np.full(D, 4.0 - EPS), "clip")):
                assert kind2 != "clip" or (4.0 - EPS) + EPS == 4.0
                pd.set_stats(mean, var, s["count"], s["ret_mean"], s["ret_var"], s["ret_count"])
                ref.vn.obs_rms.mean, ref.vn.obs_rms.var = mean.copy(), var.copy()
                term, trunc = done_pattern(rng, n, 0.3, prev)
                dones = (term | trunc) != 0
                frame = written(clip_edge_frame(rng, n, F) if kind2 == "clip" else make_frame(rng, n, F, kind2))
                tobs_frame = clip_edge_frame(rng, n, F) if kind2 == "clip" else make_frame(rng, n, F, kind2)
                rew = rng.normal(0, 1, n).astype(F32)
                recs = make_records(rng, pd, term, trunc, tobs_frame)
                out, term_rows = pd.step(frame, rew, term, trunc, recs, False)
                stacked, tobs = ref.step(frame, rew, dones, {int(e): tobs_frame[e].copy() for e in np.nonzero(dones)[0]}, False)
                what = f"n {n} F {F} k {k} set_stats var {var[0]:.3g}"
                s2 = pd.stats()
                assert np.array_equal(s2["mean"], mean) and np.array_equal(s2["var"], var)
                check_state(pd, ref, stacked, what)
                check_normalized(out, stacked, mean, var, what)
                if len(recs):
                    check_double_path(term_rows, np.stack([tobs[int(e)] for e in recs["env"]]), mean, var, what + " terminal rows")
                rows = stacked[: min(n, 4096)]
                check_double_path(pd.normalize_rows(rows), rows, mean, var, what + " normalize rows")
                if kind2 == "clip":
                    hit = stacked == F32(20.25)
                    assert (out[hit] == F32(CLIP)).all() and (out[stacked == F32(-19.75)] == F32(-CLIP)).all()
                    assert (out[(stacked == 0) & ~np.signbit(stacked)] == F32(-0.125)).all()
                prev = dones
            # training resumes from var 0 (the last set_stats but one) on a fresh step
            pd.set_stats(s["mean"], np.zeros(D), s["count"], s["ret_mean"], s["ret_var"], s["ret_count"])
            ref.vn.obs_rms.mean, ref.vn.obs_rms.var = s["mean"].copy(), np.zeros(D)
            term, trunc = done_pattern(rng, n, p, prev)
            dones = (term | trunc) != 0
            frame, tobs_frame = written(make_frame(rng, n, F, kind)), make_frame(rng, n, F, kind)
            rew = rng.normal(0, 1, n).astype(F32)
            recs = make_records(rng, pd, term, trunc, tobs_frame)
            out, _ = pd.step(frame, rew, term, trunc, recs, True)
            stacked, _ = ref.step(frame, rew, dones, {}, True)
            s = pd.stats()
            check_state(pd, ref, stacked, "training after set_stats")
            check_normalized(out, stacked, s["mean"], s["var"], "training after set_stats")
            check_stats(s, ref.vn, exact, m2, "training after set_stats")
            check_sums(pd, stacked, "training after set_stats")
    finally:
        pd.close()


def _sm_count():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------------
# GPU tests of the pipeline
# ---------------------------------------------------------------------------------------------------------------------------
GRID_N = 4097   # > 256 colsum blocks (the fold loop's second pass over the column words); p = 0.3 gives several done-list passes


@pytest.mark.gpu
@pytest.mark.parametrize("F", [26, 17])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 7, 8])
def test_pipeline_stack_depths(F, k):
    """Every frame width x stack depth at 4097 envs, a different done rate per depth."""
    th = loop_thresholds(_sm_count(), F, k)
    assert GRID_N > th["fold_col"]
    p = (0.0, 0.02, 0.3, 1.0)[k % 4]
    run_case(GRID_N, F, k, p)
    _report(f"stack_depths/F{F}/k{k}/p{p}")


@pytest.mark.gpu
@pytest.mark.parametrize("F", [26, 17])
@pytest.mark.parametrize("n", [1, 15, 16, 17, 18945])
def test_pipeline_sizes(F, n):
    """Sizes at the edges of a block's env lanes, and one past the colsum kernel's first grid-stride pass (18 944 = 8 x 148 x 16
    on a B200; checked against the SM count)."""
    if n == 18945:
        th = loop_thresholds(_sm_count(), F, 4)
        n = max(n, th["colsum"] + 1)
    run_case(n, F, 4, 0.3 if n > 17 else 0.5, seed=n)
    _report(f"sizes/F{F}/n{n}")


@pytest.mark.gpu
@pytest.mark.parametrize("F,k", [(26, 1), (26, 4), (26, 8), (17, 1)])
def test_pipeline_past_every_grid_stride_loop(F, k):
    """One size past every loop threshold of the configuration (returns, normalise, colsum, both fold ranges), a few steps."""
    th = loop_thresholds(_sm_count(), F, k)
    n = max(400009, max(th.values()) + 9)
    assert all(n > v for v in th.values()), th
    run_case(n, F, k, 0.02, T=4, events=False, sums_every=2)
    _report(f"large/F{F}/k{k}/n{n}")


@pytest.mark.gpu
@pytest.mark.parametrize("F,k", [(26, 1), (26, 4), (17, 3), (26, 8)])
def test_pipeline_dyadic_statistics_bit_exact(F, k):
    """Dyadic frames over a power-of-two batch: every sum is exact, so obs_rms must equal the restatement bit for bit (a merge
    that contracts SB3's separately rounded products into FMAs, or sums that miss a frame, shows here)."""
    run_case(4096, F, k, 0.3, kind="dyadic")
    _report(f"dyadic/F{F}/k{k}")


# ---------------------------------------------------------------------------------------------------------------------------
# the rollout kernels that read the same done list
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("count,rows", [(0, 64), (64, 64), (300, 64), (5000, 4096)])
def test_bootstrap_timeouts(count, rows):
    """rewards[env] += f32(gamma) * V[r] for the truncated-and-not-terminated records r < min(count, rows); the records past
    `rows` that needed a value are counted in *overflow."""
    import torch

    from hlynr_intercept_b200 import _lib

    L = _lib.load()
    n = max(count, rows, 1) + 17
    rng = np.random.default_rng(count + rows)
    dt = abi.done_record_numpy_dtype()
    recs = np.zeros(max(count, 1), dt)
    recs["env"][:count] = rng.permutation(n)[:count]
    recs["flags"][:count] = rng.choice([abi.DONE_TERMINATED, abi.DONE_TRUNCATED, abi.DONE_TERMINATED | abi.DONE_TRUNCATED,
                                        abi.DONE_TRUNCATED | abi.INFO_INTERCEPTED], count)
    rew = rng.normal(0, 1, n).astype(F32)
    tv = rng.normal(0, 5, rows).astype(F32)
    want = rew.copy()
    need = (recs["flags"][:count] & abi.DONE_TRUNCATED != 0) & (recs["flags"][:count] & abi.DONE_TERMINATED == 0)
    m = min(count, rows)
    g = F32(GAMMA)
    for r in np.nonzero(need[:m])[0]:
        want[recs["env"][r]] = want[recs["env"][r]] + g * tv[r]
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    rew_d, tv_d = d(rew), d(tv)
    rec_d = d(recs.view(np.uint8).reshape(-1))
    cnt_d = torch.tensor([count], dtype=torch.int32, device="cuda")
    ovf = torch.zeros(1, dtype=torch.int32, device="cuda")
    p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
    _lib.check(L.hlynr_bootstrap_timeouts(p(rew_d), p(rec_d), p(cnt_d), rows, p(tv_d), GAMMA, p(ovf), 0, None))
    torch.cuda.synchronize()
    assert np.array_equal(rew_d.cpu().numpy().view(np.uint32), want.view(np.uint32))
    assert int(ovf.item()) == int(need[m:].sum())


GAE_CASES = [(T, N) for T in (1, 2, 513) for N in (1, 255, 257)] + [(1, (1 << 20) + 3), (2, (1 << 20) + 3), (8, (1 << 20) + 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 0.0), (1.0, 1.0)])
@pytest.mark.parametrize("pattern", ["random", "all_starts", "all_done"])
@pytest.mark.parametrize("T,N", GAE_CASES)
def test_gae_bit_exact(T, N, gamma, lam, pattern):
    """GAE(lambda) bit for bit against sb3_post.compute_returns_and_advantage: one env, partial and full blocks, 2^20 + 3 envs
    (a partial last block), 513 steps; gamma 1 with lambda 0 and 1; every step an episode start; every env done at the end."""
    import torch

    from hlynr_intercept_b200 import _lib

    L = _lib.load()
    rng = np.random.default_rng(T * 7 + N)
    r = rng.normal(0, 3, (T, N)).astype(F32)
    v = rng.normal(0, 2, (T, N)).astype(F32)
    starts = np.ones((T, N), F32) if pattern == "all_starts" else (rng.uniform(size=(T, N)) < 0.1).astype(F32)
    lv = rng.normal(0, 2, N).astype(F32)
    ld = np.ones(N, bool) if pattern == "all_done" else rng.uniform(size=N) < 0.2
    want_adv, want_ret = sb3_post.compute_returns_and_advantage(r, v, starts, lv, ld, gamma, lam)
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    tr, tv, ts, tlv, tld = d(r), d(v), d(starts), d(lv), d(ld.astype(np.uint8))
    adv, ret = torch.empty_like(tr), torch.empty_like(tr)
    p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
    _lib.check(L.hlynr_gae(p(tr), p(tv), p(ts), p(tlv), p(tld), T, N, gamma, lam, p(adv), p(ret), 0, None))
    torch.cuda.synchronize()
    assert np.array_equal(adv.cpu().numpy().view(np.uint32), want_adv.view(np.uint32))
    assert np.array_equal(ret.cpu().numpy().view(np.uint32), want_ret.view(np.uint32))
