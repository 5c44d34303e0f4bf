"""The fused actor-critic forward (csrc/hlynr_policy.cu) against a float64 restatement of the network, at the LayerNorm,
sampling and size edges where a kernel goes wrong.

forward64() is the reference: weights, input and hidden activations are rounded to bf16 where the kernel rounds them (RNE
through torch.bfloat16), every GEMM accumulates in float64, LayerNorm is two-pass in float64 with each module's eps, then ReLU
and the heads in float64.  The noise reference is Philox4x32-10 from oracle.draws with the kernel's counter layout: counter
(row_lo, row_hi, call_lo, call_hi), the second block with bit 31 of row_hi set, key (seed_lo, seed_hi), float32 Box-Muller.

Tolerances (the worst values observed on a B200 are in DESIGN.md section 12; every bound is at most 10x the worst):
  * mean / value vs forward64: |diff| <= ATOL + 5e-3 |ref| per element (ATOL 5e-3 for the mean, 1e-2 for the value) and mean
    |diff| < 1e-4, with the action head x40 as in test_policy.py so that an error in a hidden layer shows in the outputs.  The
    value head is the more sensitive one (unit gain against 40 x 0.01): one bf16 flip of an H1 activation, which the rounding
    points of the reference cannot rule out, moved one value by 5.8e-3 (worst observed);
  * a common mean that comes out of the GEMM (test_layernorm_with_a_large_common_mean, mode "weight") is held by the fp32
    accumulator, which rounds it at (mean / std) * 2^-24 of the spread before any epilogue sees it; the float64 reference does
    not.  Those cases bound the mean |diff| by 1e-4 (1 + (mean / std) / 20) instead; the LayerNorm statistics of the parent
    commit (E[x^2] - mean^2) fail that bound at every ratio;
  * sampled action vs mean_kernel + exp(log_std) eps_ref: 16 float32 ulp of max(|mean|, |exp(log_std) eps|) (eps differs from
    the reference by the last bits of logf / sincospif, exp(log_std) by __expf, which is not IEEE);
  * log pi vs the float64 Gaussian formula at eps_ref: 16 float32 ulp of the sum of the magnitudes of its terms;
  * output subsets, repeated calls, re-synced weights: bit for bit.
"""
import math
import types

import numpy as np
import pytest

CLUSTERS = [1, 2, 4]
ATOL, VALUE_ATOL, RTOL, MEAN_TOL = 5e-3, 1e-2, 5e-3, 1e-4
ULP_TOL = 16
SEED = 2 ** 32 + 5           # both key words matter
CALLS = 2 ** 32 + 3          # the next call uses counter 2^32 + 4: both counter words matter
LOG_STD = [-0.5, -0.2, 0.0, 0.1, 0.3, -1.0]


def _layers(net):
    mods = list(net.network)
    return [m for m in mods if m.__class__.__name__ == "Linear"], [m for m in mods if m.__class__.__name__ == "LayerNorm"]


def _net(seed=0, device="cuda"):
    """Default init plus non-trivial biases, LayerNorm affine parameters, log_std, and the action head x40 (test_policy._nets)."""
    import torch
    from hlynr_intercept_b200.policy import ReferenceActorCritic

    torch.manual_seed(seed)
    net = ReferenceActorCritic(device=device)
    lins, lns = _layers(net)
    with torch.no_grad():
        for lin, ln in zip(lins, lns):
            lin.bias.normal_(0, 0.2)
            ln.weight.uniform_(0.5, 1.5); ln.bias.normal_(0, 0.3)
        net.action_net.weight.mul_(40.0); net.action_net.bias.normal_(0, 0.1)
        net.value_net.bias.fill_(0.37)
        net.log_std.copy_(torch.tensor(LOG_STD, device=device))
    return net


def _obs(n, seed=0, device="cuda"):
    import torch

    g = torch.Generator(device=device); g.manual_seed(seed)
    obs = (torch.randn(n, 104, device=device, generator=g) * 1.5).clamp(-10, 10)
    obs[:, 7] = 5.0 + 5.0 * torch.rand(n, device=device, generator=g)   # a positive channel in every row (VecNormalize clip 10)
    return obs.contiguous()


def forward64(net, obs, bf16=True, pre=None):
    """(mean [n, 6], value [n]) in float64.  bf16=False: no rounding at all, the plain float64 network.  pre: a list that
    receives the three pre-activations (x W^T + b)."""
    import torch

    if bf16:
        r = lambda t: t.detach().to(torch.bfloat16).double()   # noqa: E731
    else:
        r = lambda t: t.detach().double()   # noqa: E731
    lins, lns = _layers(net)
    x = r(obs)
    for lin, ln in zip(lins, lns):
        y = x @ r(lin.weight).t() + lin.bias.detach().double()
        if pre is not None:
            pre.append(y)
        mu = y.mean(-1, keepdim=True)
        d = y - mu
        var = (d * d).mean(-1, keepdim=True)
        x = r(torch.relu(d / torch.sqrt(var + ln.eps) * ln.weight.detach().double() + ln.bias.detach().double()))
    mean = x @ r(net.action_net.weight).t() + net.action_net.bias.detach().double()
    value = (x @ r(net.value_net.weight).t() + net.value_net.bias.detach().double())[:, 0]
    return mean, value


def eps_ref(seed, counter, n):
    """float32 [n, 6] standard normals the kernel draws for rows 0..n-1 at this seed and call counter."""
    from oracle import draws

    rows = np.arange(n, dtype=np.uint64)
    ctr = np.empty((n, 4), dtype=np.uint32)
    ctr[:, 0] = rows & np.uint64(0xFFFFFFFF)
    ctr[:, 1] = rows >> np.uint64(32)
    ctr[:, 2] = counter & 0xFFFFFFFF
    ctr[:, 3] = counter >> 32
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint32)
    r0 = draws.philox4x32_10(ctr, key)
    ctr[:, 1] |= np.uint32(0x80000000)
    r1 = draws.philox4x32_10(ctr, key)
    return np.concatenate([draws.normals(r0), draws.normals(r1)[:, :2]], axis=-1)


def _fused(net, cluster, seed=SEED):
    from hlynr_intercept_b200.policy import FusedActorCritic

    fused = FusedActorCritic(net, device=0, seed=seed)
    fused.set_option("cluster", cluster)
    return fused


def _mean_value(fused, obs):
    import torch

    m, v = fused.mean_and_value(obs)
    torch.cuda.synchronize()
    return m.clone(), v.clone()


def errors(got, ref, atol=ATOL):
    """(worst |diff| / (atol + RTOL |ref|), mean |diff|, worst |diff|) of a kernel output against the float64 reference."""
    d = (got.double() - ref).abs()
    return float((d / (atol + RTOL * ref.abs())).max()), float(d.mean()), float(d.max())


def _check(fused, net, obs, mean_tol=MEAN_TOL):
    """mean and value of the kernel vs forward64; returns them."""
    import torch

    m, v = _mean_value(fused, obs)
    with torch.no_grad():
        rm, rv = forward64(net, obs)
    for name, got, ref, atol in (("mean", m, rm, ATOL), ("value", v, rv, VALUE_ATOL)):
        assert torch.isfinite(got).all(), name
        worst, mad, dmax = errors(got, ref, atol)
        assert worst <= 1.0, f"{name}: max |diff| {dmax:.3e} exceeds {atol} + {RTOL} |ref|"
        assert mad < mean_tol, f"{name}: mean |diff| {mad:.3e}"
    return m, v


def _sigma(net, obs, layer):
    """Typical spread of a layer's pre-activations over its features (median over rows of the per-row std)."""
    import torch

    pre = []
    with torch.no_grad():
        forward64(net, obs, pre=pre)
    return float(pre[layer].std(-1, unbiased=False).median())


# ---- the reference itself (CPU) -------------------------------------------------------------------------------------------

def test_forward64_without_rounding_is_the_module_in_float64():
    import torch

    net = _net(seed=3, device="cpu").double()
    obs = _obs(300, seed=1, device="cpu")
    with torch.no_grad():
        m, v = forward64(net, obs.double(), bf16=False)
        want_m, want_v = net.mean(obs.double()), net.value(obs.double())
    assert float((m - want_m).abs().max()) <= 1e-12 and float((v - want_v).abs().max()) <= 1e-12


def test_eps_ref_matches_the_oracle_normals_layout():
    """The reference draws row 2 from the counter (2, 0, call_lo, call_hi) with key (seed_lo, seed_hi); both high words matter."""
    from oracle import draws

    e = eps_ref(SEED, CALLS + 1, 3)
    assert e.shape == (3, 6) and e.dtype == np.float32 and np.isfinite(e).all()
    raw = draws.philox4x32_10(np.array([2, 0, (CALLS + 1) & 0xFFFFFFFF, 1], np.uint32), np.array([5, 1], np.uint32))
    assert np.array_equal(e[2, :4], draws.normals(raw))
    assert not np.array_equal(eps_ref(SEED, CALLS + 1, 3), eps_ref(SEED, (CALLS + 1) & 0xFFFFFFFF, 3))
    assert not np.array_equal(eps_ref(SEED, CALLS + 1, 3), eps_ref(SEED & 0xFFFFFFFF, CALLS + 1, 3))


def test_fused_policy_rejects_layernorms_it_cannot_run():
    """The kernel applies one eps to all three LayerNorms and reads gamma / beta of each: anything else is refused."""
    import torch
    from hlynr_intercept_b200.policy import FusedActorCritic

    net = _net(device="cpu")
    FusedActorCritic._modules(types.SimpleNamespace(net=net))
    _layers(net)[1][1].eps = 1e-3
    with pytest.raises(NotImplementedError, match="eps"):
        FusedActorCritic._modules(types.SimpleNamespace(net=net))
    net = _net(device="cpu")
    net.network[4] = torch.nn.LayerNorm(512, elementwise_affine=False)
    with pytest.raises(NotImplementedError, match="affine"):
        FusedActorCritic._modules(types.SimpleNamespace(net=net))


# ---- LayerNorm edges ----------------------------------------------------------------------------------------------------------

def _offset_net(layer, ratio, mode, obs):
    """A net whose hidden layer `layer` has pre-activations with a common mean of `ratio` times their spread.
    bias:   b_l += ratio * sigma_l (the accumulators stay small, the bias is large);
    weight: every row of W_l gets the same weight alpha on one input that is positive in every row (obs channel 7 in [5, 10];
            for a hidden layer, feature 0 of the layer before, given gamma 0.5 and beta 3), so the common mean comes out of
            the GEMM accumulators and differs from row to row."""
    import torch

    net = _net(seed=10 + layer)
    lins, lns = _layers(net)
    with torch.no_grad():
        if mode == "bias":
            lins[layer].bias.add_(ratio * _sigma(net, obs, layer))
        else:
            if layer > 0:
                lns[layer - 1].weight[0] = 0.5; lns[layer - 1].bias[0] = 3.0
            j = 7 if layer == 0 else 0
            lins[layer].weight[:, j] = 0.0
            sigma = _sigma(net, obs, layer)
            xj = float(obs[:, 7].mean()) if layer == 0 else 3.0
            lins[layer].weight[:, j] = ratio * sigma / xj
    return net


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
@pytest.mark.parametrize("mode", ["bias", "weight"])
@pytest.mark.parametrize("ratio", [100, 300, 1000])
@pytest.mark.parametrize("layer", [0, 1, 2])
def test_layernorm_with_a_large_common_mean(layer, ratio, mode, cluster):
    """LayerNorm is shift invariant; its statistics must be too (E[x^2] - mean^2 in fp32 is not)."""
    obs = _obs(3000, seed=layer)
    net = _offset_net(layer, ratio, mode, obs)
    _check(_fused(net, cluster), net, obs, mean_tol=MEAN_TOL * (1 + ratio / 20) if mode == "weight" else MEAN_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
@pytest.mark.parametrize("case", ["layer0", "layer1", "layer2", "all_eps1e-3"])
def test_layernorm_variance_near_eps(case, cluster):
    """Pre-activation variance about eps, so that eps changes the normalised values by about 30 %."""
    import torch

    obs = _obs(2000, seed=4)
    net = _net(seed=4)
    lins, lns = _layers(net)
    layers = [0, 1, 2] if case.startswith("all") else [int(case[-1])]
    eps = 1e-3 if case.startswith("all") else 1e-5
    with torch.no_grad():
        for ln in lns:
            ln.eps = eps
        for l in layers:
            s = math.sqrt(eps) / _sigma(net, obs, l)
            lins[l].weight.mul_(s); lins[l].bias.mul_(s)
    _check(_fused(net, cluster), net, obs)


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
@pytest.mark.parametrize("layer", [0, 1, 2])
def test_layernorm_of_a_constant_row(layer, cluster):
    """W_l = 0 and a constant bias: zero variance, the layer's output is relu(beta) for every row, so every output row is the
    same, bit for bit."""
    import torch

    obs = _obs(1000, seed=5)
    net = _net(seed=5)
    lins, _ = _layers(net)
    with torch.no_grad():
        lins[layer].weight.zero_(); lins[layer].bias.fill_(0.3)
    m, v = _check(_fused(net, cluster), net, obs)
    assert torch.equal(m, m[:1].expand_as(m)) and torch.equal(v, v[:1].expand_as(v))


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
def test_dead_features_give_the_head_biases(cluster):
    """beta_3 strongly negative: H3 = 0 in every row, so mean == action bias and value == value bias, bit for bit."""
    import torch

    obs = _obs(700, seed=6)
    net = _net(seed=6)
    _, lns = _layers(net)
    with torch.no_grad():
        lns[2].weight.fill_(0.1); lns[2].bias.fill_(-10.0)   # |normalised| <= sqrt(255): gamma x + beta < 0 always
    m, v = _check(_fused(net, cluster), net, obs)
    assert torch.equal(m, net.action_net.bias.detach().expand_as(m))
    assert torch.equal(v, net.value_net.bias.detach().expand_as(v))


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
def test_input_extremes(cluster):
    """Rows at the VecNormalize clip +-10, rows of zeros (layer 1 sees its bias only), a normal tail; and a single clipped row."""
    import torch

    g = torch.Generator(device="cuda"); g.manual_seed(7)
    clip = torch.where(torch.rand(200, 104, device="cuda", generator=g) < 0.5, -10.0, 10.0)
    clip[:20] = 10.0; clip[20:40] = -10.0
    obs = torch.cat([clip, torch.zeros(150, 104, device="cuda"), _obs(173, seed=7)]).contiguous()
    net = _net(seed=7)
    fused = _fused(net, cluster)
    _check(fused, net, obs)
    _check(fused, net, clip[:1].contiguous())


# ---- sampling -----------------------------------------------------------------------------------------------------------------

def _ulps(x):
    return np.spacing(np.abs(np.asarray(x, dtype=np.float32))).astype(np.float64)


def noise_errors(a, lp, m, log_std, eps):
    """(worst action error, worst log pi error) in units of ULP_TOL float32 ulp of the stated magnitudes."""
    a, lp, m = (t.double().cpu().numpy() for t in (a, lp, m))
    ls = np.asarray(log_std, np.float64)
    e = eps.astype(np.float64)
    se = np.exp(ls) * e
    da = np.abs(a - (m + se)) / (ULP_TOL * _ulps(np.maximum(np.abs(m), np.abs(se))))
    terms = -0.5 * e * e - ls
    want_lp = terms.sum(-1) - 3.0 * math.log(2 * math.pi)
    dl = np.abs(lp - want_lp) / (ULP_TOL * _ulps(np.abs(terms).sum(-1) + 3.0 * math.log(2 * math.pi)))
    return float(da.max()), float(dl.max())


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
@pytest.mark.parametrize("n", [129, 37965, 131072 + 77])
def test_noise_is_pinned_per_row(n, cluster):
    """eps of every row is Philox at (row, call counter) keyed by the seed: a wrong row for the later tiles of a persistent CTA
    or of another cluster rank, a dropped high word of the counter or the seed, or swapped words fail here."""
    import torch

    net = _net(seed=8)
    fused = _fused(net, cluster)
    obs = _obs(n, seed=8)
    clipped = torch.empty(n, 6, device="cuda")
    fused.calls = CALLS
    a, _, lp, m = (t.clone() for t in fused.forward(obs, want=("actions", "values", "logp", "mean"), out=dict(clipped=clipped)))
    torch.cuda.synchronize()
    assert fused.calls == CALLS + 1
    da, dl = noise_errors(a, lp, m, LOG_STD, eps_ref(SEED, CALLS + 1, n))
    assert da <= 1.0, f"actions differ from mean + exp(log_std) eps_ref by {da * ULP_TOL:.1f} ulp"
    assert dl <= 1.0, f"log pi differs from the Gaussian formula at eps_ref by {dl * ULP_TOL:.1f} ulp"
    assert torch.equal(clipped, a.clamp(-1.0, 1.0))
    # deterministic: the action is the mean, log pi is the density at eps = 0
    ad, _, lpd, md = fused.forward(obs, deterministic=True, want=("actions", "values", "logp", "mean"), out=dict(clipped=clipped))
    torch.cuda.synchronize()
    assert torch.equal(ad, md) and torch.equal(md, m) and torch.equal(clipped, md.clamp(-1.0, 1.0))
    want = -sum(LOG_STD) - 3.0 * math.log(2 * math.pi)
    assert float((lpd.double() - want).abs().max()) <= 4 * float(_ulps(want))
    fused.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
def test_output_subsets_are_the_same_bits(cluster):
    """Each output alone, and all of them written into rows of rollout buffers from a row of an observation buffer (as the
    collector calls it), give the bits of the full call at the same counter."""
    import torch

    n, T = 1111, 3
    net = _net(seed=9)
    fused = _fused(net, cluster)
    obs_buf = torch.zeros(T + 1, n, 104, device="cuda")
    obs_buf[2] = _obs(n, seed=9)
    obs = obs_buf[2].clone()

    def call(**kw):
        fused.calls = CALLS
        r = fused.forward(obs, **kw)
        torch.cuda.synchronize()
        return [None if t is None else t.clone() for t in r]

    clipped = torch.empty(n, 6, device="cuda")
    a, v, lp, m = call(want=("actions", "values", "logp", "mean"), out=dict(clipped=clipped))
    clipped = clipped.clone()
    assert torch.equal(call(want=("actions",))[0], a)
    assert torch.equal(call(want=("logp",))[2], lp)
    assert torch.equal(call(want=("values",))[1], v)
    assert torch.equal(call(want=("mean",))[3], m)
    only = torch.empty(n, 6, device="cuda")
    call(want=(), out=dict(clipped=only))
    assert torch.equal(only, clipped)
    bufs = dict(actions=torch.zeros(T, n, 6, device="cuda"), values=torch.zeros(T, n, device="cuda"),
                logp=torch.zeros(T, n, device="cuda"), mean=torch.zeros(T, n, 6, device="cuda"),
                clipped=torch.zeros(T, n, 6, device="cuda"))
    fused.calls = CALLS
    fused.forward(obs_buf[2], out={k: b[1] for k, b in bufs.items()})
    torch.cuda.synchronize()
    for k, want in (("actions", a), ("values", v), ("logp", lp), ("mean", m), ("clipped", clipped)):
        assert torch.equal(bufs[k][1], want), k
        assert (bufs[k][0] == 0).all() and (bufs[k][2] == 0).all(), k
    fused.close()


# ---- sizes and state ----------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
def test_production_sizes_and_handle_reuse(cluster):
    """131 072 rows (the rollout size) and 2 x 131 072 + 77: many tiles per persistent CTA, so the mbarrier parities and the
    weight-ring phases wrap many times.  Large, small, large again on one handle: the same bits, no stale grid or state."""
    import torch

    net = _net(seed=11)
    fused = _fused(net, cluster)
    for n in (131072, 2 * 131072 + 77):
        obs = _obs(n, seed=n)
        m, v = _check(fused, net, obs)
        _check(fused, net, obs[:300].contiguous())
        m2, v2 = _mean_value(fused, obs)
        assert torch.equal(m2, m) and torch.equal(v2, v)
        del obs
    fused.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", CLUSTERS)
def test_sync_weights_reads_every_parameter(cluster):
    """Change every parameter tensor, sync: the handle matches the reference and a fresh handle, bit for bit (noise included)."""
    import torch

    n = 2000
    net = _net(seed=12)
    obs = _obs(n, seed=12)
    fused = _fused(net, cluster)
    _check(fused, net, obs)
    g = torch.Generator(device="cuda"); g.manual_seed(12)
    with torch.no_grad():
        for p in net.parameters():
            p.add_(0.1 * p.abs().mean() * torch.randn(p.shape, device="cuda", generator=g) + 0.02)
    fused.sync_weights()
    fresh = _fused(net, cluster)
    _check(fused, net, obs)
    outs = []
    for h in (fused, fresh):
        h.calls = CALLS
        outs.append([t.clone() for t in h.forward(obs, want=("actions", "values", "logp", "mean"))])
        torch.cuda.synchronize()
    for x, y in zip(*outs):
        assert torch.equal(x, y)
    da, dl = noise_errors(outs[0][0], outs[0][2], outs[0][3], net.log_std.detach().cpu().numpy(), eps_ref(SEED, CALLS + 1, n))
    assert da <= 1.0 and dl <= 1.0
    fused.close(); fresh.close()
