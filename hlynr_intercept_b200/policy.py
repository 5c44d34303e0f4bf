"""The reference's actor-critic network and its fused sm_100a forward (include/hlynr_policy.h).

`ReferenceActorCritic` is a plain torch module with the architecture the reference trains (rl_system/scripts/
train_flat_ppo.py:37-85 CustomMLP as SB3 features extractor, :419-429 net_arch=[]: action_net / value_net directly on the 256
features, state-independent log_std): it is the fp32 definition the fused kernel is checked against and the container of the
weights.  `FusedActorCritic` runs the same forward as ONE hand-written kernel (tcgen05 GEMMs with bf16 operands and fp32
accumulation in TMEM, TMA-fed weight tiles, bias + LayerNorm + ReLU as the epilogue between layers, both heads, Gaussian
sampling and log-probability) on device tensors, for `DeviceRolloutCollector`.  Its input width is that of the first Linear,
1-256: 104 for frame_stack 4 of the 26-D observation, 68 for frame_stack 4 of the 17-D one, and so on.
"""
import ctypes as C
import math

from . import _lib, abi


def _torch():
    import torch

    return torch


class ReferenceActorCritic:
    """Factory: torch.nn.Module with forward(obs) -> (actions, values, log_probs), value(obs), mean(obs)."""

    def __new__(cls, obs_dim=104, act_dim=6, net_arch=(512, 512, 256), log_std_init=0.0, device="cuda"):
        torch = _torch()
        nn = torch.nn

        class _Net(nn.Module):
            def __init__(self):
                super().__init__()
                layers, d = [], obs_dim
                for h in net_arch:   # CustomMLP: Linear -> LayerNorm -> ReLU, orthogonal init with gain sqrt(2), zero bias
                    lin = nn.Linear(d, h)
                    nn.init.orthogonal_(lin.weight, gain=math.sqrt(2))
                    nn.init.constant_(lin.bias, 0.0)
                    layers += [lin, nn.LayerNorm(h), nn.ReLU()]
                    d = h
                self.network = nn.Sequential(*layers)
                self.action_net = nn.Linear(d, act_dim)     # SB3 ActorCriticPolicy: ortho gain 0.01 / 1.0
                self.value_net = nn.Linear(d, 1)
                nn.init.orthogonal_(self.action_net.weight, gain=0.01); nn.init.constant_(self.action_net.bias, 0.0)
                nn.init.orthogonal_(self.value_net.weight, gain=1.0); nn.init.constant_(self.value_net.bias, 0.0)
                self.log_std = nn.Parameter(torch.full((act_dim,), float(log_std_init)))

            def features(self, obs):
                return self.network(obs)

            def mean(self, obs):
                return self.action_net(self.features(obs))

            def value(self, obs):
                return self.value_net(self.features(obs)).squeeze(-1)

            def forward(self, obs):
                f = self.features(obs)
                mean, value = self.action_net(f), self.value_net(f).squeeze(-1)
                eps = torch.randn_like(mean)
                actions = mean + self.log_std.exp() * eps
                logp = (-0.5 * eps ** 2 - self.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
                return actions, value, logp

        return _Net().to(device)


def bf16_emulated_forward(net, obs):
    """The network evaluated the way the fused kernel rounds: weights, input and hidden activations rounded to bf16, fp32
    accumulation, fp32 bias / LayerNorm / ReLU.  Returns (mean, value); used by the tests for a tight comparison."""
    torch = _torch()
    r = lambda t: t.to(torch.bfloat16).to(torch.float32)  # noqa: E731
    x = r(obs.float())
    mods = list(net.network)
    for k in range(0, len(mods), 3):
        lin, ln = mods[k], mods[k + 1]
        y = x.double() @ r(lin.weight).double().t() + lin.bias.double()
        y = torch.nn.functional.layer_norm(y.float(), (lin.out_features,), ln.weight, ln.bias, ln.eps)
        x = r(torch.relu(y))
    mean = (x.double() @ r(net.action_net.weight).double().t() + net.action_net.bias.double()).float()
    value = (x.double() @ r(net.value_net.weight).double().t() + net.value_net.bias.double()).float().squeeze(-1)
    return mean, value


class FusedActorCritic:
    """hlynr_policy_* behind the policy interface DeviceRolloutCollector uses: __call__(obs) -> (actions, values, log_probs),
    value(obs), value_rows(obs, n_rows_dev).  `net` holds the weights (a ReferenceActorCritic, or any object with the same
    attribute names, e.g. an SB3 policy: .features_extractor.network / .action_net / .value_net / .log_std).  The input width
    `in_dim` is read from the first Linear."""

    fused = True
    MAX_IN = 256   # HLYNR_POLICY_MAX_IN: four 64-wide K blocks of the first GEMM

    def __init__(self, net, device=0, seed=0):
        torch = _torch()
        self.L = _lib.load()
        self.net = net
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        self.in_dim = int(self._modules()[0][0].weight.shape[1])
        h = C.c_void_p()
        _lib.check(self.L.hlynr_policy_create_dim(self.device_index, self.in_dim, C.byref(h)))
        self.h = h
        self.seed = int(seed)
        self._buf = {}
        self.sync_weights()

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    @property
    def calls(self):
        """The noise counter of the last forward: the next one draws at calls + 1.  It lives on the device and every forward
        advances it there, so a forward captured in a CUDA graph draws fresh noise on every replay.  Reading it synchronises the
        current stream; setting it is ordered on that stream."""
        v = C.c_uint64()
        _lib.check(self.L.hlynr_policy_get_counter(self.h, C.byref(v), self._stream()))
        return v.value

    @calls.setter
    def calls(self, value):
        _lib.check(self.L.hlynr_policy_set_counter(self.h, int(value), self._stream()))

    def state_dict(self):
        """The noise counter and seed, what a resumed run needs to draw the same noise; the weights and the optimiser stay with
        torch's own state_dict.  Synchronises the current stream."""
        return {"calls": self.calls, "seed": self.seed}

    def load_state_dict(self, state):
        self.calls = int(state["calls"])
        self.seed = int(state["seed"])

    def _modules(self):
        net = self.net
        seq = net.network if hasattr(net, "network") else net.features_extractor.network
        mods = list(seq)
        lins = [m for m in mods if m.__class__.__name__ == "Linear"]
        lns = [m for m in mods if m.__class__.__name__ == "LayerNorm"]
        shapes = [tuple(m.weight.shape) for m in lins]
        in_dim = shapes[0][1] if shapes else 0
        if (shapes != [(512, in_dim), (512, 512), (256, 512)] or not 1 <= in_dim <= FusedActorCritic.MAX_IN or len(lns) != 3
                or getattr(self, "in_dim", in_dim) != in_dim):
            raise NotImplementedError("the fused forward is built for the reference's default architecture: in_dim -> [512, 512, 256] "
                                      "with LayerNorm + ReLU (train_flat_ppo.py:410), in_dim 1-256 and fixed for the handle; "
                                      "other shapes run through torch")
        if tuple(net.action_net.weight.shape) != (6, 256) or tuple(net.value_net.weight.shape) != (1, 256):
            raise NotImplementedError("action_net must be Linear(256, 6) and value_net Linear(256, 1)")
        if any(m.weight is None or m.bias is None for m in lns):
            raise NotImplementedError("the fused forward needs LayerNorms with affine parameters (elementwise_affine=True, bias=True)")
        if len({float(m.eps) for m in lns}) != 1:   # the kernel applies one eps to all three LayerNorms
            raise NotImplementedError(f"the fused forward needs one LayerNorm eps for all layers, got {[m.eps for m in lns]}")
        return lins, lns

    def sync_weights(self):
        """Copies the module's current fp32 parameters into the kernel's bf16 operand buffers (call after an optimiser step)."""
        torch = _torch()
        lins, lns = self._modules()
        net = self.net
        ts = []

        def p(t):
            t = t.detach().to(device=self.device, dtype=torch.float32).contiguous()
            ts.append(t)   # keep alive until the pack kernels have been queued on this stream
            return C.c_void_p(t.data_ptr())

        w = abi.HlynrPolicyWeights(
            w1=p(lins[0].weight), b1=p(lins[0].bias), ln1_g=p(lns[0].weight), ln1_b=p(lns[0].bias),
            w2=p(lins[1].weight), b2=p(lins[1].bias), ln2_g=p(lns[1].weight), ln2_b=p(lns[1].bias),
            w3=p(lins[2].weight), b3=p(lins[2].bias), ln3_g=p(lns[2].weight), ln3_b=p(lns[2].bias),
            wa=p(net.action_net.weight), ba=p(net.action_net.bias), wv=p(net.value_net.weight), bv=p(net.value_net.bias),
            log_std=p(net.log_std), ln_eps=float(lns[0].eps))
        _lib.check(self.L.hlynr_policy_set_weights(self.h, C.byref(w), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()   # the temporaries above may be freed now

    def _out(self, name, shape):
        torch = _torch()
        t = self._buf.get(name)
        if t is None or tuple(t.shape) != tuple(shape):
            t = self._buf[name] = torch.empty(shape, dtype=torch.float32, device=self.device)
        return t

    def forward(self, obs, deterministic=False, n_rows_dev=None, want=("actions", "values", "logp"), out=None):
        """obs: float32 cuda tensor [n, in_dim] (contiguous).  Returns (actions [n,6], values [n], log_probs [n]); the tensors are
        reused by the next call.  n_rows_dev: optional int32 cuda tensor [1] limiting the rows that are computed.
        Every call, of any kind, advances `calls` by one on the device and samples at the new value.
        out: optional dict of caller tensors the kernel writes into directly ('actions', 'values', 'logp', 'mean', and
        'clipped' = the action clipped to [-1, 1]^6 as SB3 passes it to env.step), e.g. rows of a rollout buffer."""
        torch = _torch()
        if obs.dim() == 0 or obs.shape[-1] != self.in_dim:
            raise ValueError(f"obs rows must be {self.in_dim} wide (the policy's input width), got shape {tuple(obs.shape)}")
        if not (obs.is_cuda and obs.dtype == torch.float32 and obs.dim() == 2 and obs.is_contiguous()):
            obs = obs.to(device=self.device, dtype=torch.float32).reshape(-1, self.in_dim).contiguous()
        n = obs.shape[0]
        out = out or {}

        def buf(name, shape):
            t = out.get(name)
            if t is not None:
                if not (t.is_cuda and t.dtype == torch.float32 and tuple(t.shape) == tuple(shape) and t.is_contiguous()):
                    raise ValueError(f"out['{name}'] must be a contiguous cuda float32 tensor of shape {tuple(shape)}")
                return t
            return self._out(name, shape) if name in want else None

        a, v, lp, m = buf("actions", (n, 6)), buf("values", (n,)), buf("logp", (n,)), buf("mean", (n, 6))
        cl = buf("clipped", (n, 6))
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
        _lib.check(self.L.hlynr_policy_forward_dev(self.h, ptr(obs), n, ptr(n_rows_dev), ptr(a), ptr(v), ptr(lp), ptr(m), ptr(cl),
                                                   self.seed, int(bool(deterministic)), self._stream()))
        return (a, v, lp) if m is None else (a, v, lp, m)

    __call__ = forward

    def value(self, obs):
        return self.forward(obs, deterministic=True, want=("values",))[1]

    def value_rows(self, obs, n_rows_dev):
        """Values of rows [0, *n_rows_dev) only (the value net on 'the finished episodes of this step', no host round trip);
        rows beyond the count keep whatever the buffer held."""
        return self.forward(obs, deterministic=True, n_rows_dev=n_rows_dev, want=("values",))[1]

    def mean_and_value(self, obs):
        _, v, _, m = self.forward(obs, deterministic=True, want=("values", "mean"))
        return m, v

    def set_option(self, name, value):
        _lib.check(self.L.hlynr_policy_set_option(self.h, name.encode(), int(value)))

    def parameters(self):
        return self.net.parameters()

    def launch_count(self):
        v = C.c_int64()
        _lib.check(self.L.hlynr_policy_launch_count(self.h, C.byref(v)))
        return v.value

    def close(self):
        if getattr(self, "h", None):
            self.L.hlynr_policy_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
