"""ABC model plugin — the duck-typed object every sampler takes (reference examples/Mixture.py:5-53,
README.md:66-104): attributes `epsilon, theta_dim, y_obs, y_dim`, methods `generate_samples`,
`prior_log_prob`, `discrepancy`, `calculate_log_kernel`, `calculate_log_kernel_dis`.

`AbsNormalModel` is the fused family the reference's `Mixture_set` belongs to:
    y | theta ~ N(link(theta) + noise_loc, diag(noise_scale^2)),  link = |.| or identity,
    prior DiagGaussian (or any `prior=` DiagGaussian / Uniform / Gamma / GaussianMixture), discrepancy = L2
    distance to y_obs, Gaussian ABC kernel of width epsilon.
Its torch methods follow the reference formulas (usable on CPU or CUDA tensors, batched); its
`lower()` gives the POD the kernels consume, `lower_prior()` the POD of a `prior=` distribution.  `lower_model()` also recognises a *reference*
`Mixture_set` instance (duck-typed probe of its deterministic methods) so existing user scripts can
pass their own model object unchanged.
"""
import hashlib
import struct

import torch

from . import _abi
from .distribution import DiagGaussian, Gamma, GaussianMixture, Uniform

PRIOR_CLASSES = (DiagGaussian, Uniform, Gamma, GaussianMixture)


class AbsNormalModel:
    """`prior`: a DiagGaussian / Uniform / Gamma / GaussianMixture of `theta_dim` that replaces the DiagGaussian of
    `prior_loc` / `prior_log_scale`.  The kernels run a non-Gaussian prior with FAST arithmetic and the native RNG
    (glabc_model_prior_set)."""

    def __init__(self, epsilon, y_obs=(1.5, 1.5), noise_var=0.05, prior_loc=None, prior_log_scale=None,
                 noise_loc=None, link="abs", device=None, prior=None):
        self.epsilon = epsilon
        self.y_obs = torch.as_tensor(y_obs, dtype=torch.float32).view(1, -1)
        self.theta_dim = self.y_obs.shape[1]
        self.y_dim = self.theta_dim
        d = self.theta_dim
        nv = torch.as_tensor(noise_var, dtype=torch.float32).reshape(-1).expand(d).clone()
        self.noise_log_scale = torch.log(nv.sqrt())             # Mixture.py:19
        self.noise_loc = torch.zeros(d) if noise_loc is None else torch.as_tensor(noise_loc, dtype=torch.float32)
        self.prior_loc = torch.zeros(d) if prior_loc is None else torch.as_tensor(prior_loc, dtype=torch.float32)
        self.prior_log_scale = torch.zeros(d) if prior_log_scale is None else torch.as_tensor(prior_log_scale, dtype=torch.float32)
        if link not in ("abs", "identity"):
            raise ValueError("link must be 'abs' or 'identity'")
        self.link = link
        if prior is not None:
            if not isinstance(prior, PRIOR_CLASSES):
                raise TypeError(f"prior must be one of {', '.join(c.__name__ for c in PRIOR_CLASSES)}")
            if prior.lower().dim != d:
                raise ValueError(f"prior dimension {prior.lower().dim} does not match theta_dim {d}")
        self.prior = prior
        if device is not None:
            self.to(device)

    def to(self, device):
        for name in ("y_obs", "noise_log_scale", "noise_loc", "prior_loc", "prior_log_scale"):
            setattr(self, name, getattr(self, name).to(device))
        return self

    # -- plugin methods (reference Mixture.py:13-53) ------------------------------------------
    def generate_samples(self, theta, num_samples=1):
        theta = theta.to(self.y_obs.device)
        mean = torch.abs(theta) if self.link == "abs" else theta
        lik = DiagGaussian(self.theta_dim, self.noise_loc, self.noise_log_scale)
        if theta.dim() == 1:
            return mean + lik.sample(num_samples)
        n = theta.shape[0]
        if n == 1:
            return mean + lik.sample(num_samples)
        if num_samples == 1:
            return mean + lik.sample(n)
        return mean.unsqueeze(1).repeat(1, num_samples, 1) + lik.sample(num_samples * n).view(n, num_samples, -1)

    def prior_log_prob(self, samples):
        samples = samples.to(self.y_obs.device).view(-1, self.theta_dim)
        if self.prior is not None:   # the distribution's parameters stay on the CPU
            return self.prior.log_prob(samples.cpu()).to(samples.device)
        return DiagGaussian(self.theta_dim, self.prior_loc, self.prior_log_scale).log_prob(samples)

    def discrepancy(self, y):
        y = y.to(self.y_obs.device).view(-1, self.y_dim)
        return torch.sqrt(torch.sum((y - self.y_obs) ** 2, dim=1))

    def calculate_log_kernel_dis(self, dis, epsilon=None):
        eps = self.epsilon if epsilon is None else epsilon
        eps_t = torch.as_tensor([float(eps)], dtype=torch.float32, device=dis.device)
        return DiagGaussian(1, torch.zeros(1, device=dis.device), torch.log(eps_t)).log_prob(dis.view(-1, 1))

    def calculate_log_kernel(self, y, epsilon=None):
        return self.calculate_log_kernel_dis(self.discrepancy(y), epsilon)

    # -- lowering -----------------------------------------------------------------------------
    def lower(self):
        d = self.theta_dim
        if d > 4:
            raise NotImplementedError("fused kernels are instantiated for theta_dim 1..4")
        pod = _abi.ModelPOD(family=_abi.MODEL_ABS_NORMAL if self.link == "abs" else _abi.MODEL_ID_NORMAL,
                            theta_dim=d, y_dim=d)
        cpu = lambda t: t.detach().float().cpu().reshape(-1)  # noqa: E731
        _abi.fill(pod.y_obs, cpu(self.y_obs).tolist())
        _abi.fill(pod.noise_loc, cpu(self.noise_loc).tolist())
        _abi.fill(pod.noise_scale, torch.exp(cpu(self.noise_log_scale)).tolist())
        _abi.fill(pod.prior_loc, cpu(self.prior_loc).tolist())
        _abi.fill(pod.prior_log_scale, cpu(self.prior_log_scale).tolist())
        _abi.fill(pod.prior_scale, torch.exp(cpu(self.prior_log_scale)).tolist())
        eps_t = torch.tensor([float(self.epsilon)], dtype=torch.float32)
        pod.eps_log_scale = float(torch.log(eps_t))            # Mixture.py:43
        pod.eps_scale = float(torch.exp(torch.log(eps_t)))     # distribution.py:178 (0.05 -> 0.049999997)
        pod.epsilon = float(self.epsilon)                      # GLMALA.py:90 squares the Python float
        return pod

    def lower_prior(self):
        """POD of the `prior=` distribution for glabc_model_prior_set, or None for the DiagGaussian `lower()` carries"""
        return None if self.prior is None else self.prior.lower()


class Mixture_set(AbsNormalModel):
    """The README / examples model (reference Mixture.py:5-11): 2-D theta, y_obs = (1.5, 1.5),
    simulator noise variance 0.05, prior N(0, I)."""

    def __init__(self, epsilon, device=None):
        super().__init__(epsilon, y_obs=(1.5, 1.5), noise_var=0.05, device=device)


class UserModel:
    """An ABC model given as CUDA C++ source (SURVEY.md 8(f) n1): the three plugin methods every sampler calls —
    `generate_samples`, `prior_log_prob`, `discrepancy` (examples/Mixture.py:13-36, README.md:66-104) — written as device
    functions, compiled at run time INTO the fused GlobalMCMC step kernel (csrc/user_model.cu):

        __device__ void  glabc_user_simulate(const float* theta, const float* noise, const float* params, float* y);
        __device__ float glabc_user_prior_log_prob(const float* theta, const float* params);
        __device__ float glabc_user_discrepancy(const float* y, const float* params);

    `noise` holds `n_noise` independent N(0,1) draws per simulator call, `params` the model's constants.  The Gaussian
    ABC kernel of width `epsilon` (Mixture.py:38-53) stays the library's.  `check()` compiles the source without a GPU.

    The plugin methods (`generate_samples`, `prior_log_prob`, `discrepancy`, `calculate_log_kernel`) run the compiled
    functions on the GPU (glabc_user_simulate / glabc_user_evaluate): inputs on any device, float32 outputs on the engine's
    device.  There is no `y_obs`: the observation lives in `params`.

    Samplers that take it: GlobalMCMC, GLMCMC, GLMALA (theta_dim <= 5), GLMCMC_NF (theta_dim 2: the flow) and
    AGLMCMC(..., pooled=True) (theta_dim <= 4: the KernelDensity kernels), the last two through the block-iSIR kernels compiled
    with the model.  Per-chain AGLMCMC (pooled=False) refuses it: its adaptation kernels are built for the fused family.

    A 2-D `params` of shape [G, n_params] makes a *batched* model: G observed datasets fitted in one run (simulation-based
    calibration, coverage studies, many subjects with one simulator).  GlobalMCMC, GLMCMC and GLMALA then take
    `chains_per_dataset=m`: the chain with global id `chain_id_base + c` belongs to dataset `(chain_id_base + c) // m` and
    its model functions read that dataset's row, so a chain-major trace [G m, rows, d] views as [G, m, rows, d].  Chain g of
    a batched run equals chain g of a run of `dataset(g // m)` (same seed, same global id), bit for bit.  The plugin methods
    of a batched model refuse to run (use `dataset(g)`), and GLMCMC_NF / pooled AGLMCMC refuse it: they train one proposal
    on all chains."""

    def __init__(self, source, theta_dim, y_dim, n_noise, epsilon, params=()):
        self.source, self.theta_dim, self.y_dim, self.n_noise = str(source), int(theta_dim), int(y_dim), int(n_noise)
        self.epsilon = float(epsilon)
        self.table = None                         # batched: float32 [G, n_params] on the CPU
        self._dev_table = {}                      # its device copies, by device
        if getattr(params, "ndim", None) == 2 or (isinstance(params, (list, tuple)) and len(params) > 0
                                                   and all(isinstance(r, (list, tuple)) for r in params)):
            table = torch.as_tensor(params, dtype=torch.float32).detach().cpu().contiguous()
            if table.shape[0] < 1:
                raise ValueError("a batched UserModel needs at least one dataset (params of shape [G, n_params], G >= 1)")
            if table.shape[1] > _abi.USER_MAX_PARAMS:
                raise ValueError(f"at most {_abi.USER_MAX_PARAMS} params")
            self.table = table
            self.params = None
            return
        self.params = [float(p) for p in params]
        if len(self.params) > _abi.USER_MAX_PARAMS:
            raise ValueError(f"at most {_abi.USER_MAX_PARAMS} params")

    @property
    def batched(self):
        return self.table is not None

    @property
    def n_datasets(self):
        """G of a batched model, 1 otherwise"""
        return self.table.shape[0] if self.batched else 1

    @property
    def n_params(self):
        return self.table.shape[1] if self.batched else len(self.params)

    def dataset(self, g):
        """the ordinary single-dataset UserModel of row g (itself for g == 0 of an unbatched model)"""
        g = int(g)
        if not 0 <= g < self.n_datasets:
            raise IndexError(f"dataset {g} of {self.n_datasets}")
        if not self.batched:
            return self
        return UserModel(self.source, self.theta_dim, self.y_dim, self.n_noise, self.epsilon, params=self.table[g].tolist())

    def _single(self, what):
        if self.batched:
            raise ValueError(f"{what} of a batched UserModel ({self.n_datasets} datasets) is ambiguous: call it on "
                             "model.dataset(g), the single-dataset model of row g")

    # -- plugin methods (reference Mixture.py:13-53), compiled -----------------------------------
    def generate_samples(self, theta, num_samples=1, *, seed=None, row_base=0):
        """Simulator draws, shaped as AbsNormalModel.generate_samples: theta [d] or [1, d] -> [m, y_dim]; [n, d] -> [n, y_dim]
        for m = 1 and [n, m, y_dim] for m > 1.  Row i * m + j (repeat j of theta row i) draws its noise from the Philox stream
        of id row_base + i * m + j at step 0 under key `seed` (default: samplers.default_seed()), so
        `generate_samples(theta0, seed=s, row_base=chain_id_base)` is the initial y a run with seed s draws for Initial_y=None."""
        self._single("generate_samples")
        from .engine import get_engine
        from .samplers import default_seed
        eng = get_engine()
        theta = torch.as_tensor(theta, dtype=torch.float32)
        if theta.dim() not in (1, 2) or theta.shape[-1] != self.theta_dim:
            raise ValueError(f"theta must be [{self.theta_dim}] or [n, {self.theta_dim}], got {tuple(theta.shape)}")
        m = int(num_samples)
        if m < 1:
            raise ValueError("num_samples must be at least 1")
        rows = theta.reshape(-1, self.theta_dim)
        n = rows.shape[0]
        seed = default_seed() if seed is None else int(seed)
        rows = rows.to(eng.device)
        y = eng.user_simulate(self, rows if m == 1 else rows.repeat_interleave(m, dim=0), seed, row_base)
        return y if n == 1 or m == 1 else y.view(n, m, self.y_dim)

    def prior_log_prob(self, samples):
        self._single("prior_log_prob")
        from .engine import get_engine
        return get_engine().user_evaluate(self, _abi.USER_PRIOR, torch.as_tensor(samples).reshape(-1, self.theta_dim))

    def discrepancy(self, y):
        self._single("discrepancy")
        from .engine import get_engine
        return get_engine().user_evaluate(self, _abi.USER_DISCREPANCY, torch.as_tensor(y).reshape(-1, self.y_dim))

    def calculate_log_kernel_dis(self, dis, epsilon=None):
        """log N(dis; 0, eps^2), the torch formula of AbsNormalModel.calculate_log_kernel_dis"""
        from .engine import get_engine
        dev = get_engine().device
        eps = self.epsilon if epsilon is None else epsilon
        eps_t = torch.as_tensor([float(eps)], dtype=torch.float32, device=dev)
        dis = torch.as_tensor(dis, dtype=torch.float32).to(dev)
        return DiagGaussian(1, torch.zeros(1, device=dev), torch.log(eps_t)).log_prob(dis.view(-1, 1))

    def calculate_log_kernel(self, y, epsilon=None):
        """the step kernels' kernel term of the model's epsilon, on the device; another epsilon goes through
        calculate_log_kernel_dis"""
        self._single("calculate_log_kernel")
        if epsilon is not None and float(epsilon) != self.epsilon:
            return self.calculate_log_kernel_dis(self.discrepancy(y), epsilon)
        from .engine import get_engine
        return get_engine().user_evaluate(self, _abi.USER_LOG_KERNEL, torch.as_tensor(y).reshape(-1, self.y_dim))

    def fingerprint(self):
        """sha256 of what a run computes with: source, dims, n_noise, params (as the float32 the kernels read) and epsilon.
        A user-model checkpoint carries it, and a resume refuses a checkpoint of another model.  A batched model's covers its
        whole table (G, n_params and every row)."""
        h = hashlib.sha256()
        h.update(struct.pack("<4i", self.theta_dim, self.y_dim, self.n_noise, self.n_params))
        if self.batched:
            h.update(struct.pack("<q", self.n_datasets))
            h.update(self.table.numpy().tobytes())
        else:
            h.update(torch.tensor(self.params, dtype=torch.float32).numpy().tobytes())
        h.update(struct.pack("<d", self.epsilon))
        h.update(self.source.encode())
        return h.hexdigest()

    def user_pod(self, device=None, chains_per_dataset=0):
        """glabc_user_model_t.  A batched model's table is copied to `device` (once; the copy lives as long as the model), or
        left NULL without a device (a compile check needs none)."""
        pod = _abi.UserModelPOD(theta_dim=self.theta_dim, y_dim=self.y_dim, n_noise=self.n_noise, n_params=self.n_params,
                                source=self.source.encode(), epsilon=self.epsilon)
        if not self.batched:
            _abi.fill(pod.params, self.params)
            return pod
        pod.n_datasets = self.n_datasets
        pod.chains_per_dataset = int(chains_per_dataset)
        if device is not None:
            key = str(torch.device(device))
            if key not in self._dev_table:
                self._dev_table[key] = self.table.to(device)
            pod.dataset_params = self._dev_table[key].data_ptr()
        return pod

    def check(self, cc=100, proposals=None):
        """compile-only validation (NVRTC, no GPU needed); raises ValueError with the compiler log.
        `proposals`: the (Local_Proposal, Global_Proposal or Importance_Proposal) pair a run will bind, to compile the
        kernels for their kinds; None in either place (GLMALA has no Local_Proposal) or for the pair means DiagGaussian.
        A batched model compiles the batched kernels."""
        import ctypes as C
        log = C.create_string_buffer(8192)
        pod = self.user_pod()
        local, far = proposals if proposals is not None else (None, None)
        kinds = [_abi.DIST_DIAG_GAUSSIAN if d is None else lower_proposal(d).kind for d in (local, far)]
        st = _abi.load().glabc_user_model_check_proposals(C.byref(pod), kinds[0], kinds[1], int(cc), log, len(log))
        if st != _abi.OK:
            raise ValueError(f"user model rejected (status {st}): {log.value.decode(errors='replace')}")
        return True


# examples/Mixture.py:13-36 written as a user model (params = {y_obs0, y_obs1, noise_sd}): the worked example of the
# run-time compiled path, and what bench.py times beside the built-in family
MIXTURE_USER_SOURCE = r"""
__device__ void glabc_user_simulate(const float* theta, const float* noise, const float* params, float* y)
{
    y[0] = fabsf(theta[0]) + params[2] * noise[0];
    y[1] = fabsf(theta[1]) + params[2] * noise[1];
}
__device__ float glabc_user_prior_log_prob(const float* theta, const float* params)
{
    return -1.8378770664093453f - 0.5f * (theta[0] * theta[0] + theta[1] * theta[1]);
}
__device__ float glabc_user_discrepancy(const float* y, const float* params)
{
    const float a = y[0] - params[0], b = y[1] - params[1];
    return sqrtf(a * a + b * b);
}
"""


def mixture_user_model(epsilon=0.05):
    return UserModel(MIXTURE_USER_SOURCE, theta_dim=2, y_dim=2, n_noise=2, epsilon=epsilon, params=[1.5, 1.5, 0.05 ** 0.5])


def _as_prior(dist):
    """one of our distribution classes for `dist`: itself, or the same distribution built from a reference
    (glabcmcmc.distribution) instance of the same class name, recognised by its attributes; None otherwise"""
    if isinstance(dist, PRIOR_CLASSES):
        return dist
    name = type(dist).__name__
    has = lambda *a: all(hasattr(dist, x) for x in a)  # noqa: E731
    if name == "DiagGaussian" and has("loc", "log_scale", "shape", "d"):
        return DiagGaussian(tuple(dist.shape), dist.loc, dist.log_scale)
    if name == "Uniform" and has("shape", "low", "high"):
        return Uniform(tuple(dist.shape), dist.low, dist.high)
    if name == "Gamma" and has("Shape", "Rate"):
        return Gamma(dist.Shape, dist.Rate)
    if name == "GaussianMixture" and has("n_modes", "dim", "loc", "log_scale", "weight_scores"):
        return GaussianMixture(int(dist.n_modes), int(dist.dim), loc=torch.as_tensor(dist.loc)[0].numpy(),
                               scale=torch.exp(torch.as_tensor(dist.log_scale)[0]).numpy(),
                               weights=torch.softmax(torch.as_tensor(dist.weight_scores), 1)[0].numpy())
    return None


def _foreign_prior(abc_set, d, th):
    """the lowerable `prior` attribute of a foreign model, if its prior_log_prob agrees with it on the probe set and on
    points outside the support (-inf matching -inf); None otherwise"""
    prior = _as_prior(getattr(abc_set, "prior", None))
    if prior is None:
        return None
    try:
        if prior.lower().dim != d:
            return None
        pts = torch.cat([th, th * 10.0, -th.abs() - 0.5])
        want = abc_set.prior_log_prob(pts).double().reshape(-1).cpu()
        got = prior.log_prob(pts).double().reshape(-1).cpu()
    except (NotImplementedError, RuntimeError, TypeError, ValueError):
        return None
    if want.shape != got.shape or not torch.equal(torch.isneginf(want), torch.isneginf(got)):
        return None
    fin = torch.isfinite(want)
    if not torch.equal(fin, torch.isfinite(got)) or not torch.allclose(got[fin], want[fin], rtol=1e-5, atol=1e-4):
        return None
    return prior


def fused_model(abc_set):
    """our model object for `abc_set`: itself when it lowers; a foreign object is accepted only if it behaves exactly
    like the AbsNormal family on a deterministic probe (so a reference `Mixture_set` instance drops in), with a
    DiagGaussian prior found by the probe or the lowerable distribution in its `prior` attribute.  Anything else
    raises — there is no interpreted fallback."""
    if hasattr(abc_set, "lower"):
        return abc_set
    for attr in ("epsilon", "theta_dim", "y_obs", "prior_log_prob", "discrepancy", "calculate_log_kernel", "generate_samples"):
        if not hasattr(abc_set, attr):
            raise NotImplementedError(f"ABC model lacks `{attr}`; cannot lower it to a fused family")
    d = int(abc_set.theta_dim)
    y_obs = torch.as_tensor(abc_set.y_obs, dtype=torch.float32).reshape(-1)
    if y_obs.numel() != d:
        raise NotImplementedError("fused family needs y_dim == theta_dim")
    # probe: recover prior loc/scale, noise scale and link from the object's own methods
    g = torch.Generator().manual_seed(1234)
    th = torch.randn(64, d, generator=g) * 2.0
    prior = _foreign_prior(abc_set, d, th)
    # otherwise the prior: fit a diagonal Gaussian through 2d+1 evaluations, then verify on the probe set
    zero = torch.zeros(1, d)
    p0 = abc_set.prior_log_prob(zero).float().reshape(-1)[0]
    loc, ls = torch.zeros(d), torch.zeros(d)
    for i in range(d if prior is None else 0):
        e = torch.zeros(1, d)
        e[0, i] = 1.0
        pp = abc_set.prior_log_prob(e).float().reshape(-1)[0]
        pm = abc_set.prior_log_prob(-e).float().reshape(-1)[0]
        inv_var = -(pp + pm - 2 * p0)          # second difference of -0.5 (z-loc)^2 / s^2
        if not torch.isfinite(inv_var) or inv_var <= 0:
            raise NotImplementedError("prior is not a diagonal Gaussian; no fused lowering")
        loc[i] = (pp - pm) / (2 * inv_var)
        ls[i] = -0.5 * torch.log(inv_var)
    loc = torch.where(loc.abs() < 1e-6, torch.zeros_like(loc), loc)
    ls = torch.where(ls.abs() < 1e-6, torch.zeros_like(ls), ls)
    # simulator: same seed, compare against |theta| + s*eps and theta + s*eps
    state = torch.get_rng_state()
    try:
        torch.manual_seed(4321)
        y = abc_set.generate_samples(th, 1).float().reshape(64, d)
        torch.manual_seed(4321)
        eps = torch.randn(64, d)
    finally:
        torch.set_rng_state(state)
    link = None
    for name, mean in (("abs", th.abs()), ("identity", th)):
        resid = y - mean
        s = (resid / eps).median(dim=0).values
        if torch.allclose(resid, s * eps, rtol=1e-4, atol=1e-5):
            link, noise_scale = name, s
            break
    if link is None:
        raise NotImplementedError("simulator is not y = link(theta) + scale*eps; no fused lowering")
    model = AbsNormalModel(abc_set.epsilon, y_obs=y_obs.tolist(), noise_var=(noise_scale ** 2).tolist(),
                           prior_loc=loc.tolist(), prior_log_scale=ls.tolist(), link=link, prior=prior)
    # verify the deterministic plugin methods agree before trusting the lowering
    ok = (torch.allclose(model.prior_log_prob(th).float(), abc_set.prior_log_prob(th).float(), rtol=1e-5, atol=1e-5)
          and torch.allclose(model.discrepancy(y), abc_set.discrepancy(y).float(), rtol=1e-5, atol=1e-6)
          and torch.allclose(model.calculate_log_kernel(y), abc_set.calculate_log_kernel(y).float(), rtol=1e-5, atol=1e-4))
    if not ok:
        raise NotImplementedError("model does not match the AbsNormal family on the probe set; no fused lowering")
    return model


def lower_model(abc_set):
    """the model POD of `abc_set` (fused_model); its prior's POD is `fused_model(abc_set).lower_prior()`"""
    return fused_model(abc_set).lower()


def lower_proposal(dist):
    if hasattr(dist, "lower"):
        return dist.lower()
    # a reference glabcmcmc.distribution.DiagGaussian: same attributes
    if all(hasattr(dist, a) for a in ("loc", "log_scale", "shape", "d")) and type(dist).__name__ == "DiagGaussian":
        return DiagGaussian(tuple(dist.shape), dist.loc, dist.log_scale).lower()
    raise NotImplementedError(f"proposal {type(dist).__name__} has no fused lowering")
