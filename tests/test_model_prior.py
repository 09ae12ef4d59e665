"""CPU checks of the model prior on the host side: AbsNormalModel(prior=...) evaluates and lowers the distribution it is
given, and a foreign model is lowered with its `prior` attribute only when its own prior_log_prob agrees with it."""
import math

import numpy as np
import pytest
import torch

import glabc_b200 as g
from glabc_b200.models import fused_model, lower_model
from helpers import abi


def priors():
    return dict(uniform=g.Uniform(2, torch.tensor([1.4, -1.0]), torch.tensor([3.0, 2.0])),
                gamma=g.Gamma(torch.tensor([2.0, 3.0]), torch.tensor([10.0, 4.0])),
                mix=g.GaussianMixture(2, 2, loc=[[0.5, 0.5], [2.5, 2.5]], scale=[[0.3, 0.3]] * 2, weights=[3, 1]),
                diag=g.DiagGaussian(2, torch.tensor([0.5, -0.5]), torch.tensor([0.1, -0.2])))


def points():
    th = torch.randn(256, 2, generator=torch.Generator().manual_seed(3)) * 2.0
    return torch.cat([th, th.abs() + 0.01, torch.tensor([[1.4, -1.0], [3.0, 2.0], [0.0, 0.0], [-1e-3, 1.0]])])


@pytest.mark.parametrize("name", ["uniform", "gamma", "mix", "diag"])
def test_prior_log_prob_is_the_distributions(name):
    prior = priors()[name]
    model = g.AbsNormalModel(0.05, prior=prior, link="identity")
    z = points()
    want = prior.log_prob(z)
    got = model.prior_log_prob(z)
    assert got.dtype == want.dtype and torch.equal(torch.isneginf(got), torch.isneginf(want))
    assert torch.equal(got, want)
    if name in ("uniform", "gamma"):
        assert torch.isneginf(got).any() and torch.isfinite(got).any()


@pytest.mark.parametrize("name", ["uniform", "gamma", "mix", "diag"])
def test_lower_prior_returns_the_distributions_pod(name):
    prior = priors()[name]
    model = g.AbsNormalModel(0.05, prior=prior)
    got, want = model.lower_prior(), prior.lower()
    assert isinstance(got, abi.DistPOD) and bytes(got) == bytes(want)
    assert got.kind == {"uniform": abi.DIST_UNIFORM, "gamma": abi.DIST_GAMMA, "mix": abi.DIST_GAUSSIAN_MIXTURE,
                        "diag": abi.DIST_DIAG_GAUSSIAN}[name] and got.dim == 2
    assert bytes(model.lower()) == bytes(g.AbsNormalModel(0.05).lower())   # lower() is unchanged
    assert g.AbsNormalModel(0.05).lower_prior() is None


def test_prior_must_be_a_distribution_of_theta_dim():
    with pytest.raises(ValueError, match="theta_dim"):
        g.AbsNormalModel(0.05, prior=g.Uniform(3, torch.zeros(3), torch.ones(3)))
    with pytest.raises(TypeError):
        g.AbsNormalModel(0.05, prior=lambda z: z)


class ForeignModel:
    """a reference-style plugin object (examples/Mixture.py): identity link, noise N(0, 0.05), `prior` attribute"""

    def __init__(self, prior, prior_log_prob=None):
        self.epsilon, self.theta_dim, self.y_dim = 0.05, 2, 2
        self.y_obs = torch.tensor([[1.5, 1.5]])
        self.prior = prior
        self._plp = prior_log_prob

    def generate_samples(self, theta, num_samples=1):
        return theta + math.sqrt(0.05) * torch.randn(theta.shape[0], 2)

    def prior_log_prob(self, z):
        return self._plp(z) if self._plp is not None else self.prior.log_prob(z.view(-1, 2))

    def discrepancy(self, y):
        return torch.sqrt(torch.sum((y.view(-1, 2) - self.y_obs) ** 2, dim=1))

    def calculate_log_kernel(self, y):
        eps = torch.tensor([0.05])
        return g.DiagGaussian(1, torch.zeros(1), torch.log(eps)).log_prob(self.discrepancy(y).view(-1, 1))


class Uniform:
    """stands in for the reference's distribution.Uniform: recognised by its class name and attributes"""

    def __init__(self, low, high):
        self.shape, self.low, self.high = (2,), torch.tensor(low), torch.tensor(high)

    def log_prob(self, z):
        out = -torch.log(torch.prod(self.high - self.low)) * torch.ones(z.shape[0])
        out[((z < self.low) | (z > self.high)).any(dim=1)] = -np.inf
        return out


@pytest.mark.parametrize("name", ["uniform", "gamma", "mix"])
def test_foreign_model_with_a_prior_attribute_is_lowered(name):
    prior = priors()[name]
    fm = fused_model(ForeignModel(prior))
    assert fm.link == "identity" and bytes(fm.lower_prior()) == bytes(prior.lower())
    assert bytes(lower_model(ForeignModel(prior))) == bytes(fm.lower())


def test_foreign_model_with_a_reference_class_prior_is_lowered():
    ref = Uniform([1.4, -1.0], [3.0, 2.0])
    got = fused_model(ForeignModel(ref)).lower_prior()
    assert bytes(got) == bytes(g.Uniform(2, torch.tensor([1.4, -1.0]), torch.tensor([3.0, 2.0])).lower())


def test_foreign_model_whose_prior_log_prob_disagrees_is_refused():
    box = priors()["uniform"]
    wider = g.Uniform(2, torch.tensor([0.0, -2.0]), torch.tensor([3.0, 2.0]))   # another box: other support, other value
    with pytest.raises(NotImplementedError, match="diagonal Gaussian"):
        fused_model(ForeignModel(box, prior_log_prob=wider.log_prob))
    shifted = lambda z: box.log_prob(z.view(-1, 2)) + 0.5   # noqa: E731  same support, other value
    with pytest.raises(NotImplementedError, match="diagonal Gaussian"):
        fused_model(ForeignModel(box, prior_log_prob=shifted))
    with pytest.raises(NotImplementedError, match="diagonal Gaussian"):   # an attribute that does not lower: the Gaussian probe
        fused_model(ForeignModel(object(), prior_log_prob=box.log_prob))
