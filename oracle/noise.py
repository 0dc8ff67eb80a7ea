"""ORACLE (test infrastructure): explicit noise sources for the restated ParticleFilter.

Recipes from SURVEY.md Appendix A.6 (each checked bit-exact on CPU against the
``torch.distributions`` path in tests/test_oracle_rng.py):
  * ``MultivariateNormal(mean, cov).sample((M,))``  == mean + chol(cov) @ randn(M, N, sd)
  * ``MultivariateNormal(loc, scale_tril=L).rsample()`` == loc + L @ randn(N*M, sd)
  * ``Categorical(logits).sample((S,)).T`` == inverse CDF of float64 ``torch.rand(N*S)``
    (trajectory-major), on a sequential-fp32 CDF.
"""
import torch

from oracle import install_shims

install_shims()
from torchfilter.filters import multinomial_inverse_cdf  # noqa: E402


class TorchRNGNoise:
    """Draws from torch's global CPU generator in exactly the order torch.distributions would."""

    def init_eps(self, M, N, sd, like):
        return torch.randn(M, N, sd, dtype=like.dtype)

    def process_eps(self, rows, sd, like):
        return torch.randn(rows, sd, dtype=like.dtype)

    def resample_uniforms(self, N, S):
        return torch.rand(N * S, dtype=torch.float64).reshape(N, S)

    def resample_indices(self, probs, S, logits=None):
        return multinomial_inverse_cdf(probs, self.resample_uniforms(probs.shape[0], S))

    def randperm(self, M):
        return torch.randperm(M)


class RecordedNoise:
    """Replays pre-drawn tensors (lists consumed front to back); records what it handed out.

    ``mode``: ``"multinomial"`` (u is (N, S) float64) or ``"systematic"`` (u0 is (N,) float64;
    positions (u0 + j) / S, the north-star low-variance variant that upstream does not have).
    """

    def __init__(self, *, init_eps=None, process_eps=(), uniforms=(), mode="multinomial", arithmetic="torch"):
        self._init = init_eps
        self._eps = list(process_eps)
        self._u = list(uniforms)
        self.mode = mode  # multinomial | multinomial_fast | systematic | systematic_fast
        # "torch": torch's softmax + sequential fp32 CDF (what torch.multinomial does on CPU);
        # "pinned": the fully specified arithmetic of oracle/pinned/mmf_pinned.c (required for *_fast)
        self.arithmetic = arithmetic
        self.probs_seen = []
        self.indices = []

    def init_eps(self, M, N, sd, like):
        assert self._init.shape == (M, N, sd)
        return self._init.to(device=like.device, dtype=like.dtype)

    def process_eps(self, rows, sd, like):
        eps = self._eps.pop(0)
        assert eps.shape == (rows, sd)
        return eps.to(device=like.device, dtype=like.dtype)

    def resample_indices(self, probs, S, logits=None):
        u = self._u.pop(0)
        self.probs_seen.append(probs.detach().clone())
        if self.arithmetic == "pinned":
            from oracle import pinned

            idx = pinned.resample(logits.detach().cpu().numpy(), u.cpu().numpy(), self.mode, num_samples=S)
            idx = torch.from_numpy(idx)
            self.indices.append(idx)
            return idx
        assert self.mode in ("multinomial", "systematic"), "the blocked summation order only exists pinned"
        if self.mode == "systematic":
            assert u.shape == (probs.shape[0],)
            j = torch.arange(S, dtype=torch.float64)
            u = (u.double()[:, None] + j[None, :]) / float(S)
        assert u.shape == (probs.shape[0], S)
        idx = multinomial_inverse_cdf(probs, u)
        self.indices.append(idx)
        return idx

    def randperm(self, M):
        return torch.randperm(M)
