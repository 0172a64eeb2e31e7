"""CPU checks of the fading-channel additions: the channel-state oracle against its literal restatement and against
compute_llr, and the validation of the Monte-Carlo configuration."""
import numpy as np
import pytest

from oracle import oracle
from tests import csi_oracle, vectors


@pytest.mark.parametrize("name", list(vectors.BPS))
def test_compute_llr_csi_equals_literal(name):
    rs = np.random.RandomState(vectors.BPS[name])
    n = 300
    y = rs.randn(n) + 1j * rs.randn(n)
    h = 10 ** rs.uniform(-20, 3, n) * np.exp(2j * np.pi * rs.rand(n))
    h[::17] = 0
    for nv in (0.0001, 0.05, 0.5):
        want = csi_oracle.compute_llr_csi_literal(y, h, name, nv)
        assert np.array_equal(csi_oracle.compute_llr_csi(y, h, name, nv, chunk=64), want)
    c = oracle.modulator_constellation('16QAM') if name == '16QAM' else None
    if c is not None:
        assert np.array_equal(csi_oracle.compute_llr_csi(y, h, name, 0.05, constellation=c),
                              csi_oracle.compute_llr_csi_literal(y, h, name, 0.05, constellation=c))
    assert np.all(csi_oracle.compute_llr_csi(y, h, name, 0.05).reshape(n, -1)[h == 0] == 0)


@pytest.mark.parametrize("name", list(vectors.BPS))
def test_compute_llr_csi_with_unit_gain_is_compute_llr(name):
    y = vectors.noisy_symbols(oracle.modulate(vectors.mapper_bits(name), name), name).astype(np.complex128)
    for nv in vectors.DEMAP_NOISE_VARS + [0.0001]:
        assert np.array_equal(csi_oracle.compute_llr_csi(y, np.ones(len(y)), name, nv), oracle.compute_llr(y, name, nv))
    # a common gain g scales the distances by |g|^2: the LLRs of y g are |g|^2 times those of y (before the clip)
    g = 0.3 * np.exp(0.7j)
    a = csi_oracle.compute_llr_csi(y * g, np.full(len(y), g), name, 1.0)
    b = oracle.compute_llr(y, name, 1.0 / abs(g) ** 2)
    assert np.allclose(a, b, rtol=1e-12, atol=1e-12)


def test_sweep_config_validation():
    from modulations_b200 import montecarlo as mc
    assert mc.SweepConfig().channel == 'awgn' and mc.SweepConfig().coherence == 1
    c = mc.SweepConfig(channel='rayleigh', coherence=64)
    assert (c.channel, c.coherence) == ('rayleigh', 64)
    for bad in (dict(channel='rician'), dict(channel='AWGN'), dict(coherence=0), dict(coherence=-4),
                dict(coherence=1.5), dict(channel='rayleigh', coherence=0)):
        with pytest.raises(ValueError):
            mc.SweepConfig(**bad)
