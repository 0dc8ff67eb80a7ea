"""The oracle port (oracle/crossmodal_port.py) against the fixture produced by the REFERENCE's
own crossmodal code (oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest

from oracle import crossmodal_port
from oracle.golden_cases import run_all

GROUPS = ["dyn/", "head/", "fuse/", "vsensor/", "kf/", "pf_rng/"]


def _resolve(name):
    return getattr(crossmodal_port, name)


@pytest.mark.parametrize("group", GROUPS)
def test_port_matches_reference_fixture(golden, group):
    got = run_all(_resolve, device="cpu", only=[group])
    expected_keys = [k for k in golden if k.startswith(group)]
    assert expected_keys, group
    assert sorted(got) == sorted(expected_keys)
    for key in expected_keys:
        # same torch ops in the same order on the same CPU build: bit-identical is expected,
        # the tolerance only absorbs thread-count dependent GEMM blocking.
        np.testing.assert_allclose(got[key], golden[key], rtol=2e-6, atol=2e-6, err_msg=key)


def test_fixture_is_finite_and_nontrivial(golden):
    assert len(golden) >= 60
    for key, value in golden.items():
        if key.endswith("Seq5/log_weights"):  # quirk Q3: -inf image weight on blacked-out frames
            assert np.isneginf(value[:, 0]).any() and not np.isnan(value).any()
            continue
        assert np.isfinite(value).all(), key
        if not key.endswith("/tril"):
            assert np.abs(value).max() > 0, key


def test_reference_still_agrees_when_mounted(golden):
    """Where MMF_REFERENCE_DIR names a checkout of the reference, re-run the reference itself in a
    subprocess and compare with the committed fixture; skipped without one."""
    import os
    import subprocess
    import sys

    from oracle.make_golden import reference_available

    if not reference_available():
        pytest.skip("MMF_REFERENCE_DIR does not name a checkout of the reference")
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import numpy as np\n"
        "from oracle.make_golden import reference_resolver\n"
        "from oracle.golden_cases import run_all\n"
        "got = run_all(reference_resolver(), only=['dyn/', 'fuse/PushCrossmodalParticleFilter', 'kf/DoorCrossmodalKalmanFilter/'])\n"
        "ref = np.load(%r)\n"
        "for k, v in got.items():\n"
        "    np.testing.assert_allclose(v, ref[k], rtol=2e-6, atol=2e-6, err_msg=k)\n"
        "print('OK', len(got))\n"
    ) % (repo, os.path.join(repo, "tests", "golden", "reference_modules.npz"))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "OK" in res.stdout, res.stderr[-2000:]
