"""Pins the CPU oracle (oracle/dflex_oracle.c, a dense restatement of the reference algorithm):
* fp32 forward  == golden trajectories recorded from the unmodified reference, BIT FOR BIT;
* fp64 central finite differences of the oracle == the reference's reverse-mode gradients
  (an adjoint-free confirmation of what the hand-derived CUDA adjoint must reproduce);
* fp32 forward  == the reference's own compiled kernels on fresh random states, bit for bit (their results recorded
  in tests/golden/ref_kernels.npz by oracle/make_ref_kernel_golden.py)."""
import os
import sys

import numpy as np
import pytest

from conftest import ENVS
from emu_util import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from oracle import Oracle  # noqa: E402


def rel(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    return np.abs(a - b).max() / (np.abs(b).max() + 1e-30)


def _setup(name):
    d, model = load_golden(name)
    cfg = dict(N=int(d["meta/num_envs"]), S=int(d["meta/substeps"]), mm=int(d["meta/mass_matrix_freq"]), dt=float(d["meta/dt"]))
    return d, model, Oracle.from_model(model, cfg["N"]), cfg


@pytest.mark.parametrize("name", ENVS)
def test_oracle_forward_is_bit_exact_vs_reference(name):
    d, model, o, c = _setup(name)
    Q, D = o.desc.Q, o.desc.D
    for k in range(int(d["meta/num_cases"])):
        p = "case%d/" % k
        musc = d[p + "musc"] if (p + "musc") in d.files else None
        q, qd, traj = o.forward(d[p + "q0"], d[p + "qd0"], d[p + "act"], musc, c["S"], c["mm"], c["dt"], want_traj=True)
        assert np.array_equal(q.astype(np.float32), d[p + "traj_q"][-1]), (name, k)
        assert np.array_equal(qd.astype(np.float32), d[p + "traj_qd"][-1]), (name, k)
        # every substep of the trajectory
        traj = traj.astype(np.float32)                       # [N, S, Q+D]
        ref_q = d[p + "traj_q"].reshape(c["S"], c["N"], Q).transpose(1, 0, 2)
        ref_qd = d[p + "traj_qd"].reshape(c["S"], c["N"], D).transpose(1, 0, 2)
        assert np.array_equal(traj[:, :, :Q], ref_q) and np.array_equal(traj[:, :, Q:], ref_qd), (name, k)


@pytest.mark.parametrize("name", ENVS)
def test_finite_difference_gradient_matches_reference_adjoint(name):
    d, model, o, c = _setup(name)
    N, Q, D, M = c["N"], o.desc.Q, o.desc.D, o.desc.M
    errs = []
    for k in range(int(d["meta/num_cases"])):
        p = "case%d/" % k
        musc = d[p + "musc"].reshape(N, M) if (p + "musc") in d.files else None
        for e in range(N):
            g = o.fd_gradient(d[p + "q0"].reshape(N, Q)[e], d[p + "qd0"].reshape(N, D)[e], d[p + "act"].reshape(N, D)[e],
                              None if musc is None else musc[e], d[p + "gq_out"].reshape(N, Q)[e], d[p + "gqd_out"].reshape(N, D)[e],
                              c["S"], c["mm"], c["dt"])
            errs.append(max(rel(g[0], d[p + "grad_q"].reshape(N, Q)[e]), rel(g[1], d[p + "grad_qd"].reshape(N, D)[e]),
                            rel(g[2], d[p + "grad_act"].reshape(N, D)[e])))
            if g[3] is not None:
                errs.append(rel(g[3], d[p + "grad_musc"].reshape(N, M)[e]))
    errs = np.array(errs)
    # the reference gradient is fp32 through an ill-conditioned solve (~1e-5..1e-4 relative), and finite
    # differences straddle a kink (contact switching on exactly at reset) in a few cases
    assert np.median(errs) < 1e-4 and (errs < 5e-3).mean() >= 0.6, (name, errs)


@pytest.mark.parametrize("name", ["AntEnv", "SNUHumanoidEnv", "CartPoleSwingUpEnv"])
def test_oracle_equals_reference_kernels_on_random_states(name):
    """Inputs and the reference kernels' results: tests/golden/ref_kernels.npz (oracle/make_ref_kernel_golden.py)."""
    d, model, o, c = _setup(name)
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_kernels.npz"))
    p = "random/%s/" % name
    musc = g[p + "musc"] if (p + "musc") in g.files else None
    assert g[p + "q0"].shape[0] == 5 and (musc is None) == (o.desc.M == 0)
    oq, oqd = o.forward(g[p + "q0"], g[p + "qd0"], g[p + "act"], musc, c["S"], c["mm"], c["dt"])
    assert np.array_equal(oq.astype(np.float32), g[p + "q"]) and np.array_equal(oqd.astype(np.float32), g[p + "qd"])
