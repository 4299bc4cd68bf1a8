"""GPU parity at the sizes BASELINE.json names (C2 Humanoid 8192, C3 SNU 4096 x BPTT-128, C4 Ant 8192 per GPU), through the
C ABI, against the CPU oracles -- plus the per-phase State fields of the GPU kernels against the reference goldens and
fp64 finite differences of the adjoint for all six articulations.

Element-wise tolerance (VERDICT r1 #8): |a - b| <= rtol * |b| + atol_frac * max|b| per component, per environment; an
environment may only fail when the test shows a switching surface (contact height, joint limit) within rounding
distance for it (the reference's own branch would flip under the same perturbation).
"""
import os
import sys

import numpy as np
import pytest

from emu_util import EmuSim, load_golden
from tolerances import GRAD_RTOL, fwd_rtol

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
pytestmark = pytest.mark.gpu


def _batch(name, N, seed, noise=(2e-3, 2e-2)):
    d, model = load_golden(name)
    from oracle import Oracle
    n0 = int(d["meta/num_envs"])
    o = Oracle.from_model(model, n0)
    Q, D, M = o.desc.Q, o.desc.D, o.desc.M
    rng = np.random.default_rng(seed)
    p = "case%d/" % (int(d["meta/num_cases"]) - 1)
    pick = rng.integers(0, n0, N)
    q0 = (d[p + "q0"].reshape(n0, Q)[pick] + noise[0] * rng.standard_normal((N, Q))).astype(np.float32)
    qd0 = (d[p + "qd0"].reshape(n0, D)[pick] + noise[1] * rng.standard_normal((N, D))).astype(np.float32)
    act = (d[p + "act"].reshape(n0, D)[pick] * rng.uniform(0.5, 1.5, (N, D))).astype(np.float32)
    musc = (d[p + "musc"].reshape(n0, M)[pick] * rng.uniform(0.5, 1.5, (N, M))).astype(np.float32) if M else None
    cfg = dict(S=int(d["meta/substeps"]), mm=int(d["meta/mass_matrix_freq"]), dt=float(d["meta/dt"]))
    return d, model, o, q0, qd0, act, musc, cfg


from parity_util import elementwise_bad_envs  # noqa: E402


@pytest.mark.parametrize("name,N", [("HumanoidEnv", 8192), ("SNUHumanoidEnv", 4096), ("AntEnv", 8192)])
def test_cuda_matches_oracles_at_named_size(name, N):
    """The whole batch is stepped on the GPU (forward + adjoint); a spread sample of 256 environments goes through the
    C oracle (forward, bit-exact restatement of the reference) and the host emulation (adjoint)."""
    import torch
    from diffrl_b200.engine import ArticulationEngine
    d, model, o, q0, qd0, act, musc, c = _batch(name, N, 31)
    Q, D, M = o.desc.Q, o.desc.D, o.desc.M
    eng = ArticulationEngine(o.desc, N, "cuda:0")
    t = lambda a: None if a is None else torch.tensor(np.ascontiguousarray(a).ravel(), device="cuda:0")
    rng = np.random.default_rng(4)
    gq_out, gqd_out = rng.standard_normal((N, Q)).astype(np.float32), rng.standard_normal((N, D)).astype(np.float32)
    q, qd, tape, _ = eng.forward(t(q0), t(qd0), t(act), t(musc), c["S"], c["mm"], c["dt"])
    gq, gqd, gact, gm = eng.backward(t(act), t(musc), tape, t(gq_out), t(gqd_out), c["S"], c["mm"], c["dt"])
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(x).all()) for x in (q, qd, gq, gqd, gact))
    sample = np.linspace(0, N - 1, 256).astype(np.int64)          # first, last and a spread of tiles
    ms = None if musc is None else musc[sample]
    oq, oqd = o.forward(q0[sample], qd0[sample], act[sample], ms, c["S"], c["mm"], c["dt"])
    tol = fwd_rtol(name)
    bad_q = elementwise_bad_envs(q.cpu().numpy().reshape(N, Q)[sample], oq, Q, tol)
    bad_qd = elementwise_bad_envs(qd.cpu().numpy().reshape(N, D)[sample], oqd, D, tol)
    bad = sorted(set(bad_q) | set(bad_qd))
    # An environment outside the tolerance must be ILL-CONDITIONED, not wrong: its error has to stay within a small multiple of
    # what the oracle itself moves when that environment's input is perturbed by one fp32 ulp (switching surfaces of the
    # contact model and cond(H) ~ 1e4 amplify rounding; two correct fp32 implementations cannot agree better than that).
    qn, qdn = q.cpu().numpy().reshape(N, Q), qd.cpu().numpy().reshape(N, D)
    for e in bad:
        i = sample[e]
        mi = None if musc is None else musc[i:i + 1]
        moved = 0.0
        for sgn in (1.0, -1.0):
            oq_p, oqd_p = o.forward(q0[i:i + 1] * (1.0 + sgn * 1.2e-7), qd0[i:i + 1] * (1.0 - sgn * 1.2e-7), act[i:i + 1], mi, c["S"], c["mm"], c["dt"])
            moved = max(moved, np.abs(oq_p - oq.reshape(-1, Q)[e]).max() / np.abs(oq).max(), np.abs(oqd_p - oqd.reshape(-1, D)[e]).max() / np.abs(oqd).max())
        err = max(np.abs(qn[i] - oq.reshape(-1, Q)[e]).max() / np.abs(oq).max(), np.abs(qdn[i] - oqd.reshape(-1, D)[e]).max() / np.abs(oqd).max())
        assert err <= max(tol, 8.0 * moved), (name, "env %d: error %.2e vs the oracle, one-ulp sensitivity of the oracle %.2e" % (i, err, moved))
    assert len(bad) <= 8, (name, len(bad))
    # adjoint: host emulation of the same phase code (serial, contiguous scratch, level recursions) on the sample
    emu = EmuSim(model, int(d["meta/num_envs"]))
    emu.N = len(sample)
    eq, eqd, etape, _ = emu.forward(q0[sample].ravel(), qd0[sample].ravel(), act[sample].ravel(), None if ms is None else ms.ravel(), c["S"], c["mm"], c["dt"])
    egq, egqd, egact, egm = emu.backward(act[sample].ravel(), None if ms is None else ms.ravel(), etape, gq_out[sample].ravel(), gqd_out[sample].ravel(), c["S"], c["mm"], c["dt"])
    good = np.setdiff1d(np.arange(len(sample)), bad)
    suspects = set()
    for got, ref, w in ((gq, egq, Q), (gqd, egqd, D), (gact, egact, D)) + (((gm, egm, M),) if M else ()):
        g = got.cpu().numpy().reshape(N, w)[sample][good]
        r = ref.reshape(-1, w)[good]
        suspects |= set(good[elementwise_bad_envs(g, r, w, 4 * GRAD_RTOL)])
    # A gradient outside the tolerance is only acceptable on a SWITCHING SURFACE of the contact / limit model (c >= 0,
    # min(vn, 0), min(kf |vt|, mu c ke), q < lower: the derivative jumps there while the forward value is continuous): the
    # emulation's OWN gradient of that environment must jump by a comparable amount when its input moves by one fp32 ulp.
    assert len(suspects) <= 8, (name, len(suspects))
    one = EmuSim(model, int(d["meta/num_envs"]))
    one.N = 1
    for e in sorted(suspects):
        i = sample[e]
        mi = None if musc is None else musc[i]
        grads = []
        for sgn in (0.0, 1.0, -1.0):
            qp, qdp = q0[i] * (1.0 + sgn * 1.2e-7), qd0[i] * (1.0 - sgn * 1.2e-7)
            _, _, tp, _ = one.forward(qp, qdp, act[i], mi, c["S"], c["mm"], c["dt"])
            grads.append(np.concatenate([x for x in one.backward(act[i], mi, tp, gq_out[i], gqd_out[i], c["S"], c["mm"], c["dt"]) if x is not None]))
        scale = np.abs(grads[0]).max()
        jump = max(np.abs(grads[1] - grads[0]).max(), np.abs(grads[2] - grads[0]).max()) / scale
        mine = np.concatenate([x.cpu().numpy().reshape(N, -1)[i] for x in (gq, gqd, gact) + ((gm,) if M else ())])
        err = np.abs(mine - grads[0]).max() / scale
        assert err <= max(4 * GRAD_RTOL, 8.0 * jump), (name, "env %d: gradient error %.2e, one-ulp jump of the emulation's own gradient %.2e" % (i, err, jump))


def test_snu_bptt128_rollout_matches_reference_kernels():
    """C3's shape: a 128-env-step BPTT window of the muscle humanoid on 4 environments, the GPU kernels against the
    reference's OWN generated CPU kernels (their results recorded in tests/golden/ref_kernels.npz by
    oracle/make_ref_kernel_golden.py).  Forward: every env-step from the reference's state (the chaotic dynamics would
    amplify a 1e-7 rounding difference over 6144 substeps; the per-step comparison is the one that can hold 1e-5-class
    tolerances), plus the free-running GPU trajectory for the first steps.  Adjoint: the full 128-step chain of cotangents
    through both implementations' tapes."""
    import torch
    import make_ref_kernel_golden as rkg
    from diffrl_b200.engine import ArticulationEngine
    from diffrl_b200.modelpack import articulation_from_model
    name, n, T = "SNUHumanoidEnv", rkg.SNU_ENVS, rkg.SNU_STEPS
    d, model = load_golden(name)
    gold = np.load(os.path.join(ROOT, "tests", "golden", "ref_kernels.npz"))
    ref = {k[len("snu_bptt128/"):]: torch.from_numpy(gold[k]) for k in gold.files if k.startswith("snu_bptt128/")}
    S, mm, dt = int(d["meta/substeps"]), int(d["meta/mass_matrix_freq"]), float(d["meta/dt"])
    desc, _ = articulation_from_model(model, int(d["meta/num_envs"]))
    eng = ArticulationEngine(desc, n, "cuda:0")
    Q, D, M = desc.Q, desc.D, desc.M
    assert ref["q"].shape == (T + 1, n * Q) and ref["qd"].shape == (T + 1, n * D)
    g = torch.Generator().manual_seed(rkg.SNU_SEED)
    q, qd = ref["q"][0], ref["qd"][0]
    act = torch.zeros(n * D)
    cu = lambda x: x.to("cuda:0").contiguous()
    ref_states, muscs, tapes_gpu = [], [], []
    worst_step, free_q, free_qd = 0.0, cu(q), cu(qd)
    tol = fwd_rtol(name)
    free_err = []
    for t in range(T):
        musc = rkg.snu_musc(g, n * M)
        if t == 0:        # the recorded run drew the same activations
            assert torch.equal(musc[: ref["musc_head"].numel()], ref["musc_head"])
        q_ref, qd_ref = ref["q"][t + 1], ref["qd"][t + 1]
        gq_, gqd_, tape, _ = eng.forward(cu(q), cu(qd), cu(act), cu(musc), S, mm, dt)        # from the REFERENCE's state
        err = max(float((gq_.cpu() - q_ref).abs().max() / q_ref.abs().max()), float((gqd_.cpu() - qd_ref).abs().max() / (qd_ref.abs().max() + 1.0)))
        worst_step = max(worst_step, err)
        if t < 8:
            free_q, free_qd, _, _ = eng.forward(free_q, free_qd, cu(act), cu(musc), S, mm, dt, want_tape=False)
            free_err.append(float((free_q.cpu() - q_ref).abs().max() / q_ref.abs().max()))
        ref_states.append((q, qd)); muscs.append(musc); tapes_gpu.append(tape)
        q, qd = q_ref.detach(), qd_ref.detach()
    assert worst_step < tol, worst_step
    assert free_err[0] < tol and free_err[-1] < 1e-3, free_err        # free-running: bounded growth over the first 8 env-steps
    # adjoint chain over the whole window (cotangent 1 on the final state): the reference's cotangents are propagated, the GPU
    # adjoint of every env-step gets the reference's incoming cotangents (per-step adjoint parity; the chain's own
    # conditioning would otherwise dominate after a few steps)
    # (the recorded chain stops where the reference's own cotangents overflowed fp32: nothing left to compare beyond)
    rows, cots, gm_errs = [], {}, []
    for k in range(ref["ref_jump"].shape[0]):
        t = T - 1 - k
        gq_r, gqd_r = ref["cot_q"][k], ref["cot_qd"][k]
        cots[t] = (gq_r, gqd_r)
        gq_n, gqd_n = ref["cot_q"][k + 1], ref["cot_qd"][k + 1]
        gq_g, gqd_g, _, gm_g = eng.backward(cu(act), cu(muscs[t]), tapes_gpu[t], cu(gq_r), cu(gqd_r), S, mm, dt)
        scale = float(max(gq_n.abs().max(), gqd_n.abs().max()))
        e_gm = 0.0
        if k % rkg.GRAD_MUSC_EVERY == 0:            # the recorded sample of the muscle-activation gradients
            gm_r = ref["grad_musc"][k // rkg.GRAD_MUSC_EVERY]
            e_gm = float((gm_g.cpu() - gm_r).abs().max() / (gm_r.abs().max() + 1e-30))
            gm_errs.append(e_gm)
        rows.append((t, float((gq_g.cpu() - gq_n).abs().max()) / scale, float((gqd_g.cpu() - gqd_n).abs().max()) / scale,
                     e_gm, scale, float(ref["ref_jump"][k])))
    assert len(rows) >= 64, len(rows)
    for errs, what in (([r[1] for r in rows], "gq"), ([r[2] for r in rows], "gqd"), (gm_errs, "gmusc")):
        errs = np.array(errs)
        assert np.median(errs) < GRAD_RTOL and np.quantile(errs, 0.9) < 4 * GRAD_RTOL, (what, float(np.median(errs)), float(np.quantile(errs, 0.9)))
    # a step outside 8 x the tolerance must sit on a switching surface of the contact / limit model: the reference's (or the
    # kernels') own gradient of that step jumps by a comparable amount when the step's input state moves by 1-4 fp32 ulp
    outliers = [r for r in rows if max(r[1:4]) >= 8 * GRAD_RTOL]
    assert len(outliers) <= max(2, len(rows) // 20), [(r[0], max(r[1:4])) for r in outliers]
    for r in outliers:
        t = r[0]
        q0, qd0 = ref_states[t]
        cot = cots[t]
        _, _, tape0, _ = eng.forward(cu(q0), cu(qd0), cu(act), cu(muscs[t]), S, mm, dt)
        gbase = eng.backward(cu(act), cu(muscs[t]), tape0, cu(cot[0]), cu(cot[1]), S, mm, dt)
        jump = r[5]                                  # the reference's own jump under the same perturbations (recorded)
        # random sign patterns of 1 and 4 ulp: a switching surface nearby flips for some
        for fq, fqd in rkg.perturbations(t, q0.numel(), qd0.numel()):
            qp, qdp = q0 * fq, qd0 * fqd
            _, _, tp, _ = eng.forward(cu(qp), cu(qdp), cu(act), cu(muscs[t]), S, mm, dt)
            gp = eng.backward(cu(act), cu(muscs[t]), tp, cu(cot[0]), cu(cot[1]), S, mm, dt)
            jump = max(jump, float((gp[0] - gbase[0]).abs().max()) / r[4], float((gp[1] - gbase[1]).abs().max()) / r[4])
        assert max(r[1:4]) <= 8.0 * jump, ("step %d: adjoint error %.2e, largest jump of the reference's / the kernels' own gradient "
                                           "under 1-4 ulp input perturbations %.2e" % (t, max(r[1:4]), jump))


@pytest.mark.parametrize("name", ["CartPoleSwingUpEnv", "AntEnv", "HumanoidEnv", "SNUHumanoidEnv", "HopperEnv", "CheetahEnv"])
def test_gpu_derived_state_matches_reference_goldens(name):
    """Every per-phase State field the GPU kernels can dump (DfxDerived: X_sc ... H, L) against the reference's State
    tensors of the first and of the last substep (tests/golden caseK/first|last/*)."""
    import torch
    from diffrl_b200.engine import ArticulationEngine
    d, model = load_golden(name)
    N, S, mm, dt = int(d["meta/num_envs"]), int(d["meta/substeps"]), int(d["meta/mass_matrix_freq"]), float(d["meta/dt"])
    eng = ArticulationEngine.from_model(model, "cuda:0", N)
    t = lambda a: torch.tensor(a, device="cuda:0")
    rel = lambda a, b: float(np.abs(np.asarray(a, np.float64).ravel() - np.asarray(b, np.float64).ravel()).max() / (np.abs(b).max() + 1e-30))
    fields = ["body_X_sc", "body_X_sm", "joint_S_s", "body_v_s", "body_a_s", "body_f_s", "body_ft_s", "joint_tau", "joint_qdd"]
    for k in range(int(d["meta/num_cases"])):
        p = "case%d/" % k
        musc = t(d[p + "musc"]) if (p + "musc") in d.files else None
        # first substep: a 1-substep step of dt/S with a fresh mass matrix
        _, _, _, dv = eng.forward(t(d[p + "q0"]), t(d[p + "qd0"]), t(d[p + "act"]), musc, 1, 1, dt / S, want_tape=False, derived=fields + ["H", "L"])
        for f in fields[:-1] + ["H", "L"]:
            assert rel(dv[f].cpu().numpy(), d[p + "first/" + f]) < 2e-5, (name, k, "first", f)
        assert rel(dv["joint_qdd"].cpu().numpy(), d[p + "first/joint_qdd"]) < 2e-4, (name, k)      # conditioned by H
        # last substep of the full env-step
        _, _, _, dv = eng.forward(t(d[p + "q0"]), t(d[p + "qd0"]), t(d[p + "act"]), musc, S, mm, dt, want_tape=False, derived=fields)
        for f in fields[:-1]:
            assert rel(dv[f].cpu().numpy(), d[p + "last/" + f]) < 20 * fwd_rtol(name), (name, k, "last", f)


@pytest.mark.parametrize("name", ["CartPoleSwingUpEnv", "AntEnv", "HumanoidEnv", "SNUHumanoidEnv", "HopperEnv", "CheetahEnv"])
def test_cuda_adjoint_matches_fp64_finite_differences_all_envs(name):
    import torch
    from diffrl_b200.engine import ArticulationEngine
    N = 4
    d, model, o, q0, qd0, act, musc, c = _batch(name, N, 9, noise=(1e-3, 1e-2))
    Q, D, M = o.desc.Q, o.desc.D, o.desc.M
    rng = np.random.default_rng(3)
    gq_out, gqd_out = rng.standard_normal((N, Q)).astype(np.float32), rng.standard_normal((N, D)).astype(np.float32)
    eng = ArticulationEngine(o.desc, N, "cuda:0")
    t = lambda a: None if a is None else torch.tensor(a.ravel(), device="cuda:0")
    _, _, tape, _ = eng.forward(t(q0), t(qd0), t(act), t(musc), c["S"], c["mm"], c["dt"])
    gq, gqd, gact, gm = eng.backward(t(act), t(musc), tape, t(gq_out), t(gqd_out), c["S"], c["mm"], c["dt"])
    errs = []
    for e in range(N):
        f = o.fd_gradient(q0[e], qd0[e], act[e], None if musc is None else musc[e], gq_out[e], gqd_out[e], c["S"], c["mm"], c["dt"])
        scale = max(np.abs(f[0]).max(), np.abs(f[1]).max(), np.abs(f[2]).max())
        err = max(np.abs(gq.cpu().numpy().reshape(N, Q)[e] - f[0]).max(), np.abs(gqd.cpu().numpy().reshape(N, D)[e] - f[1]).max(),
                  np.abs(gact.cpu().numpy().reshape(N, D)[e] - f[2]).max()) / scale
        if M:
            err = max(err, np.abs(gm.cpu().numpy().reshape(N, M)[e] - f[3]).max() / (np.abs(f[3]).max() + 1e-30))
        errs.append(err)
    # fp32 adjoint vs fp64 central differences of a stiff contact model (48 substeps for the humanoids)
    assert np.median(errs) < (1e-3 if name not in ("HumanoidEnv", "SNUHumanoidEnv") else 5e-3), (name, errs)


@pytest.mark.parametrize("name", ["AntEnv", "HumanoidEnv", "SNUHumanoidEnv", "CheetahEnv"])
def test_bf16_tape_gradients_within_stated_tolerance(name):
    """Config C2 ("bf16 states"): with dfx_set_tape_dtype(1) the tape keeps (v, a, f_tot) of every row as bf16.  The forward
    results are bit-identical to the fp32-tape run, the tape shrinks, the decoded rows are the fp32 rows rounded to bf16,
    and the gradients stay within the tolerance stated in tests/tolerances.py of the REFERENCE's gradients."""
    import torch
    import diffrl_b200
    from diffrl_b200.engine import ArticulationEngine
    from tolerances import BF16_TAPE_ACTION_GRAD_RTOL, BF16_TAPE_STATE_GRAD_RTOL, BF16_TAPE_STATE_GRAD_RTOL_DEFAULT
    d, model = load_golden(name)
    N, S, mm, dt = int(d["meta/num_envs"]), int(d["meta/substeps"]), int(d["meta/mass_matrix_freq"]), float(d["meta/dt"])
    rel = lambda a, b: float(np.abs(np.asarray(a, np.float64).ravel() - np.asarray(b, np.float64).ravel()).max() / (np.abs(b).max() + 1e-30))
    t = lambda a: torch.tensor(a, device="cuda:0")
    eng32 = ArticulationEngine.from_model(model, "cuda:0", N)
    diffrl_b200.set_tape_dtype("bf16")
    try:
        eng16 = ArticulationEngine.from_model(model, "cuda:0", N)
    finally:
        diffrl_b200.set_tape_dtype("fp32")
    assert eng16.tape_bf16 and not eng32.tape_bf16
    assert eng16.tape_floats(S, mm) < 0.9 * eng32.tape_floats(S, mm)
    tol_s = BF16_TAPE_STATE_GRAD_RTOL.get(name, BF16_TAPE_STATE_GRAD_RTOL_DEFAULT)
    for k in range(int(d["meta/num_cases"])):
        p = "case%d/" % k
        musc = t(d[p + "musc"]) if (p + "musc") in d.files else None
        q32, qd32, tape32, _ = eng32.forward(t(d[p + "q0"]), t(d[p + "qd0"]), t(d[p + "act"]), musc, S, mm, dt)
        q16, qd16, tape16, _ = eng16.forward(t(d[p + "q0"]), t(d[p + "qd0"]), t(d[p + "act"]), musc, S, mm, dt)
        assert torch.equal(q32, q16) and torch.equal(qd32, qd16)
        r32, r16 = eng32.tape_rows(tape32, S), eng16.tape_rows(tape16, S)
        L, D, Q = eng32.L, eng32.D, eng32.Q
        head = Q + D + 14 * L + 6 * D
        assert torch.equal(r32[:, :, :head], r16[:, :, :head]) and torch.equal(r32[:, :, head + 18 * L:], r16[:, :, head + 18 * L:])
        assert torch.equal(r32[:, :, head:head + 18 * L].bfloat16().float(), r16[:, :, head:head + 18 * L])
        gq, gqd, gact, gm = eng16.backward(t(d[p + "act"]), musc, tape16, t(d[p + "gq_out"]), t(d[p + "gqd_out"]), S, mm, dt)
        assert rel(gq.cpu().numpy(), d[p + "grad_q"]) < tol_s and rel(gqd.cpu().numpy(), d[p + "grad_qd"]) < tol_s, (name, k)
        assert rel(gact.cpu().numpy(), d[p + "grad_act"]) < BF16_TAPE_ACTION_GRAD_RTOL, (name, k)
        if gm is not None:
            assert rel(gm.cpu().numpy(), d[p + "grad_musc"]) < BF16_TAPE_ACTION_GRAD_RTOL, (name, k)
