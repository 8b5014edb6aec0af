#!/usr/bin/env python
"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Needs a checkout of the reference (jaekor91/HMC-stellar-toy-model):

    SRHMC_REFERENCE_DIR=<checkout> python tests/golden/make_golden.py

Every array written here is an output of the reference's own code
(sampler_RHMC.py / samplers.py / utils.py loaded through oracle/ref_shim.py),
together with the inputs and the np.random draws it consumed, so the fixtures
can be replayed on a box where the reference does not exist.  The reference has
no test-suite of its own, so these files ARE the parity pin (SURVEY.md 8c).
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import ref_shim  # noqa: E402

utils, srhmc, smp = ref_shim.load()


def replay_draws(seed_state, d, niter, P_move=(1.0, 0.0, 0.0)):
    """Replay the exact np.random call sequence of run_RHMC's move-0 loop
    (sampler_RHMC.py:1022, 1046, 1075) from a saved generator state."""
    np.random.set_state(seed_state)
    normals = np.zeros((niter + 1, d))
    lnu = np.zeros(niter + 1)
    for l in range(niter + 1):
        normals[l] = np.random.randn(d)
        np.random.choice([0, 1, 2], p=list(P_move), size=1)
        lnu[l] = np.log(np.random.random(1))[0]
    return normals, lnu


def gym_state(gym):
    keys = ["num_rows", "num_cols", "B_count", "PSF_FWHM_pix", "f_lim", "mB", "flux_to_count",
            "g0", "g1", "g2", "g_xx", "g_ff", "g_ff2", "use_prior", "alpha", "use_Vc", "beta", "Vc_r_pow"]
    out = {k: np.float64(getattr(gym, k)) for k in keys}
    out["V_prior_const"] = np.float64(gym.V_prior_const if gym.V_prior_const is not None else 0.0)
    return out


def kat1():
    """SURVEY.md KAT-1: one star, noise-free data, every L2 function + one step."""
    gym = srhmc.multi_gym(dt=0.2, g_xx=1.0, g_ff=1.0)
    gym.num_rows = gym.num_cols = 32
    gym.D = gym.gen_model(np.array([[19.0, 16.0, 16.0]]))
    gym.V_prior_const = 0.0
    gym.Nobjs, gym.d = 1, 3
    q = np.array([gym.mag2flux_converter(19.5), 16.3, 15.8])
    H, dH = gym.H(q, grad=True)
    p = np.array([0.5, -0.25, 0.125]) * np.sqrt(H)
    q1, p1 = gym.RHMC_single_step(np.copy(q), np.copy(p), 1e-6, 1000)
    E0 = gym.V(q, f_pos=True) + gym.T(p, H)
    E1 = gym.V(q1, f_pos=True) + gym.T(p1, gym.H(q1))
    # ten consecutive steps
    qs, ps = [q], [p]
    qq, pp = np.copy(q), np.copy(p)
    for _ in range(10):
        qq, pp = gym.RHMC_single_step(qq, pp, 1e-6, 1000)
        qs.append(qq)
        ps.append(pp)
    return dict(D=gym.D, q=q, p=p, V=gym.V(q, f_pos=True), dVdq=gym.dVdq(q), H=H, dH=dH, T=gym.T(p, H),
                dphidq=gym.dphidq(q), dtaudq=gym.dtaudq(q, p), dtaudp=gym.dtaudp(q, p), q1=q1, p1=p1,
                E0=E0, E1=E1, q_traj=np.array(qs), p_traj=np.array(ps), dt=0.2, **gym_state(gym))


def kat2():
    """SURVEY.md KAT-2: two stars, prior + repulsion."""
    gym = srhmc.multi_gym(dt=1e-2, g_xx=0.005, g_ff=25.0, g_ff2=2.0)
    gym.num_rows = gym.num_cols = 32
    gym.fmin = gym.mag2flux_converter(20.5)
    gym.fmax = gym.mag2flux_converter(15.0)
    gym.use_prior, gym.alpha = True, 1.5
    gym.use_Vc, gym.beta, gym.Vc_r_pow, gym.f_expnt = True, 1e-4, 4.0, np.zeros(2)
    gym.D = gym.gen_model(np.array([[18.0, 10.0, 12.0], [20.0, 13.0, 12.5]]))
    gym.Nobjs, gym.d = 2, 6
    q = np.array([gym.mag2flux_converter(18.2), 10.2, 11.9, gym.mag2flux_converter(19.7), 12.8, 12.6])
    V = gym.V(q, f_pos=True)
    H, dH = gym.H(q, grad=True)
    p = np.array([0.3, -0.2, 0.1, -0.4, 0.25, 0.15]) * np.sqrt(H)
    qs, ps = [q], [p]
    qq, pp = np.copy(q), np.copy(p)
    for _ in range(5):
        qq, pp = gym.RHMC_single_step(qq, pp, 1e-6, 1000)
        qs.append(qq)
        ps.append(pp)
    return dict(D=gym.D, q=q, p=p, V=V, dVdq=gym.dVdq(q), H=H, dH=dH, T=gym.T(p, H), dphidq=gym.dphidq(q),
                q_traj=np.array(qs), p_traj=np.array(ps), dt=1e-2, **gym_state(gym))


def kat3():
    """SURVEY.md KAT-3: samplers.lightsource_gym functions."""
    ref = srhmc.multi_gym(dt=0.2, g_xx=1.0, g_ff=1.0)
    ref.num_rows = ref.num_cols = 32
    D = ref.gen_model(np.array([[19.0, 16.0, 16.0]]))
    gym = smp.lightsource_gym()
    gym.num_rows = gym.num_cols = 32
    gym.D = D
    gym.f_lim = 0.0
    gym.Nobjs, gym.d = 1, 3
    gym.compute_factors()
    q = np.array([ref.mag2flux_converter(19.5), 16.3, 15.8])
    p = np.array([0.5, -0.25, 0.125])
    dqdt, dpdt, E = gym.RHMC_efficient_computation(q, p, debug=False)
    dVdqq = gym.RHMC_efficient_computation(q, p, debug=False, dVdqq_only=True)
    M = gym.mass_matrix(q)
    return dict(D=D, q=q, p=p, dqdt=dqdt, dpdt=dpdt, E_eff=E, dVdqq=dVdqq,
                factors=np.array([gym.factor0, gym.factor1, gym.factor2]), mass=M,
                dlnDetdq=gym.dlnDetdq(q), dpMpdq=gym.dpMpdq(q, p), K=gym.K(p, M), E=gym.E(q, p, M),
                V=gym.V(q), dVdq=gym.dVdq(q), B_count=np.float64(gym.B_count),
                PSF_FWHM_pix=np.float64(gym.PSF_FWHM_pix))


def chain_one_star(mT=19.0, seed=1903, niter=60, nsteps=10, dt=0.2, size=32, sep=1.0, mM=None):
    """C1/C2: one star, Poisson data, full run_RHMC chain (RHMC-single-full-inference-test.py)."""
    np.random.seed(seed)
    gym = srhmc.multi_gym(dt=0.0, Nsteps=0, g_xx=1.0, g_ff=1.0)
    gym.num_rows = gym.num_cols = size
    gym.V_prior_const = 0.0
    q_true = np.array([[mT, size / 2.0, size / 2.0]])
    gym.gen_mock_data(q_true)
    q_model = np.array([[mM if mM is not None else mT, size / 2.0 + sep, size / 2.0]])
    state = np.random.get_state()
    with ref_shim.quiet():
        gym.run_RHMC(np.copy(q_model), f_pos=True, delta=1e-6, Niter=niter, Nsteps=nsteps, dt=dt,
                     save_traj=False, N_max=1)
    normals, lnu = replay_draws(state, 3, niter)
    return dict(D=gym.D, q_model=q_model, normals=normals, lnu=lnu, niter=niter, nsteps=nsteps, dt=dt,
                q_chain=gym.q_chain, p_chain=gym.p_chain, E_chain=gym.E_chain, V_chain=gym.V_chain,
                T_chain=gym.T_chain, A_chain=gym.A_chain, **gym_state(gym))


def chain_multi(nobj=30, seed=77, niter=12, nsteps=30, dt=1e-2, size=32, use_vc=True):
    """C3: RHMC-big-sim2.py-like crowded field with prior, repulsion and both schedules."""
    gff2_list = utils.scheduler(1 / 10.0, 4.0, 500)
    beta_list = utils.scheduler(1e-2, 1e-12, 500)
    gym = srhmc.multi_gym(dt=0.0, Nsteps=0, g_xx=0.005, g_ff=25.0, g_ff2=2.0)
    np.random.seed(seed)
    gym.num_rows = gym.num_cols = size
    q_true = np.zeros((nobj, 3))
    q_model = np.zeros((nobj, 3))
    alpha = 1.5
    fmin = gym.mag2flux_converter(20.5)
    fmax = gym.mag2flux_converter(15.0)
    mag = gym.flux2mag_converter(utils.gen_pow_law_sample(alpha, fmin, fmax, nobj))
    for i in range(nobj):
        x = np.random.random() * (size - 2.0) + 1.0
        y = np.random.random() * (size - 2.0) + 1.0
        q_true[i] = np.array([mag[i], x, y])
    gym.use_prior, gym.alpha = True, alpha
    gym.fmin, gym.fmax = fmin, fmax
    if use_vc:
        gym.use_Vc, gym.beta, gym.f_expnt, gym.Vc_r_pow = True, 1e-4, np.zeros(nobj), 4.0
    fmin_m = gym.mag2flux_converter(22.9)
    fmax_m = gym.mag2flux_converter(21.0)
    q_model[:, 0] = gym.flux2mag_converter(utils.gen_pow_law_sample(alpha, fmin_m, fmax_m, nobj))
    q_model[:, 1] = np.random.random(size=nobj) * (size - 2.0) + 1.0
    q_model[:, 2] = np.random.random(size=nobj) * (size - 2.0) + 1.0
    gym.gen_mock_data(q_true)
    state = np.random.get_state()
    with ref_shim.quiet():
        gym.run_RHMC(np.copy(q_model), f_pos=True, delta=1e-6, Niter=niter, Nsteps=nsteps, dt=dt,
                     save_traj=False, schedule_g_ff2=gff2_list, schedule_beta=beta_list, N_max=nobj)
    normals, lnu = replay_draws(state, 3 * nobj, niter)
    st = gym_state(gym)
    st["g_ff2"] = np.float64(2.0)  # value at construction; the schedule overrides it per iteration
    st["beta"] = np.float64(1e-4)
    return dict(D=gym.D, q_true=q_true, q_model=q_model, normals=normals, lnu=lnu, niter=niter, nsteps=nsteps,
                dt=dt, schedule_g_ff2=gff2_list[: niter + 1], schedule_beta=beta_list[: niter + 1],
                q_chain=gym.q_chain, p_chain=gym.p_chain, E_chain=gym.E_chain, V_chain=gym.V_chain,
                T_chain=gym.T_chain, A_chain=gym.A_chain, **st)


def single_traj(mT=19.0, mM=20.0, sep=1.0, nsteps=200, dt=0.1, seed=5):
    """C1: RHMC-single-tests.py energy-conservation trajectory (16x16, implicit solver)."""
    np.random.seed(seed)
    gym = srhmc.single_gym(dt=0.0, Nsteps=0, g_xx=1.0, g_ff=1.0)
    gym.num_rows = gym.num_cols = 16
    gym.V_prior_const = 0.0
    gym.gen_mock_data(np.array([[mT, 8.0, 8.0]]))
    q_model = np.array([[mM, 8.0 + sep, 8.0]])
    gym.Nsteps, gym.dt = nsteps, dt
    gym.run_single_RHMC(q_model_0=np.copy(q_model), f_pos=True, solver="implicit", delta=1e-6, p_initial=None)
    return dict(D=gym.D, q_model=q_model, p0=gym.p_chain[0], nsteps=nsteps, dt=dt, q_chain=gym.q_chain,
                p_chain=gym.p_chain, E_chain=gym.E_chain, V_chain=gym.V_chain, T_chain=gym.T_chain,
                **gym_state(gym))


def field_eval(nobj=204, size=64, seed=4):
    """C4-shaped single evaluation: 204 stars on 64x64 with prior (RHMC-big-sim4.py constants)."""
    np.random.seed(seed)
    gym = srhmc.multi_gym(dt=0.0, Nsteps=0, g_xx=0.05, g_ff=4.0, g_ff2=4.0)
    gym.num_rows = gym.num_cols = size
    alpha = 2.0
    fmin = gym.mag2flux_converter(20.0)
    fmax = gym.mag2flux_converter(15.0)
    gym.fmin, gym.fmax = fmin, fmax
    gym.use_prior, gym.alpha = True, alpha
    q_true = np.zeros((nobj, 3))
    q_true[:, 0] = gym.flux2mag_converter(utils.gen_pow_law_sample(alpha, fmin, fmax, nobj))
    q_true[:, 1] = np.random.random(nobj) * (size - 2.0) + 1.0
    q_true[:, 2] = np.random.random(nobj) * (size - 2.0) + 1.0
    gym.gen_mock_data(q_true)
    q = gym.format_q(np.copy(q_true))
    q[0::3] *= 1.05
    q[1::3] += 0.1 * np.random.randn(nobj)
    q[2::3] += 0.1 * np.random.randn(nobj)
    gym.Nobjs, gym.d = nobj, 3 * nobj
    V = gym.V(q, f_pos=True)
    H, dH = gym.H(q, grad=True)
    p = np.random.randn(3 * nobj) * np.sqrt(H)
    gym.dt = 5e-2
    q1, p1 = gym.RHMC_single_step(np.copy(q), np.copy(p), 1e-6, 1000)
    return dict(D=gym.D, q=q, p=p, V=V, dVdq=gym.dVdq(q), H=H, dH=dH, T=gym.T(p, H), q1=q1, p1=p1, dt=5e-2,
                **gym_state(gym))


def light_chains(seed=11, niter=40, mT=19.0):
    """One-star lightsource_gym chains (one-star-inference-single.py): HMC_random, RHMC_random_diag."""
    np.random.seed(seed)
    gym = smp.lightsource_gym()
    gym.num_rows = gym.num_cols = 32
    q0 = np.array([[utils.mag2flux(mT) * gym.flux_to_count, 16.0 + np.random.randn(), 16.0 + np.random.randn()]])
    gym.gen_mock_data(q_true=q0)
    gym.HMC_find_best_dt(q0, default=True, dt_f_coeff=0.05, dt_xy_coeff=2.0)
    dt_vec = np.copy(gym.dt)
    f_lim = utils.mag2flux(22.0) * gym.flux_to_count
    state = np.random.get_state()
    with ref_shim.quiet():
        gym.HMC_random(np.copy(q0), Nchain=1, Niter=niter, steps_max=20, steps_min=5, f_lim=f_lim)
    hmc = dict(q=gym.q_chain[0].copy(), E=gym.E_chain[0, :, 0].copy(), dE=gym.dE_chain[0, :, 0].copy(),
               A=gym.A_chain[0, :, 0].copy())
    # replay the draw sequence: randn(d) at start, then per iteration randn(d), randint, random
    np.random.set_state(state)
    d = 3
    normals = np.zeros((niter + 1, d))
    steps = np.zeros(niter, dtype=np.int64)
    lnu = np.zeros(niter)
    normals[0] = np.random.randn(d)
    for i in range(1, niter + 1):
        normals[i] = np.random.randn(d)
        steps[i - 1] = np.random.randint(low=5, high=20, size=1)[0]
        lnu[i - 1] = np.log(np.random.random(1))[0]
    # diagonal-mass RHMC with the same draw layout
    gym.compute_factors()
    state2 = np.random.get_state()
    with ref_shim.quiet():
        gym.RHMC_random_diag(np.copy(q0), Nchain=1, Niter=niter, steps_max=20, steps_min=5, f_lim=f_lim,
                             dt_global=5e-2)
    diag = dict(q=gym.q_chain[0].copy(), E=gym.E_chain[0, :, 0].copy(), dE=gym.dE_chain[0, :, 0].copy(),
                A=gym.A_chain[0, :, 0].copy())
    np.random.set_state(state2)
    normals2 = np.zeros((niter + 1, d))
    steps2 = np.zeros(niter, dtype=np.int64)
    lnu2 = np.zeros(niter)
    normals2[0] = np.random.randn(d)
    for i in range(1, niter + 1):
        normals2[i] = np.random.randn(d)
        steps2[i - 1] = np.random.randint(low=5, high=20, size=1)[0]
        lnu2[i - 1] = np.log(np.random.random(1))[0]
    return dict(D=gym.D, q0=q0.reshape(-1), dt_vec=dt_vec, f_lim=f_lim, niter=niter,
                hmc_q=hmc["q"], hmc_E=hmc["E"], hmc_dE=hmc["dE"], hmc_A=hmc["A"],
                hmc_normals=normals, hmc_steps=steps, hmc_lnu=lnu,
                diag_q=diag["q"], diag_E=diag["E"], diag_dE=diag["dE"], diag_A=diag["A"],
                diag_normals=normals2, diag_steps=steps2, diag_lnu=lnu2, dt_global=5e-2,
                factors=np.array([gym.factor0, gym.factor1, gym.factor2]),
                B_count=np.float64(gym.B_count), PSF_FWHM_pix=np.float64(gym.PSF_FWHM_pix))


def light_hess(seed=21, niter=40, mT=19.0):
    """lightsource_gym.RHMC_random (Hessian metric) and RHMC_efficient_computation on Poisson data."""
    np.random.seed(seed)
    gym = smp.lightsource_gym()
    gym.num_rows = gym.num_cols = 32
    q0 = np.array([[utils.mag2flux(mT) * gym.flux_to_count, 16.0 + 0.3 * np.random.randn(), 16.0 + 0.3 * np.random.randn()]])
    gym.gen_mock_data(q_true=q0)
    f_lim = utils.mag2flux(22.0) * gym.flux_to_count
    gym.f_lim = f_lim
    gym.Nobjs, gym.d = 1, 3
    qe = q0.reshape(-1) * np.array([1.02, 1.0, 1.0]) + np.array([0.0, 0.21, -0.13])
    pe = np.array([0.01, -0.4, 0.3])
    dqdt, dpdt, E = gym.RHMC_efficient_computation(qe, pe, debug=False)
    d2 = gym.RHMC_efficient_computation(qe, pe, debug=False, dVdqq_only=True)
    q_start = np.copy(q0)
    with ref_shim.quiet():
        gym.RHMC_random(q_start, Nchain=1, Niter=niter, steps_max=12, steps_min=4, f_lim=f_lim, dt_RHMC_xy=0.3,
                        dt_RHMC_f=0.3, debug=False)
    return dict(D=gym.D, q0=q0.reshape(-1), f_lim=f_lim, niter=niter, seed=seed, qe=qe, pe=pe, dqdt=dqdt, dpdt=dpdt,
                E_eff=E, dVdqq=d2, q_chain=gym.q_chain[0].copy(), E_chain=gym.E_chain[0, :, 0].copy(),
                dE_chain=gym.dE_chain[0, :, 0].copy(), A_chain=gym.A_chain[0, :, 0].copy(),
                q_after=q_start.reshape(-1).copy(), next_uniform=np.random.random(1),
                B_count=np.float64(gym.B_count), PSF_FWHM_pix=np.float64(gym.PSF_FWHM_pix))


def best_dt(seed=31, mT=19.0):
    """lightsource_gym.HMC_find_best_dt followed by a short HMC_random (one-star-inference-single.py:21-71)."""
    np.random.seed(seed)
    gym = smp.lightsource_gym()
    gym.num_rows = gym.num_cols = 32
    q0 = np.array([[utils.mag2flux(mT) * gym.flux_to_count, 16.0 + np.random.randn(), 16.0 + np.random.randn()]])
    gym.gen_mock_data(q_true=q0)
    model_data = np.ones((32, 32)) * gym.B_count * 1.1
    qs = q0.reshape(-1)
    Vs = gym.V_single(qs, model_data)
    gs = np.array(gym.dVdq_single(qs, model_data, return_all=True))
    with ref_shim.quiet():
        gym.HMC_find_best_dt(q0, default=False, dt_f_coeff=1, dt_xy_coeff=10, Niter_per_trial=20, Ntrial=6,
                             steps_min=5, steps_max=12, A_target_f=0.99, A_target_xy=0.5)
    dt_vec = np.copy(gym.dt)
    f_lim = utils.mag2flux(22.0) * gym.flux_to_count
    with ref_shim.quiet():
        gym.HMC_random(np.copy(q0), Nchain=1, Niter=25, steps_max=20, steps_min=5, f_lim=f_lim)
    return dict(D=gym.D, q0=qs, seed=seed, dt_vec=dt_vec, f_lim=f_lim, model_data=model_data, V_single=Vs,
                dVdq_single=gs, q_chain=gym.q_chain[0].copy(), E_chain=gym.E_chain[0, :, 0].copy(),
                A_chain=gym.A_chain[0, :, 0].copy(), next_uniform=np.random.random(1),
                B_count=np.float64(gym.B_count), PSF_FWHM_pix=np.float64(gym.PSF_FWHM_pix))


def rj_chain(seed=77, niter=60, nobj=20, nmodel=5, nsteps=5, dt=5e-2):
    """RHMC-big-sim4.py flow in miniature: reversible-jump RHMC (birth/death, split/merge around two RHMC legs)."""
    gym = srhmc.multi_gym(dt=0.0, Nsteps=0, g_xx=0.05, g_ff=4.0, g_ff2=4.0)
    np.random.seed(seed)
    gym.num_rows = gym.num_cols = 32
    q_true = np.zeros((nobj, 3))
    q_model = np.zeros((nmodel, 3))
    alpha = 2.0
    fmin = gym.mag2flux_converter(20.0)
    fmax = gym.mag2flux_converter(15.0)
    mag = gym.flux2mag_converter(utils.gen_pow_law_sample(alpha, fmin, fmax, nobj))
    for i in range(nobj):
        x = np.random.random() * (gym.num_rows - 2.0) + 1.0
        y = np.random.random() * (gym.num_cols - 2.0) + 1.0
        q_true[i] = np.array([mag[i], x, y])
    gym.fmin, gym.fmax = fmin, fmax
    gym.K_split, gym.beta_a, gym.beta_b = 1.0, 4.0, 4.0
    gym.use_prior, gym.alpha = True, alpha
    mag = gym.flux2mag_converter(utils.gen_pow_law_sample(alpha, fmin, fmax, nmodel))
    q_model[:, 0] = mag
    q_model[:, 1] = np.random.random(size=nmodel) * (gym.num_rows - 2.0) + 1.0
    q_model[:, 2] = np.random.random(size=nmodel) * (gym.num_cols - 2.0) + 1.0
    gym.gen_mock_data(q_true)
    with ref_shim.quiet():
        gym.run_RHMC(np.copy(q_model), f_pos=True, delta=1e-6, Niter=niter, Nsteps=nsteps, dt=dt, save_traj=False,
                     verbose=False, q_true=q_true, P_move=[0.4, 0.3, 0.3], N_max=30)
    return dict(D=gym.D, q_true=q_true, q_model=q_model, seed=seed, niter=niter, nsteps=nsteps, dt=dt,
                q_chain=gym.q_chain, p_chain=gym.p_chain, E_chain=gym.E_chain, V_chain=gym.V_chain, T_chain=gym.T_chain,
                A_chain=gym.A_chain, move_chain=gym.move_chain, N_chain=gym.N_chain, next_uniform=np.random.random(1),
                **gym_state(gym))


def find_peaks(seed=41):
    """lightsource_gym.find_peaks (samplers.py:129-254) on a 32x32 image with three stars; the jitter draws are recorded."""
    np.random.seed(seed)
    gym = smp.lightsource_gym()
    gym.num_rows = gym.num_cols = 32
    fl = lambda m: utils.mag2flux(m) * gym.flux_to_count
    q_true = np.array([[fl(18.0), 9.3, 11.7], [fl(19.5), 21.2, 20.4], [fl(20.5), 24.6, 7.9]])
    gym.gen_mock_data(q_true=q_true)
    state = np.random.get_state()
    n_side = int(0.25 * 32) - 1
    jitter = np.random.randn(n_side * n_side, 2)
    np.random.set_state(state)
    with ref_shim.quiet():
        gym.find_peaks(linear_pix_density=0.25, Nstep=400, dt_f_coeff=1e-1, dt_xy_coeff=1e-1)
    q_final = np.copy(gym.q_seed)
    np.random.set_state(state)
    with ref_shim.quiet():
        gym.find_peaks(linear_pix_density=0.25, no_perturb=True)
    return dict(D=gym.D, q_true=q_true, jitter=jitter, q_seed0=np.copy(gym.q_seed), q_seed=q_final, seed=seed,
                next_uniform=np.random.random(1), B_count=np.float64(gym.B_count), PSF_FWHM_pix=np.float64(gym.PSF_FWHM_pix),
                mB=np.float64(gym.mB), flux_to_count=np.float64(gym.flux_to_count))


def conv_stats():
    """utils.convergence_stats (utils.py:86-167, Python-2 division restored by the shim) on AR(1) chains with different
    autocorrelation per variable, and on chains with a short and an odd thinned length."""
    out = {}
    for tag, (seed, nchain, niter, thin, warm) in {"a": (3, 8, 600, 5, 0), "b": (4, 5, 333, 2, 51)}.items():
        rng = np.random.RandomState(seed)
        phi = np.array([0.2, 0.7, 0.95])
        x = np.zeros((nchain, niter, 3))
        eps = rng.randn(nchain, niter, 3)
        for t in range(1, niter):
            x[:, t] = phi * x[:, t - 1] + eps[:, t]
        x += rng.randn(nchain, 1, 3) * 0.1
        R, neff = utils.convergence_stats(x, thin_rate=thin, warm_up_num=warm)
        out.update({"chain_" + tag: x, "thin_" + tag: thin, "warm_" + tag: warm, "R_" + tag: R, "neff_" + tag: neff})
    return out


def main():
    only = sys.argv[1:]
    if only:
        makers = {"light_hess": light_hess, "best_dt": best_dt, "rj_chain": rj_chain, "conv_stats": conv_stats, "find_peaks": find_peaks}
        for name in only:
            arrays = makers[name]()
            path = os.path.join(HERE, name + ".npz")
            np.savez_compressed(path, **arrays)
            print("%-24s %8.1f KB" % (name, os.path.getsize(path) / 1024.0))
        return
    cases = {
        "kat1": kat1(),
        "kat2": kat2(),
        "kat3": kat3(),
        "chain_one_star_m19": chain_one_star(19.0, seed=1903, sep=0.0),
        "chain_one_star_m21": chain_one_star(21.0, seed=2103, sep=0.0),
        "chain_one_star_m20_sep1": chain_one_star(20.0, seed=2003, mM=19.0, sep=1.0, dt=0.05, niter=40),
        "chain_one_star_m15": chain_one_star(15.0, seed=1503, sep=0.0, niter=30),
        "chain_multi30_vc": chain_multi(30, niter=12),
        "chain_multi100": chain_multi(100, niter=4, nsteps=20, dt=5e-4, use_vc=False),
        "single_traj": single_traj(),
        "field_eval_204": field_eval(),
        "light_chains": light_chains(),
        "light_hess": light_hess(),
        "best_dt": best_dt(),
        "rj_chain": rj_chain(),
        "conv_stats": conv_stats(),
        "find_peaks": find_peaks(),
    }
    for name, arrays in cases.items():
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **arrays)
        print("%-24s %8.1f KB" % (name, os.path.getsize(path) / 1024.0))


if __name__ == "__main__":
    main()
