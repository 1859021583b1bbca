"""`gem.make(env_id, **kwargs)` for a matrix of user-level kwargs — motor parameters / limits / nominal values, supplies, loads, taus,
state filters, reference generators with explicit ranges and margins, reward-function settings, constraint specs, wrappers — built once
with the unmodified reference (`--impl reference`) and once with this repo's host package aliased as `gym_electric_motor`
(`--impl b200`, which also derives the C-ABI config).  Each case is a source snippet evaluated with `gem` bound to the respective
package, so both sides see literally the same user code.  Prints {case: {"verdict", "summary"}}; the summaries (names, limits, nominal
state, spaces, tau, motor / load parameters, supply, reward weights / range / bias, constraint list, generator margins) must agree.
No stepping, no GPU.  `--impl reference` needs the reference checkout (REF); its output is stored in
tests/golden/agent_surface/kwargs_matrix_reference.npz (tests/golden/make_agent_surface_golden.py)."""
import json
import sys
import warnings

import numpy as np

REF = "/root/reference"
HERE = __file__.rsplit("/", 2)[0]

PRELUDE = """
import numpy as np
ps = gem.physical_systems
rg = gem.reference_generators
rf = gem.reward_functions
psw = gem.physical_system_wrappers
"""

CASES = {
    "pmsm_motor_parameter": 'gem.make("Cont-CC-PMSM-v0", motor=dict(motor_parameter=dict(r_s=25e-3, l_d=0.5e-3, psi_p=70e-3, p=4)))',
    "pmsm_limits_nominal": 'gem.make("Cont-SC-PMSM-v0", motor=dict(limit_values=dict(omega=500.0, i=300.0, u=400.0), nominal_values=dict(omega=400.0, i=200.0, u=400.0)))',
    "pmsm_supply_dict": 'gem.make("Finite-CC-PMSM-v0", supply=dict(u_nominal=350.0))',
    "pmsm_supply_instance": 'gem.make("Cont-TC-PMSM-v0", supply=ps.IdealVoltageSupply(u_nominal=500.0))',
    "pmsm_tau_filter": 'gem.make("Cont-CC-PMSM-v0", tau=5e-5, state_filter=["omega", "i_sd", "i_sq", "epsilon"])',
    "pmsm_load_poly": 'gem.make("Cont-CC-PMSM-v0", load=ps.PolynomialStaticLoad(load_parameter=dict(a=0.1, b=0.02, c=1e-4, j_load=0.01)))',
    "pmsm_load_const": 'gem.make("Cont-TC-PMSM-v0", load=ps.ConstantSpeedLoad(omega_fixed=150.0))',
    "pmsm_load_dict": 'gem.make("Cont-SC-PMSM-v0", load=dict(load_parameter=dict(a=0.0, b=0.0, c=0.0, j_load=2e-3)))',
    "synrm_parameter": 'gem.make("Cont-CC-SynRM-v0", motor=dict(motor_parameter=dict(l_d=80e-3, l_q=20e-3, r_s=0.7)))',
    "eesm_parameter": 'gem.make("Cont-CC-EESM-v0", motor=dict(motor_parameter=dict(r_e=8e-3, l_e=2e-3, l_m=1.4e-3)), supply=dict(u_nominal=320.0))',
    "scim_parameter": 'gem.make("Cont-SC-SCIM-v0", motor=dict(motor_parameter=dict(r_s=3.0, r_r=1.4, l_m=0.15), limit_values=dict(i=8.0)))',
    "dfim_parameter": 'gem.make("Cont-TC-DFIM-v0", motor=dict(motor_parameter=dict(r_s=5e-3, l_m=3e-3)))',
    "permex_parameter": 'gem.make("Cont-SC-PermExDc-v0", motor=dict(motor_parameter=dict(r_a=25e-3, l_a=3e-5, psi_e=0.2, j_rotor=0.03)))',
    "series_limits": 'gem.make("Cont-CC-SeriesDc-v0", motor=dict(limit_values=dict(i=120.0, omega=250.0), nominal_values=dict(i=60.0)))',
    "shunt_supply": 'gem.make("Finite-SC-ShuntDc-v0", supply=dict(u_nominal=300.0), tau=2e-5)',
    "extex_parameter": 'gem.make("Cont-TC-ExtExDc-v0", motor=dict(motor_parameter=dict(l_e_prime=0.01, r_e=6.0)))',
    "interlock_b6": 'gem.make("Finite-CC-PMSM-v0", converter=dict(interlocking_time=1e-6))',
    "converter_instance_1qc": 'gem.make("Cont-CC-PermExDc-v0", converter=ps.ContOneQuadrantConverter())',
    "converter_instance_2qc": 'gem.make("Finite-SC-SeriesDc-v0", converter=ps.FiniteTwoQuadrantConverter(interlocking_time=2e-6))',
    "wiener_ranges": 'gem.make("Cont-SC-PMSM-v0", reference_generator=rg.WienerProcessReferenceGenerator(reference_state="omega", sigma_range=(1e-3, 1e-2), episode_lengths=(200, 300), limit_margin=(-0.2, 0.7)))',
    "wiener_dict": 'gem.make("Cont-TC-PMSM-v0", reference_generator=dict(sigma_range=(5e-3, 5e-2), limit_margin=0.4))',
    "const_ref": 'gem.make("Cont-SC-PermExDc-v0", reference_generator=rg.ConstReferenceGenerator(reference_state="omega", reference_value=0.35))',
    "sinus_ref": 'gem.make("Cont-SC-SeriesDc-v0", reference_generator=rg.SinusoidalReferenceGenerator(reference_state="omega", amplitude_range=(0.1, 0.4), frequency_range=(2, 9), offset_range=(-0.1, 0.3), episode_lengths=1000))',
    "step_ref_margin": 'gem.make("Cont-TC-SynRM-v0", reference_generator=rg.StepReferenceGenerator(reference_state="torque", limit_margin=(-0.5, 0.5), amplitude_range=(0, 0.6)))',
    "triangle_ref_other_state": 'gem.make("Cont-CC-PermExDc-v0", reference_generator=rg.TriangularReferenceGenerator(reference_state="omega"))',
    "multi_ref": 'gem.make("Cont-CC-PMSM-v0", reference_generator=rg.MultipleReferenceGenerator([rg.ConstReferenceGenerator(reference_state="i_sd", reference_value=-0.1), rg.WienerProcessReferenceGenerator(reference_state="i_sq", limit_margin=0.5)]))',
    "switched_ref": 'gem.make("Cont-SC-PMSM-v0", reference_generator=rg.SwitchedReferenceGenerator([rg.SinusoidalReferenceGenerator(reference_state="omega"), rg.WienerProcessReferenceGenerator(reference_state="omega")], p=[0.3, 0.7], super_episode_length=(500, 900)))',
    "reward_dict": 'gem.make("Cont-CC-PMSM-v0", reward_function=dict(gamma=0.99, reward_power=2))',
    "reward_weights_bias": 'gem.make("Cont-CC-PMSM-v0", reward_function=rf.WeightedSumOfErrors(reward_weights=dict(i_sd=2.0, i_sq=1.0, omega=0.5), bias="positive", gamma=0.8))',
    "reward_violation": 'gem.make("Cont-SC-PermExDc-v0", reward_function=rf.WeightedSumOfErrors(reward_weights=[1, 0, 0.5, 0, 0], violation_reward=-42.0, reward_power=[1, 1, 0.5, 1, 1], bias=0.2))',
    "constraints_names": 'gem.make("Cont-CC-PMSM-v0", constraints=("i_sd", "i_sq", "omega"))',
    "constraints_squared": 'gem.make("Cont-CC-EESM-v0", constraints=(gem.constraints.SquaredConstraint(("i_sd", "i_sq")), gem.constraints.LimitConstraint(("i_e", "torque"))))',
    "constraints_none": 'gem.make("Finite-TC-SCIM-v0", constraints=())',
    "wrappers_cossin_dead": 'gem.make("Cont-CC-PMSM-v0", physical_system_wrappers=[psw.CosSinProcessor(angle="epsilon"), psw.DqToAbcActionProcessor.make("PMSM"), psw.DeadTimeProcessor(steps=2)])',
    "wrappers_flux_observer": 'gem.make("Cont-CC-SCIM-v0", physical_system_wrappers=[psw.FluxObserver()], state_filter=["i_sd", "i_sq", "psi_abs", "psi_angle"])',
    "wrappers_noise": 'gem.make("Cont-SC-PermExDc-v0", physical_system_wrappers=[psw.StateNoiseProcessor(states=["omega", "i"], random_dist="uniform", random_kwargs=dict(low=-0.01, high=0.01))])',
    "rc_supply": 'gem.make("Cont-SC-PermExDc-v0", supply=ps.RCVoltageSupply(u_nominal=80.0, supply_parameter=dict(R=0.5, C=2e-3)))',
    "ac1_supply": 'gem.make("Cont-CC-SeriesDc-v0", supply=ps.AC1PhaseSupply(u_nominal=230.0, supply_parameter=dict(frequency=50, phase=0.3)))',
    "motor_initializer": 'gem.make("Cont-CC-PMSM-v0", motor=dict(motor_initializer=dict(states=dict(i_sd=-10.0, i_sq=20.0, epsilon=1.0))))',
    "initializer_partial_quirk": 'gem.make("Cont-CC-PMSM-v0", motor=dict(motor_initializer=dict(states=dict(i_sq=20.0))))',
    "initializer_reversed": 'gem.make("Cont-SC-PMSM-v0", motor=dict(motor_initializer=dict(states=dict(epsilon=0.5, i_sq=15.0, i_sd=-5.0))))',
    "initializer_eesm": 'gem.make("Cont-CC-EESM-v0", motor=dict(motor_initializer=dict(states=dict(i_e=30.0, i_sd=-10.0))))',
    "initializer_extex": 'gem.make("Cont-CC-ExtExDc-v0", motor=dict(motor_initializer=dict(states=dict(i_e=1.5, i_a=10.0))))',
    "initializer_scim": 'gem.make("Cont-CC-SCIM-v0", motor=dict(motor_initializer=dict(states=dict(i_sbeta=1.0, i_salpha=-0.5, psi_ralpha=0.0, psi_rbeta=0.0, epsilon=0.0))))',
    "initializer_load_const": 'gem.make("Cont-SC-PermExDc-v0", load=dict(load_initializer=dict(states=dict(omega=50.0))))',
    "euler_solver": 'gem.make("Cont-CC-PMSM-v0", ode_solver=ps.EulerSolver())',
    "euler_solver_n": 'gem.make("Finite-SC-PermExDc-v0", ode_solver=ps.EulerSolver(nsteps=4))',
    "solve_ivp_solver": 'gem.make("Cont-TC-SCIM-v0", ode_solver=ps.ScipySolveIvpSolver())',
    "odeint_solver": 'gem.make("Cont-CC-SynRM-v0", ode_solver=ps.ScipyOdeIntSolver())',
    "ext_speed_load": 'gem.make("Cont-CC-PMSM-v0", ode_solver=ps.EulerSolver(), load=ps.ExternalSpeedLoad(speed_profile=lambda t, a, f: a * np.sin(2 * np.pi * f * t) + 60.0, speed_profile_kwargs=dict(a=20.0, f=25.0)))',
    "ext_speed_load_dc": 'gem.make("Cont-CC-SeriesDc-v0", ode_solver=ps.EulerSolver(nsteps=2), load=ps.ExternalSpeedLoad(speed_profile=lambda t: 30.0 + 500.0 * t, tau=1e-4))',
    "control_space_dq": 'gem.make("Cont-CC-PMSM-v0", physical_system_wrappers=[psw.DqToAbcActionProcessor.make("PMSM")], load=ps.ConstantSpeedLoad(omega_fixed=200.0))',
    "dfim_dq_wrapper": 'gem.make("Cont-CC-DFIM-v0", physical_system_wrappers=[psw.FluxObserver(), psw.DqToAbcActionProcessor.make("DFIM")])',
    "rc_supply_pmsm": 'gem.make("Cont-CC-PMSM-v0", supply=ps.RCVoltageSupply(u_nominal=300.0, supply_parameter=dict(R=0.2, C=1e-3)), converter=dict(interlocking_time=2e-6))',
    "ac1_supply_finite": 'gem.make("Finite-CC-PermExDc-v0", supply=ps.AC1PhaseSupply(u_nominal=60.0, supply_parameter=dict(frequency=400, phase=1.0)))',
    "interlock_cont_multi": 'gem.make("Cont-CC-ExtExDc-v0", converter=ps.ContMultiConverter([ps.ContFourQuadrantConverter(interlocking_time=1e-6), ps.ContTwoQuadrantConverter(interlocking_time=2e-6)]))',
    "finite_multi_interlock": 'gem.make("Finite-CC-ExtExDc-v0", converter=ps.FiniteMultiConverter([ps.FiniteFourQuadrantConverter(interlocking_time=1e-6), ps.FiniteTwoQuadrantConverter()]))',
    "const_ref_reward_pmsm": 'gem.make("Cont-CC-PMSM-v0", reference_generator=rg.MultipleReferenceGenerator([rg.ConstReferenceGenerator(reference_state="i_sd", reference_value=-0.2), rg.ConstReferenceGenerator(reference_state="i_sq", reference_value=0.3)]), reward_function=dict(gamma=0.95, reward_power=2))',
    "const_ref_terminates": 'gem.make("Cont-CC-PermExDc-v0", reference_generator=rg.ConstReferenceGenerator(reference_state="i", reference_value=0.9), load=ps.ConstantSpeedLoad(omega_fixed=10.0))',
    "const_ref_bias_violation": 'gem.make("Finite-SC-PermExDc-v0", reference_generator=rg.ConstReferenceGenerator(reference_state="omega", reference_value=0.5), reward_function=rf.WeightedSumOfErrors(bias="positive", violation_reward=-7.0, gamma=0.5), tau=1e-4)',
    "const_ref_squared_constraint": 'gem.make("Cont-TC-SynRM-v0", reference_generator=rg.ConstReferenceGenerator(reference_state="torque", reference_value=0.1), constraints=(gem.constraints.SquaredConstraint(("i_sd", "i_sq")), "omega"), reward_function=dict(reward_power=0.5))',
    "currentsum_extex": 'gem.make("Cont-CC-ExtExDc-v0", physical_system_wrappers=[psw.CurrentSumProcessor(currents=["i_a", "i_e"])])',
    "dead_before_dq": 'gem.make("Cont-CC-PMSM-v0", physical_system_wrappers=[psw.DeadTimeProcessor(steps=1), psw.DqToAbcActionProcessor.make("PMSM")])',
    "dq_then_dead": 'gem.make("Cont-SC-PMSM-v0", physical_system_wrappers=[psw.DqToAbcActionProcessor.make("PMSM"), psw.DeadTimeProcessor(steps=2)])',
    "eesm_dq": 'gem.make("Cont-CC-EESM-v0", physical_system_wrappers=[psw.DqToAbcActionProcessor.make("EESM")])',
    "synrm_dq": 'gem.make("Cont-TC-SynRM-v0", physical_system_wrappers=[psw.DqToAbcActionProcessor.make("SynRM")])',
    "torque_limit_explicit": 'gem.make("Cont-TC-PMSM-v0", motor=dict(limit_values=dict(torque=100.0), nominal_values=dict(torque=80.0)))',
    "j_rotor_sc": 'gem.make("Cont-SC-PMSM-v0", motor=dict(motor_parameter=dict(j_rotor=0.01)), load=dict(load_parameter=dict(a=0.02, b=0.001, c=0.0, j_load=0.005)))',
    "scim_fin_interlock": 'gem.make("Finite-CC-SCIM-v0", converter=dict(interlocking_time=5e-7))',
    "dfim_fin_interlock": 'gem.make("Finite-TC-DFIM-v0", converter=ps.FiniteMultiConverter([ps.FiniteB6BridgeConverter(interlocking_time=1e-6), ps.FiniteB6BridgeConverter(interlocking_time=1e-6)]))',
    "eesm_fin_defaults_tau": 'gem.make("Finite-CC-EESM-v0", tau=2e-5)',
    "reward_weights_list": 'gem.make("Cont-CC-ShuntDc-v0", reward_function=dict(reward_weights=[0, 0, 1.0, 0.5, 0, 0, 0.25]))',
    "limit_margin_multi": 'gem.make("Cont-CC-SCIM-v0", reference_generator=rg.MultipleReferenceGenerator([rg.WienerProcessReferenceGenerator, rg.WienerProcessReferenceGenerator], sub_args=[dict(reference_state="i_sd", limit_margin=(0.0, 0.3)), dict(reference_state="i_sq", limit_margin=0.6)]))',
    "cossin_flux_angle": 'gem.make("Cont-SC-SCIM-v0", physical_system_wrappers=[psw.FluxObserver(), psw.CosSinProcessor(angle="psi_angle")])',
    # ---- user errors: both sides must refuse (tests compare the exception type; the message where the reference has a stable one)
    "err_unknown_motor_key": 'gem.make("Cont-CC-PMSM-v0", motor=dict(motor_parameter=dict(r_x=1.0)))',
    "err_unknown_limit_key": 'gem.make("Cont-CC-PMSM-v0", motor=dict(limit_values=dict(current=1.0)))',
    "err_unknown_load_key": 'gem.make("Cont-SC-PMSM-v0", load=dict(load_parameter=dict(d=1.0)))',
    "err_init_out_of_bounds": 'gem.make("Cont-CC-PMSM-v0", motor=dict(motor_initializer=dict(states=dict(i_sd=-1000.0))))',
    "err_string_component": 'gem.make("Cont-CC-PMSM-v0", converter="Finite-B6C")',
    "err_state_filter_name": 'gem.make("Cont-CC-PMSM-v0", state_filter=["i_sd", "nope"])',
    "err_reference_state": 'gem.make("Cont-CC-PMSM-v0", reference_generator=rg.WienerProcessReferenceGenerator(reference_state="nope"))',
    "err_reward_weight_name": 'gem.make("Cont-CC-PMSM-v0", reward_function=dict(reward_weights=dict(nope=1.0)))',
    "err_constraint_name": 'gem.make("Cont-CC-PMSM-v0", constraints=("nope",))',
    "err_dead_time_zero": 'gem.make("Cont-CC-PMSM-v0", physical_system_wrappers=[psw.DeadTimeProcessor(steps=0)])',
    "err_cossin_angle": 'gem.make("Cont-CC-PMSM-v0", physical_system_wrappers=[psw.CosSinProcessor(angle="nope")])',
    "err_flux_observer_pmsm": 'gem.make("Cont-CC-PMSM-v0", physical_system_wrappers=[psw.FluxObserver()])',
    "err_dq_on_dc": 'gem.make("Cont-CC-PermExDc-v0", physical_system_wrappers=[psw.DqToAbcActionProcessor.make("PMSM")])',
    "err_scim_dq_without_observer": 'gem.make("Cont-CC-SCIM-v0", physical_system_wrappers=[psw.DqToAbcActionProcessor.make("SCIM")])',
    "err_limit_margin_type": 'gem.make("Cont-SC-PMSM-v0", reference_generator=rg.WienerProcessReferenceGenerator(reference_state="omega", limit_margin="wide"))',
    "err_multi_same_state": 'gem.make("Cont-CC-PMSM-v0", reference_generator=rg.MultipleReferenceGenerator([rg.WienerProcessReferenceGenerator(reference_state="i_sd"), rg.ConstReferenceGenerator(reference_state="i_sd")]))',
    "err_unknown_env_id": 'gem.make("Cont-CC-BLDC-v0")',
    "shunt_cc_default_filter": 'gem.make("Cont-CC-ShuntDc-v0", state_filter=["i_a", "i_e", "i_sum"])',
    "shunt_limits": 'gem.make("Finite-TC-ShuntDc-v0", motor=dict(limit_values=dict(i_a=80.0, i_e=4.0, omega=300.0)))',
    "extex_supply_limits": 'gem.make("Finite-CC-ExtExDc-v0", supply=dict(u_nominal=100.0), motor=dict(nominal_values=dict(i_a=40.0, i_e=3.0)))',
    "dfim_supply": 'gem.make("Finite-SC-DFIM-v0", supply=dict(u_nominal=700.0))',
    "scim_load": 'gem.make("Cont-TC-SCIM-v0", load=ps.PolynomialStaticLoad(dict(a=0.05, b=0.01, c=0.0, j_load=5e-3)))',
    "eesm_sc_reward": 'gem.make("Cont-SC-EESM-v0", reward_function=dict(reward_weights=dict(omega=1.0, i_e=0.1), gamma=0.95))',
    "eesm_ref_ie": 'gem.make("Cont-CC-EESM-v0", reference_generator=rg.MultipleReferenceGenerator([rg.WienerProcessReferenceGenerator(reference_state="i_e", limit_margin=(0.0, 0.6)), rg.ConstReferenceGenerator(reference_state="i_sq", reference_value=0.2)]))',
    "limit_constraint_all": 'gem.make("Cont-CC-PermExDc-v0", constraints=(gem.constraints.LimitConstraint("all_states"),))',
    "limit_constraint_mixed": 'gem.make("Cont-SC-PMSM-v0", constraints=("omega", gem.constraints.SquaredConstraint(("i_sd", "i_sq")), "torque"))',
    "reward_power_scalar": 'gem.make("Cont-TC-PermExDc-v0", reward_function=dict(reward_power=0.5, bias=1.0))',
    "reward_normed": 'gem.make("Cont-CC-SCIM-v0", reward_function=rf.WeightedSumOfErrors(reward_weights=dict(i_sd=3.0, i_sq=1.0), normed_reward_weights=True))',
    "laplace_ref": 'gem.make("Cont-SC-ShuntDc-v0", reference_generator=rg.LaplaceProcessReferenceGenerator(reference_state="omega", sigma_range=(1e-3, 1e-2)))',
    "sawtooth_ref": 'gem.make("Finite-SC-PMSM-v0", reference_generator=rg.SawtoothReferenceGenerator(reference_state="omega", amplitude_range=(0.0, 0.3), frequency_range=(1, 4)))',
    "gaussian_initializer": 'gem.make("Cont-CC-SeriesDc-v0", motor=dict(motor_initializer=dict(random_init="gaussian", random_params=(25.0, 3.0), states=dict(i=0.0))))',
    "uniform_initializer_pmsm": 'gem.make("Finite-CC-PMSM-v0", motor=dict(motor_initializer=dict(random_init="uniform", interval=[[-100, 100], [-100, 100], [-3.0, 3.0]])))',
    "tau_finite_dc": 'gem.make("Finite-CC-PermExDc-v0", tau=2e-5, converter=dict(interlocking_time=1e-6))',
    "omega_load_instance_sc": 'gem.make("Cont-SC-SynRM-v0", load=ps.PolynomialStaticLoad(load_parameter=dict(a=0.01, b=0.01, c=0.0, j_load=1e-3), limits=dict(omega=200.0)))',
    "dq_wrapper_scim": 'gem.make("Cont-CC-SCIM-v0", physical_system_wrappers=[psw.FluxObserver(), psw.DqToAbcActionProcessor.make("SCIM")])',
    "cossin_remove": 'gem.make("Cont-SC-PMSM-v0", physical_system_wrappers=[psw.CosSinProcessor(angle="epsilon", remove_angle=True)])',
    "dead_time_finite": 'gem.make("Finite-CC-SynRM-v0", physical_system_wrappers=[psw.DeadTimeProcessor(steps=3)])',
    "load_initializer_uniform": 'gem.make("Cont-SC-PermExDc-v0", load=dict(load_initializer=dict(random_init="uniform", interval=[[20.0, 60.0]])))',
}


# every registered id with its defaults
for _a in ("Cont", "Finite"):
    for _c in ("CC", "TC", "SC"):
        for _m in ("PermExDc", "SeriesDc", "ShuntDc", "ExtExDc", "PMSM", "SynRM", "EESM", "SCIM", "DFIM"):
            CASES[f"default_{_a}-{_c}-{_m}"] = f'gem.make("{_a}-{_c}-{_m}-v0")'


def summary(env):
    ps_ = env.physical_system.unwrapped
    sp = env.action_space
    rgen = env.reference_generator
    subs = getattr(rgen, "_sub_generators", [rgen])
    margins = []
    for g in subs:
        for h in getattr(g, "_sub_generators", [g]):
            m = getattr(h, "_limit_margin", None)
            margins.append(None if m is None else [float(v) for v in np.ravel(m)])
    cons = []
    for c in env.constraint_monitor.constraints:
        names = getattr(c, "_states", None)
        if names is None:
            names = list(np.asarray(env.physical_system.state_names)[np.asarray(c._observed_states, dtype=bool)])
        cons.append([type(c).__name__, sorted(str(s) for s in names)])
    return dict(
        env_class=type(env.unwrapped).__name__, state_names=list(env.state_names), reference_names=list(rgen.reference_names),
        limits=[float(v) for v in env.limits], nominal_state=[float(v) for v in env.nominal_state], tau=float(ps_.tau),
        state_low=[float(v) for v in env.observation_space.spaces[0].low], state_high=[float(v) for v in env.observation_space.spaces[0].high],
        ref_low=[float(v) for v in env.observation_space.spaces[1].low], ref_high=[float(v) for v in env.observation_space.spaces[1].high],
        action=[type(sp).__name__, [int(v) for v in np.atleast_1d(getattr(sp, "nvec", getattr(sp, "n", 0)))] if not hasattr(sp, "low")
                else [[float(v) for v in sp.low], [float(v) for v in sp.high]]],
        motor_parameter={k: float(v) for k, v in sorted(ps_.electrical_motor.motor_parameter.items()) if np.ndim(v) == 0},
        j_total=float(ps_.mechanical_load.j_total), u_sup=float(ps_.supply.u_nominal), supply_class=type(ps_.supply).__name__,
        converter_class=type(ps_.converter).__name__, interlocking_time=float(ps_.converter._interlocking_time),
        reward_weights=[float(v) for v in np.asarray(env.reward_function._reward_weights, dtype=float)],
        reward_power=[float(v) for v in np.broadcast_to(np.asarray(env.reward_function._n, dtype=float), (len(env.physical_system.state_names),))],
        reward_bias=float(env.reward_function._bias), violation_reward=float(env.reward_function._violation_reward),
        reward_range=[float(v) for v in env.reward_function.reward_range], constraints=sorted(cons), generator_margins=margins,
    )


def trajectory(env, impl):
    """reset + five steps with fixed actions: the filtered state vectors, the terminated flags and — when every reference generator is a
    ConstReferenceGenerator, i.e. the references are not random — the rewards.  Reference: the env itself (default dopri5 solver unless the
    case names one).  This package: its C-ABI config run by the CPU ORACLE (tests may use it; the kernel is compared with the oracle in
    the `-m gpu` tests) — so the whole chain user kwargs -> host classes -> gemb200_config -> physics is compared number by number.
    Cases with random initial states, random supply phase or state noise have no comparable numbers (different RNG streams): None."""
    sp = env.action_space
    solver = type(env.physical_system.unwrapped._ode_solver).__name__
    if hasattr(sp, "low"):
        shape = np.array([1.0, -0.6, 0.35, 0.8, -0.9, 0.5])[: sp.shape[0]]  # not the same value on every phase (that would be a zero vector)
        actions = [np.clip(v * shape, sp.low, sp.high) for v in (0.3, -0.2, 0.5, -0.7, 0.1)]
        if solver in ("ScipyOdeSolver", "EulerSolver"):
            # solvers with an exact twin in the oracle (its dopri5 restatement / Euler): 300 more steps with seeded random actions, held
            # for 10 steps each so that currents build up and constraints trigger; a terminated episode is followed by a reset on both sides
            rng = np.random.default_rng(11)
            for _ in range(30):
                a = np.clip(rng.uniform(-0.8, 0.8, size=sp.shape), sp.low, sp.high)
                actions += [a] * 10
    elif hasattr(sp, "nvec"):
        actions = [np.array(v[: len(sp.nvec)]) for v in ([1, 1], [2, 0], [0, 1], [3, 2], [1, 0])]
        if solver in ("ScipyOdeSolver", "EulerSolver"):
            rng = np.random.default_rng(12)
            for _ in range(60):
                actions += [np.array([int(rng.integers(0, m)) for m in sp.nvec])] * 5
    else:
        actions = [v % sp.n for v in (1, 2, 0, 5, 3)]
        if solver in ("ScipyOdeSolver", "EulerSolver"):
            rng = np.random.default_rng(12)
            for _ in range(60):
                actions += [int(rng.integers(0, sp.n))] * 5
    if impl == "reference":
        ps_ = env.physical_system.unwrapped
        if getattr(ps_.electrical_motor, "_initializer", {}).get("random_init") or getattr(ps_.mechanical_load, "_initializer", {}).get("random_init"):
            return None
        if type(ps_.supply).__name__ == "AC1PhaseSupply" and not ps_.supply._fixed_phi:
            return None
        chain, w = [], env.physical_system
        while w is not w.unwrapped:
            chain.append(type(w).__name__)
            w = w._physical_system
        if "StateNoiseProcessor" in chain:
            return None
        const_refs = all(type(g).__name__ == "ConstReferenceGenerator" for g in getattr(env.reference_generator, "_sub_generators", [env.reference_generator]))
        (state, _), _ = env.reset(seed=0)
        states, rewards, terms = [np.asarray(state, dtype=float).tolist()], [], []
        for a in actions:
            (state, _), reward, terminated, _, _ = env.step(a)
            states.append(np.asarray(state, dtype=float).tolist())
            rewards.append(float(reward))
            terms.append(bool(terminated))
            if terminated:
                if len(actions) <= 5:
                    break
                (state, _), _ = env.reset()
                states.append(np.asarray(state, dtype=float).tolist())
        return dict(states=states, terminated=terms, rewards=rewards if const_refs else None, solver=solver)
    sys.path.insert(0, HERE.rsplit("/", 1)[0])
    from gym_electric_motor_b200 import _cabi as K
    from oracle.gem_oracle import Oracle

    cfg = env.build_config()
    if cfg.init_random or any(cfg.sop_kind[k] == K.SOP_NOISE for k in range(cfg.n_state_ops)) or (cfg.supply_kind == K.SUPPLY_AC1 and cfg.supply_param[2] == 0.0):
        return None
    cfg.dtype = K.F64
    cfg.n_envs = 1
    if solver == "ScipyOdeSolver":
        # the device runs the scipy wrappers as RK4 x2 (accuracy pinned by the dopri5 goldens); HERE the point is the configuration chain, so
        # the oracle runs its restatement of scipy's dopri5 — the reference's own algorithm, including its dropped-step pathology
        # (DESIGN.md finding 1, which the zero-state SC envs hit) — and the comparison can be tight
        from oracle.gem_oracle import SOLVER_DOPRI5

        cfg.solver_kind, cfg.solver_nsteps = SOLVER_DOPRI5, 1
    ora = Oracle(cfg)
    const_refs = all(cfg.ref_kind[r] == K.REF_CONST for r in range(cfg.n_ref))
    obs, _ = ora.reset()
    states, rewards, terms = [obs[0][env.state_filter].tolist()], [], []
    for a in actions:
        obs, _, rew, term = ora.step(np.asarray(a).reshape(1, -1))
        states.append(obs[0][env.state_filter].tolist())
        rewards.append(float(rew[0]))
        terms.append(bool(term[0]))
        if term[0]:
            if len(actions) <= 5:
                break
            obs, _ = ora.reset()
            states.append(obs[0][env.state_filter].tolist())
    return dict(states=states, terminated=terms, rewards=rewards if const_refs else None, solver=solver)


def main(impl):
    warnings.filterwarnings("ignore")
    sys.dont_write_bytecode = True
    sys.path.insert(0, HERE + "/_shims")
    if impl == "reference":
        sys.path.insert(0, REF + "/src")
        import gym_electric_motor as gem
        from gym_electric_motor.core import ElectricMotorVisualization

        class NoViz(ElectricMotorVisualization):
            pass

        real_make = gem.make
        gem.make = lambda env_id, **kw: real_make(env_id, visualization=NoViz(), **kw)  # keep matplotlib out of it
    else:
        sys.path.insert(0, HERE.rsplit("/", 1)[0])
        import gym_electric_motor_b200 as gem

        gem.install_as_gym_electric_motor()
    out = {}
    for name, src in CASES.items():
        ns = {"gem": gem}
        rec = dict(verdict="ok", summary=None, trajectory=None)
        try:
            exec(PRELUDE, ns)
            env = eval(src, ns)
            rec["summary"] = summary(env)
            rec["trajectory"] = trajectory(env, impl)
        except Exception as e:
            rec["verdict"] = f"{type(e).__name__}: {str(e)[:200]}"
        out[name] = rec
    print(json.dumps(out))


if __name__ == "__main__":
    main(sys.argv[sys.argv.index("--impl") + 1] if "--impl" in sys.argv else "b200")
