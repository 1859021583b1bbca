"""Execute the reference-side binding printed in INTEGRATION.md (section B: a `PhysicalSystem` subclass a reference maintainer would add,
forwarding to libgemb200.so through ctypes): build an SCMLSystem, hand it to the stub, and let it fill `gemb200_config` and call
`gemb200_create`.  Without a GPU the call must get past validation and stop at the CUDA stage.  `--impl reference` builds the system
with the unmodified reference (the checkout harness.REF), `--impl b200` with this package aliased as `gym_electric_motor`.  Prints the
stub's verdict and every value the stub reads from the system as one JSON object."""
import json, re, sys, warnings
warnings.filterwarnings("ignore"); sys.dont_write_bytecode=True
HERE = __file__.rsplit("/", 2)[0]
impl = sys.argv[sys.argv.index("--impl") + 1] if "--impl" in sys.argv else "b200"
sys.path.insert(0, HERE + "/_shims"); sys.path.insert(0, HERE.rsplit("/", 1)[0])
if impl == "reference":
    from harness import REF
    sys.path.insert(0, REF + "/src")
    import gym_electric_motor as gem
    from gym_electric_motor.core import ElectricMotorVisualization
    class NoViz(ElectricMotorVisualization): pass
    env = gem.make("Cont-CC-PMSM-v0", visualization=NoViz())
else:
    import gym_electric_motor_b200 as gemb
    gemb.install_as_gym_electric_motor()
    import gym_electric_motor as gem
    # the stub would live in the reference tree, which keeps the PhysicalSystem base class in core.py; this package keeps it with the systems
    gem.core.PhysicalSystem = gem.physical_systems.PhysicalSystem
    env = gem.make("Cont-CC-PMSM-v0")
md = open(HERE.rsplit("/", 1)[0] + "/INTEGRATION.md").read()
code = re.search(r"```python\n(# gym_electric_motor/physical_systems/b200_system.py.*?)```", md, re.S).group(1)
ns = {}
exec(compile(code, "integration_stub", "exec"), ns)
ps = env.physical_system.unwrapped
mp = ps.electrical_motor.motor_parameter
reads = dict(motor=type(ps.electrical_motor).__name__, motor_parameter=[float(mp.get(k, 0.0)) for k in ("p", "r_s", "l_d", "l_q", "psi_p", "j_rotor")],
             tau=float(ps.tau), u_sup=float(ps.supply.u_nominal), limits=[float(v) for v in ps.limits], nominal_state=[float(v) for v in ps.nominal_state],
             state_names=list(ps.state_names), omega_fixed=float(getattr(ps.mechanical_load, "omega_fixed", 0.0)),
             action_space=[[float(v) for v in ps.action_space.low], [float(v) for v in ps.action_space.high]])
try:
    sys_ = ns["B200SCMLSystem"](ps, num_envs=16)
    verdict = "created (GPU present)"
except Exception as e:
    verdict = f"{type(e).__name__} {str(e)[:200]}"
print(json.dumps(dict(verdict=verdict, reads=reads)))
