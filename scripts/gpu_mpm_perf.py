"""MPM timing on the GPU box (BASELINE config 3: 100k particles, 64^3 grid): the default scene, the same without BCs, and
(mode "full") a sand scene and 1M particles on 128^3 (the round-1 four-kernel path the fused one replaced measured 46.6 us on
the same box, profiles/r02_mpm_fused_first_perf.log). Usage: python scripts/gpu_mpm_perf.py [substeps] [full|quick]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from pixie_b200.synthetic import synthetic_scene
from pixie_b200.mpm_solver_warp import MPM_Simulator_WARP

DEV = "cuda:0"


def make(n=100_000, ng=64, materials=(0,), bcs=True):
    sc = synthetic_scene(n, ng, seed=0, materials=materials)
    s = MPM_Simulator_WARP(10)
    s.load_initial_data_from_torch(torch.from_numpy(sc["x"]).to(DEV), torch.from_numpy(sc["vol"]).to(DEV), None, n_grid=ng, grid_lim=2.0)
    s.set_parameters_dict({"material": "jelly", "g": [0.0, 0.0, -9.8], "density": 1000.0, "E": 1e5, "nu": 0.3, "yield_stress": 2e3,
                           "grid_v_damping_scale": 0.9999, "rpic_damping": 0.0, "friction_angle": 30.0, "hardening": 1, "xi": 0.1,
                           "softening": 0.1, "plastic_viscosity": 10.0, "bulk_modulus": 1e5})
    s.mpm_model.E = torch.from_numpy(sc["E"]).to(DEV); s.mpm_model.nu = torch.from_numpy(sc["nu"]).to(DEV)
    s.mpm_state.particle_material = torch.from_numpy(sc["material"]).to(DEV)
    s.reset_densities_and_update_masses(torch.from_numpy(sc["density"]).to(DEV))
    s.import_particle_v_from_torch(torch.from_numpy(sc["v"]).to(DEV)); s.finalize_mu_lam()
    if bcs:
        s.add_bounding_box()
        s.set_velocity_on_cuboid(point=[1.0, 1.0, 0.62], size=[0.51, 0.51, 0.04], velocity=[0, 0, 0])
        s.add_impulse_on_particles(force=[0.05, 0.0, -0.02], dt=1e-4, point=[1.0, 1.0, 1.2], size=[0.2, 0.2, 0.1], num_dt=20, start_time=0.0)
    return s


def time_it(tag, steps, **kw):
    s = make(**kw)
    s.p2g2p_n(100, 1e-4); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e9
    for _ in range(3):
        e0.record(); s.p2g2p_n(steps, 1e-4); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / steps * 1e3)
    x = s.mpm_state.particle_x.numpy()
    print(f"{tag:32s} {best:7.2f} us/substep  {kw.get('n', 100_000) / best * 1e6:.3e} particle-steps/s  x in [{x.min():.3f},{x.max():.3f}] finite={np.isfinite(x).all()}", flush=True)
    return best


if __name__ == "__main__":
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
    mode = sys.argv[2] if len(sys.argv) > 2 else "full"
    time_it("fused", steps)
    time_it("fused, no BCs", steps, bcs=False)
    if mode == "full":
        time_it("fused, sand", steps, materials=(2,))
        time_it("fused, 1M / 128^3", 200, n=1_000_000, ng=128)
