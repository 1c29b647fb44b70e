"""Generate the committed fixtures under tests/golden/.

  python tests/golden/make_golden.py maps
      (build container only: needs /root/reference and cv2)  Exports the five
      bundled PNG maps as uint8 occupancy grids with the reference's own calls
      (src/mdp/path_planning_2d.cu:191-197: imread GRAYSCALE, threshold 250
      BINARY_INV) into tests/golden/maps/<name>.npy.

  python tests/golden/make_golden.py ref [outdir]
      (GPU box: needs oracle/_ref/libpp2d_ref_mdp.so, never reads
      /root/reference)  Runs the UNMODIFIED reference CUDA kernels on every
      bundled map and on small synthetic maps and stores J, action, sweep
      count, per-batch residuals (and the model tables for the small maps)
      as <outdir>/ref_<name>.npz.  The files committed in tests/golden/ were
      produced this way on a B200 (see DESIGN.md "Oracle pin").

  python tests/golden/make_golden.py pi [outdir]
      (GPU box)  policyIteration() with the reference's own kernels ->
      pi_ref_<name>.npz.

  python tests/golden/make_golden.py pomdp [outdir]
      (GPU box)  Reference POMDP kernels: tables, Bayes updates, FIB sweeps,
      cuRAND uniforms, forward sampling -> pomdp_<name>.npz.

  python tests/golden/make_golden.py sim [outdir]
      (build container: CPU only)  The three filter methods of the reference's
      dummy_simulator, compiled from its own source lines (oracle/Makefile:
      ref_sim), on the scenarios of tests/sim_oracle_py.py -> sim_<name>.npz.

  python tests/golden/make_golden.py tree [outdir]
      (GPU box)  The reference's own QV-tree host code (SearchTree, VNode,
      QNode, evaluateFibCpu, evaluatePbviCpu) -> tree_<case>.npz.

  python tests/golden/make_golden.py live_cases [outdir]
      Records of the cases that only the live reference tests used to run,
      so that a checkout without oracle/_ref still compares against them:
      ref_rand_512x384.npz (test_reference_pin_gpu random_512),
      bench_ref_<h>x<w>.npz (test_mdp_gpu, the benchmarked sizes solved to
      convergence: sweeps, residuals, CRC-32 of every J and action row),
      kernels_ref_syn_23x31.npz (test_pomdp_gpu: model tables, Bayes updates,
      FIB) and, where a GPU is present, pbvi_ref_map_5x5_g0.7_n25.npz
      (test_pbvi_gpu).  They are computed without the reference: by the CPU
      restatements (oracle/) and, for PBVI, by the library with its cuBLAS
      checker.  With these library and oracle sources the live tests passed
      against the reference on a B200 on exactly these inputs, asserting
      bit-for-bit equality, so the records hold the reference's bits.
"""
import ctypes
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402


def make_maps():
    import cv2
    src = "/root/reference/path_planning_2d/maps"
    os.makedirs(os.path.join(HERE, "maps"), exist_ok=True)
    for name in cases.BUNDLED:
        img = cv2.imread(os.path.join(src, name + ".png"), cv2.IMREAD_GRAYSCALE)
        _, grid = cv2.threshold(img, 250.0, 1.0, cv2.THRESH_BINARY_INV)
        grid = np.ascontiguousarray(grid, dtype=np.uint8)
        np.save(os.path.join(HERE, "maps", name + ".npy"), grid)
        print(name, grid.shape, int(grid.sum()), "occupied")
        # PNG fixtures for the C++ map loader (our own encodings of the grids,
        # not copies of the reference files): gray, and RGB with near-threshold
        # colours to exercise the BGR->gray weights.
        gray = np.where(grid == 1, 0, 255).astype(np.uint8)
        rng = np.random.default_rng(len(name))
        noisy = gray.copy()
        sel = rng.random(gray.shape) < 0.3
        noisy[sel] = rng.integers(240, 256, size=int(sel.sum()))
        cv2.imwrite(os.path.join(HERE, "maps", name + "_gray.png"), noisy)
        rgb = np.stack([noisy] * 3, -1).astype(np.int32)
        rgb += rng.integers(-4, 5, size=rgb.shape)
        cv2.imwrite(os.path.join(HERE, "maps", name + "_rgb.png"),
                    np.clip(rgb, 0, 255).astype(np.uint8))


def ref_lib():
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libpp2d_ref_mdp.so"))
    vp, u32 = ctypes.c_void_p, ctypes.c_uint32
    lib.ref_mdp_solve.restype = ctypes.c_int
    lib.ref_mdp_solve.argtypes = [u32, u32, vp, u32, u32, ctypes.c_float, vp,
                                  vp, vp, ctypes.c_int]
    lib.ref_mdp_tables.restype = ctypes.c_int
    lib.ref_mdp_tables.argtypes = [u32, u32, vp, u32, u32, vp, vp]
    lib.ref_mdp_time_sweeps.restype = ctypes.c_int
    lib.ref_mdp_time_sweeps.argtypes = [u32, u32, vp, u32, u32, ctypes.c_float,
                                        ctypes.c_int, ctypes.c_int,
                                        ctypes.POINTER(ctypes.c_float)]
    return lib


def ref_solve(lib, grid, goal, gamma, max_batches=0):
    h, w = grid.shape
    J = np.zeros(h * w, np.float32)
    A = np.zeros(h * w, np.uint8)
    res = np.zeros(256, np.float64)
    n = lib.ref_mdp_solve(h, w, grid.ctypes.data, goal[0], goal[1], gamma,
                          J.ctypes.data, A.ctypes.data, res.ctypes.data,
                          max_batches)
    return J.reshape(h, w), A.reshape(h, w), n, res[:n // 100].copy()


def ref_tables(lib, grid, goal):
    h, w = grid.shape
    tp = np.zeros(h * w * 81, np.float32)
    sc = np.zeros(h * w * 9, np.float32)
    lib.ref_mdp_tables(h, w, grid.ctypes.data, goal[0], goal[1],
                       tp.ctypes.data, sc.ctypes.data)
    return tp.reshape(h * w, 9, 9), sc.reshape(h * w, 9)


def golden_cases():
    """(name, grid, goal, gamma, max_batches, with_tables)"""
    out = []
    for name, (goal, _start) in cases.BUNDLED.items():
        out.append((name, cases.load_bundled(name), goal, cases.GAMMA, 0, True))
    # synthetic: ragged sizes, other discount factors, one batch only
    for i, (h, w, p, g) in enumerate([(37, 53, 0.2, 0.95), (64, 130, 0.35, 0.9),
                                      (129, 31, 0.1, 0.99), (1, 17, 0.2, 0.95),
                                      (23, 1, 0.2, 0.95), (2, 2, 0.0, 0.5)]):
        grid, goal = cases.synthetic_map(h, w, p, seed=100 + i)
        out.append((f"syn{i}_{h}x{w}", grid, goal, g, 1, h * w <= 4096))
    return out


def make_ref(outdir):
    os.makedirs(outdir, exist_ok=True)
    lib = ref_lib()
    for name, grid, goal, gamma, max_batches, with_tables in golden_cases():
        J, A, n, res = ref_solve(lib, grid, goal, gamma, max_batches)
        data = dict(grid=grid, goal=np.array(goal), gamma=np.float32(gamma),
                    J=J, action=A, sweeps=np.int32(n), residuals=res)
        if with_tables:
            tp, sc = ref_tables(lib, grid, goal)
            data.update(trans_prob=tp, stage_cost=sc)
        np.savez_compressed(os.path.join(outdir, f"ref_{name}.npz"), **data)
        print(name, grid.shape, "sweeps", n, "residuals", res)


def make_pi(outdir):
    """policyIteration() of the reference (dead code there) with its own kernels
    cudaOneStepPolicyEvaluation / cudaPolicyImprovment (oracle/_ref, GPU box)."""
    os.makedirs(outdir, exist_ok=True)
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libpp2d_ref_mdp.so"))
    vp, u32 = ctypes.c_void_p, ctypes.c_uint32
    lib.ref_mdp_policy_iteration.restype = ctypes.c_int
    lib.ref_mdp_policy_iteration.argtypes = [u32, u32, vp, u32, u32, ctypes.c_float, vp, vp,
                                             vp, vp, ctypes.c_int]
    todo = [(name, cases.load_bundled(name), goal) for name, (goal, _) in cases.BUNDLED.items()]
    for h, w, seed in [(37, 53, 1), (64, 130, 2), (1, 17, 3), (23, 1, 4), (2, 2, 5)]:
        grid, goal = cases.synthetic_map(h, w, 0.25, seed=seed)
        todo.append((f"syn{seed}_{h}x{w}", grid, goal))
    for name, grid, goal in todo:
        h, w = grid.shape
        J = np.zeros(h * w, np.float32)
        A = np.zeros(h * w, np.uint8)
        res = np.zeros(4096, np.float64)
        chg = np.zeros(4096, np.uint32)
        n = lib.ref_mdp_policy_iteration(h, w, grid.ctypes.data, goal[0], goal[1],
                                         cases.GAMMA, J.ctypes.data, A.ctypes.data,
                                         res.ctypes.data, chg.ctypes.data, 0)
        np.savez_compressed(os.path.join(outdir, f"pi_ref_{name}.npz"), grid=grid,
                            goal=np.array(goal), gamma=np.float32(cases.GAMMA),
                            J=J.reshape(h, w), action=A.reshape(h, w), sweeps=np.int32(n),
                            residuals=res[:n // 50], changed=chg[:n // 50])
        print(name, grid.shape, "evaluation sweeps", n, "rounds", n // 50)


def make_pomdp(outdir):
    """POMDP half: outputs of the reference kernels (oracle/_ref, GPU box)."""
    import pomdp_oracle_py as po
    os.makedirs(outdir, exist_ok=True)
    R = po.ref()
    un = np.zeros(100, np.float32)
    R.ref_pomdp_uniforms(50, un.ctypes.data)
    np.save(os.path.join(outdir, "curand_xorwow_1234.npy"), un)
    print("uniforms", un[:4])
    rng = np.random.default_rng(5)
    for name, goal in [("map_3x3", (1, 1)), ("map_10x10", (8, 7)),
                       ("sparse_map_100x40", (95, 34))]:
        grid = cases.load_bundled(name)
        h, w = grid.shape
        hw = h * w
        tp = np.zeros(hw * 81, np.float32); mp = np.zeros(hw * 16, np.float32)
        sr = np.zeros(hw * 9, np.float32)
        R.ref_pomdp_model(h, w, grid.ctypes.data, goal[0], goal[1], tp.ctypes.data,
                          mp.ctypes.data, sr.ctypes.data)
        # beliefs: uniform over free cells, and a product of tiny numbers that
        # reaches the subnormal range (exercises flush-to-zero)
        b0 = ((1 - grid.astype(np.float32)) / (1 - grid.astype(np.float32)).sum()).reshape(-1)
        b1 = (rng.random(hw, dtype=np.float32) ** 24 * 1e-30).astype(np.float32)
        b1[rng.integers(hw, size=hw // 4)] = 0
        us = np.array([0, 1, 2, 3, 4, 5, 6, 7, 8, 2, 7], np.uint8)
        zs = np.array([0, 15, 3, 5, 9, 6, 10, 12, 1, 7, 14], np.uint8)
        outs = {}
        for tag, b in (("uniform", b0), ("tiny", b1)):
            o = np.zeros((len(us), hw), np.float32)
            R.ref_pomdp_bayes(h, w, grid.ctypes.data, goal[0], goal[1], b.ctypes.data,
                              len(us), us.ctypes.data, zs.ctypes.data, o.ctypes.data)
            outs["bayes_" + tag] = o
        fib = np.zeros(hw * 9, np.float32)
        n_fib = R.ref_pomdp_fib(h, w, grid.ctypes.data, goal[0], goal[1], cases.GAMMA,
                                fib.ctypes.data, 20)
        samples = rng.integers(hw, size=50).astype(np.uint32)
        # only free cells are valid state samples
        free = np.flatnonzero(grid.reshape(-1) == 0)
        samples = free[rng.integers(len(free), size=50)].astype(np.uint32)
        obs = np.zeros((9, 50), np.uint8)
        for a in range(9):
            R.ref_pomdp_forward_sampling(h, w, grid.ctypes.data, goal[0], goal[1], 50,
                                         samples.ctypes.data, a, obs[a].ctypes.data)
        data = dict(grid=grid, goal=np.array(goal), b_uniform=b0, b_tiny=b1, us=us,
                    zs=zs, fib=fib.reshape(hw, 9), fib_sweeps=np.int32(n_fib),
                    samples=samples, obs=obs, meas_prob=mp.reshape(hw, 16),
                    stage_reward=sr.reshape(hw, 9), **outs)
        if hw <= 4096:
            data["trans_prob"] = tp.reshape(hw, 9, 9)
        np.savez_compressed(os.path.join(outdir, f"pomdp_{name}.npz"), **data)
        print(name, "fib sweeps", n_fib, "obs sample", obs[0][:8])


def make_tree(outdir, only=None):
    """QV-tree half: the reference's own SearchTree / VNode / QNode host code
    (oracle/_ref/libpp2d_ref_pomdp_full.so: four unmodified translation units)
    run on a GPU box through the scenario of tests/tree_scenario.py; one
    process per case because the reference keeps its state in globals."""
    import subprocess
    import tree_scenario as ts
    os.makedirs(outdir, exist_ok=True)
    if only is not None:
        out = ts.run_reference_case(only)
        np.savez_compressed(os.path.join(outdir, f"tree_{only}.npz"), **out)
        print(only, "nodes", [int(v.shape[0]) for k, v in out.items() if "dump" in k])
        return
    for case in ts.CASES:
        subprocess.run([sys.executable, os.path.abspath(__file__), "tree", outdir, case],
                       check=True)


# the benchmarked grids of test_mdp_gpu: (rows, cols), goal; synthetic, 20 %, seed 12345
BENCH_SIZES = [((4096, 4096), (2048, 2048)), ((1536, 16384), (8192, 700))]


def crc_rows(a):
    """CRC-32 of every row's bytes."""
    a = np.ascontiguousarray(a)
    return np.array([zlib.crc32(r.tobytes()) for r in a], np.uint32)


def pomdp_live_case():
    """Inputs of test_pomdp_gpu's live kernel pin: grid, goal, belief, actions,
    observations, FIB sweep cap."""
    grid, goal = cases.synthetic_map(23, 31, 0.3, seed=4)
    b = (np.random.default_rng(0).random(grid.size, dtype=np.float32) ** 18
         * 1e-30).astype(np.float32)
    us = np.arange(9, dtype=np.uint8)
    zs = (np.arange(9) * 7 % 16).astype(np.uint8)
    return grid, goal, b, us, zs, 30


def make_live_cases(outdir):
    import oracle_py
    import pomdp_oracle_py as po
    os.makedirs(outdir, exist_ok=True)
    grid, goal = cases.synthetic_map(512, 384, 0.2, seed=99)
    J, A, n, res = oracle_py.value_iteration(grid, goal, cases.GAMMA, 1)
    np.savez_compressed(os.path.join(outdir, "ref_rand_512x384.npz"), grid=grid,
                        goal=np.array(goal), gamma=np.float32(cases.GAMMA), J=J, action=A,
                        sweeps=np.int32(n), residuals=res)
    print("rand_512x384 sweeps", n)
    grid, goal, b, us, zs, cap = pomdp_live_case()
    m = po.Model(grid, goal)
    fib, n_fib = m.fib(cases.GAMMA, cap)
    np.savez_compressed(os.path.join(outdir, "kernels_ref_syn_23x31.npz"),
                        trans_prob=m.tp, meas_prob=m.mp, stage_reward=m.sr,
                        bayes=np.stack([m.bayes(b, int(u), int(z))[0] for u, z in zip(us, zs)]),
                        fib=np.ascontiguousarray(fib).reshape(-1), fib_sweeps=np.int32(n_fib))
    print("syn_23x31 fib sweeps", n_fib)
    for (h, w), goal in BENCH_SIZES:
        grid, goal = cases.synthetic_map(h, w, 0.20, seed=12345, goal=goal)
        J, A, n, res = oracle_py.value_iteration(grid, goal, cases.GAMMA)
        np.savez_compressed(os.path.join(outdir, f"bench_ref_{h}x{w}.npz"),
                            goal=np.array(goal), sweeps=np.int32(n), residuals=res,
                            J_crc=crc_rows(J.view(np.uint32)), action_crc=crc_rows(A))
        print(f"bench {h}x{w} sweeps", n, "residuals", res[-2:])
    try:
        import torch
        gpu = torch.cuda.is_available()
    except ImportError:
        gpu = False
    if gpu:
        make_pbvi_5x5(outdir)


def make_pbvi_5x5(outdir):
    """pbvi_ref_*.npz layout of tools/ref_offline.py for map_5x5, goal (3, 2),
    gamma 0.7, 25 beliefs, rand_seed 1: the library with its cuBLAS checker."""
    os.environ["PP2D_PBVI_CUBLAS"] = "1"
    sys.path.insert(0, ROOT)
    from path_planning_2d_b200 import PomdpPathPlanning2d
    grid, goal, gamma, n = cases.load_bundled("map_5x5"), (3, 2), 0.7, 25
    free = 1.0 - grid.astype(np.float32).reshape(-1)
    s = np.float32(0)
    for v in free:                    # src/pomdp/path_planning_2d.cu:100-107
        s = np.float32(s + v)
    b0 = (free / s).astype(np.float32)
    with PomdpPathPlanning2d(grid, goal, gamma) as p:
        fib, fa, _ = p.fastInformedBound()
        bs, al, ac = p.pointBasedValueIteration(b0, n, rand_seed=1)
    np.savez_compressed(os.path.join(outdir, "pbvi_ref_map_5x5_g0.7_n25.npz"), grid=grid,
                        goal=np.array(goal), gamma=np.float32(gamma), b0=b0, fib=fib,
                        fib_actions=fa, belief_set=bs, pbvi=al, pbvi_actions=ac)
    print("pbvi map_5x5", bs.shape)


if __name__ == "__main__":
    if len(sys.argv) >= 2 and sys.argv[1] == "live_cases":
        make_live_cases(sys.argv[2] if len(sys.argv) > 2 else HERE)
    elif len(sys.argv) >= 2 and sys.argv[1] == "pi":
        make_pi(sys.argv[2] if len(sys.argv) > 2 else
                os.path.join(ROOT, "gpurun_out", "golden_ref"))
    elif len(sys.argv) >= 2 and sys.argv[1] == "tree":
        make_tree(sys.argv[2] if len(sys.argv) > 2 else
                  os.path.join(ROOT, "gpurun_out", "golden_ref"),
                  sys.argv[3] if len(sys.argv) > 3 else None)
    elif len(sys.argv) >= 2 and sys.argv[1] == "tree_files":
        # tree_files <outdir> <case>: the scenario on the reference started
        # from its own text checkpoint written into <outdir>/data
        import tree_scenario as ts
        os.makedirs(os.path.join(sys.argv[2], "data"), exist_ok=True)
        out = ts.run_reference_case(sys.argv[3], os.path.join(sys.argv[2], "data"))
        np.savez_compressed(os.path.join(sys.argv[2], f"tree_files_{sys.argv[3]}.npz"), **out)
    elif len(sys.argv) >= 2 and sys.argv[1] == "sim":
        # sim [outdir]: the reference's own filter methods (oracle/_ref/
        # libpp2d_ref_sim.so, CPU only -- runs in the build container) on the
        # scenarios of tests/sim_oracle_py.py -> sim_<name>.npz
        import sim_oracle_py as so
        outdir = sys.argv[2] if len(sys.argv) > 2 else HERE
        for name in so.SCENARIOS:
            out = so.run_scenario(name, "ref")
            data = {"crc": so.crc_rows(out), "last": out[:, -1]}
            if out.shape[2] <= 1000:            # small maps: every intermediate belief
                data["beliefs"] = out
            np.savez_compressed(os.path.join(outdir, f"sim_{name}.npz"), **data)
            print(name, out.shape, "NaNs:", int(np.isnan(out).sum()))
    elif len(sys.argv) >= 2 and sys.argv[1] == "maps":
        make_maps()
    elif len(sys.argv) >= 2 and sys.argv[1] == "pomdp":
        make_pomdp(sys.argv[2] if len(sys.argv) > 2 else
                   os.path.join(ROOT, "gpurun_out", "golden_ref"))
    elif len(sys.argv) >= 2 and sys.argv[1] == "ref":
        make_ref(sys.argv[2] if len(sys.argv) > 2 else
                 os.path.join(ROOT, "gpurun_out", "golden_ref"))
    else:
        print(__doc__)
