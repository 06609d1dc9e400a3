"""More random scenes than the test-suite runs (tests/scenes.py::random_scene, seeds from argv range): the frame of
the CUDA path must equal the oracle's bit for bit in both RNG modes.  Random scenes with and without textures exercise
both append policies of k_shade.
usage (GPU box): python tools/fuzz_more.py 20 80"""
import importlib, sys
sys.path.insert(0, '.'); sys.path.insert(0, 'tests')
import numpy as np
rt = importlib.import_module("raytracing2-fork_b200")
import oracle, scenes

lo, hi = int(sys.argv[1]), int(sys.argv[2])
bad = 0
for seed in range(lo, hi):
    scene, u = scenes.random_scene(seed)
    orc = oracle.OracleScene.from_scene(scene)
    for mode in (rt.RNG_REF_PCG, rt.RNG_PHILOX):
        ref = orc.render_frame(u, rng_mode=mode)
        be = rt.Backend(device=0, rng_mode=mode)
        be.upload(scene)
        be.render_frame(u)
        img = be.read_frame()
        be.close()
        if not np.array_equal(img.view(np.uint32), ref.view(np.uint32)):
            bad += 1
            print("MISMATCH seed", seed, "mode", mode, flush=True)
print(f"seeds {lo}..{hi - 1}: {bad} mismatching frames of {(hi - lo) * 2}")
sys.exit(1 if bad else 0)
