"""Mint tests/golden/refshader_images.npz (+ refshader.json) from the REFERENCE'S OWN compute shader source.

Needs a reference checkout (RT_REFERENCE=<path> make -C oracle first): every image here is what
RayTracing/Assets/Shaders/compute.glsl itself computes — rewritten syntactically by oracle/glsl2cpp.py,
compiled against the reference's vendored glm, walking the node array the reference's BVH.h built
(oracle/_ref/ref_host) — for the cases of tests/scenes.py::refshader_cases().  The GL driver's elementary
functions (cos, sin, exp, acos, pow) are the spec'd ones of DESIGN.md §4 (REF_SPEC_MATH=1).

The GPU parity tests compare the CUDA path against these files bit for bit, without the oracle in between;
tests/test_refshader_cpu.py keeps the oracle pinned to them as well.

    python tests/golden/make_golden_refshader.py [--big]
"""
import json
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]
import oracle  # noqa: E402
import refshader  # noqa: E402
import scenes  # noqa: E402


def main():
    assert refshader.available(True), "oracle/_ref/libref_shader.so missing: make -C oracle (needs RT_REFERENCE)"
    assert oracle.have_ref_host(), "oracle/_ref/ref_host missing"
    meta, images = {}, {}
    for name, (scene, u) in scenes.refshader_cases().items():
        img = refshader.render(scene, u, spec_math=True)
        images[name] = img
        meta[name] = {"crc": zlib.crc32(img.tobytes()) & 0xffffffff, "shape": list(img.shape),
                      "triangles": int(scene.triangles.size), "unique_values": int(np.unique(img).size)}
        print(name, meta[name])
    np.savez_compressed(os.path.join(HERE, "refshader_images.npz"), **images)
    if "--big" in sys.argv:   # minutes of CPU: the full-size cases, CRC only
        big = {}
        for name, (scene, u) in scenes.refshader_big_cases().items():
            img = refshader.render(scene, u, spec_math=True)
            big[name] = {"crc": zlib.crc32(img.tobytes()) & 0xffffffff, "shape": list(img.shape),
                         "triangles": int(scene.triangles.size),
                         "row_crc": [zlib.crc32(img[y].tobytes()) & 0xffffffff for y in range(img.shape[0])]}
            print(name, big[name]["crc"])
        json.dump(big, open(os.path.join(HERE, "refshader_big.json"), "w"), indent=0, sort_keys=True)
    json.dump(meta, open(os.path.join(HERE, "refshader.json"), "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
