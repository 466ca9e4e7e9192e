"""Generate tests/golden/ref_host/*.npz from the reference's OWN headers compiled for the host
(oracle/_ref/libref_host_*.so, built by `make -C oracle ref_host REF=<checkout of the reference>`).
These pin the oracle's RTO_ARITH_HOST mode: scene, camera, Octree blob (sha256 + counts) and small frames.

    python tests/golden/gen_ref_host.py
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle_py as O  # noqa: E402

DST = os.path.join(ROOT, "tests", "golden", "ref_host")
os.makedirs(DST, exist_ok=True)
CASES = [  # variant, n, nx, ny, ns[, seed_mode]
    ("brute_spl30", 488, 120, 80, 4),
    ("oct_spl30", 488, 120, 80, 4),
    ("oct_spl30", 8000, 120, 80, 2),
    ("oct_spl30", 20000, 60, 40, 1),      # overflows the leaf buckets: exercises the "Leaf nodes full" drops
    ("oct_spl300", 100000, 96, 54, 1),    # 140 undefined sphere slots (SURVEY D3)
    ("oct_spl3000", 1000000, 48, 27, 1),
    ("oct_spl30", 488, 60, 40, 3, O.SEED_UPSTREAM),   # curand_init(1984, pixel_index, 0) (main.cu:90)
]
manifest = {}
devnull = os.open(os.devnull, os.O_WRONLY)
for variant, n, nx, ny, ns, *rest in CASES:
    seed_mode = rest[0] if rest else O.SEED_HEAD
    rh = O.RefHost(variant).create_world(n, 0.1, nx, ny)
    use_octree = variant.startswith("oct")
    spl = int(variant.split("spl")[1])
    entry = {"variant": variant, "n": n, "nx": nx, "ny": ny, "ns": ns, "spl": spl, "use_octree": int(use_octree),
             "spheres_sha256": hashlib.sha256(rh.spheres().tobytes()).hexdigest(),
             "camera_hex": rh.camera().view("<u4").tolist()}
    saved = os.dup(1)
    os.dup2(devnull, 1)            # the reference printf's one line per dropped sphere
    try:
        if use_octree:
            blob = rh.build_octree()
            nodes, leaves, nc, lc = O.split_octree(blob, spl)
            entry.update(octree_sha256=hashlib.sha256(blob.tobytes()).hexdigest(), node_count=nc, leaf_count=lc)
        fb, lin, ctr = rh.render(O.make_params(nx, ny, ns, use_octree, spl, O.ARITH_HOST, seed_mode=seed_mode), want_linear=True)
    finally:
        os.dup2(saved, 1)
        os.close(saved)
    entry["counters"] = {k: ctr[k] for k in ("rays", "sphere_tests", "aabb_tests", "paths")}
    name = f"{variant}_n{n}_{nx}x{ny}x{ns}.npz"
    if seed_mode != O.SEED_HEAD:
        entry["seed_mode"] = seed_mode
        name = name.replace(".npz", "_upseed.npz")
    np.savez_compressed(os.path.join(DST, name), fb=fb, linear=lin)
    manifest[name] = entry
    rh.destroy()
    print(name, entry["counters"])
json.dump(manifest, open(os.path.join(DST, "manifest.json"), "w"), indent=1)
