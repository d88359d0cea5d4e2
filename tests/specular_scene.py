"""A specular-dominated scene for the powf tests (tests/test_powf_glibc.py, tests/test_gpu_specular.py).

The synthetic soup with shading normals and spheres, but with high ks and low kd everywhere except on the lights, and
one Ns per geometry / sphere taken in turn from NS: integer, fractional, zero and large exponents, and the ones the
reference's model files use (1, 10, 200, 1000, 1024).  With 4 lights, nearly every lit pixel evaluates powf four
times, so a frame holds tens of thousands of (dot(N,H), Ns) pairs.
"""
import numpy as np

NS = (10.0, 77.7, 200.0, 1000.0, 1024.0, 4096.0, 0.0, 0.5, 1.0, 3.0)  # the floor and back wall get the first
N_LIGHTS = 4
EYE, LOOK = (0, 1, 3), (0, 1, 0)
SEED = 11


def specular_scene(n_tris=1500, n_geoms=25, n_spheres=40, seed=SEED):
    from esctp1raytracer_b200 import scenes

    s = scenes.soup_scene(n_tris, n_geoms, N_LIGHTS, seed=seed, edge=(0.03, 0.12), specular=True, with_normals=True,
                          n_spheres=n_spheres)
    rng = np.random.default_rng(seed + 1)
    lights = set(int(g) for g in s.light_geom)
    k = 0
    for mats, rows in ((s.geom_material, [g for g in range(s.n_geoms) if g not in lights]),
                       (s.sphere_material, list(range(len(s.sphere_material))))):
        for g in rows:
            mats[g, 3:6] = rng.uniform(0.0, 0.1, 3)   # kd
            mats[g, 6:9] = rng.uniform(0.6, 1.0, 3)   # ks
            mats[g, 12] = NS[k % len(NS)]
            k += 1
    return s
