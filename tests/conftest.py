import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oc():
    """The CPU oracle (test infrastructure)."""
    from oracle import oracle
    oracle.lib()
    return oracle


@pytest.fixture(scope="session")
def ort():
    """The product package; builds libort_b200.so if it is not there yet."""
    import octree_ray_tracing_b200 as pkg
    from octree_ray_tracing_b200 import build
    if not os.path.exists(pkg.LIB_PATH):
        build.build()
    pkg.lib()
    return pkg


@pytest.fixture(scope="session")
def golden():
    def load(name):
        g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
        if "rays_sha256" in g:                  # the reference's outputs are stored; the rays are drawn again from their seed
            from golden.make_golden import golden_rays, rays_sha256
            rays = golden_rays(name)
            assert rays_sha256(rays) == str(g["rays_sha256"]), f"{name}: the rays drawn from the seed are not the ones the reference traced"
            g.update(rays)
        return g
    return load


PRODUCT_VARIANTS = (0, 1, 2, 13)                       # traverse(), FastWalker, persistent lane refill, LeanWalker tiers (default)
EXPERIMENT_VARIANTS = (3, 4, 5, 6, 7, 12, 14, 15, 16, 17, 18, 19)      # csrc/ort_experiments.cuh, only in libort_b200_exp.so


def frame_variants(ort):
    """The frame-kernel variants the loaded library carries: the product's, plus the experiments when the measurement
    build is loaded (ORT_B200_EXPERIMENTS=1, see tests/test_experiments.py)."""
    v = list(PRODUCT_VARIANTS)
    if b"experiments" in ort.lib().ort_version():
        v += list(EXPERIMENT_VARIANTS)
    return tuple(v)


def same_bits(a, b):
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype.itemsize == b.dtype.itemsize and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def assert_same_hits(got, want, what=""):
    """voxel ids and faces bit-exact; t bit-exact too (stricter than north_star's 1e-5 relative)."""
    gv, gf, gt = got[:3]
    wv, wf, wt = want[:3]
    bad_v = np.flatnonzero(np.asarray(gv, np.uint32) != np.asarray(wv, np.uint32))
    assert bad_v.size == 0, f"{what}: {bad_v.size} voxel mismatches, first at ray {bad_v[:5]}"
    bad_f = np.flatnonzero(np.asarray(gf, np.uint8) != np.asarray(wf, np.uint8))
    assert bad_f.size == 0, f"{what}: {bad_f.size} face mismatches, first at ray {bad_f[:5]}"
    gtb = np.ascontiguousarray(gt, np.float32).view(np.uint32)
    wtb = np.ascontiguousarray(wt, np.float32).view(np.uint32)
    bad_t = np.flatnonzero(gtb != wtb)
    assert bad_t.size == 0, f"{what}: {bad_t.size} hit-time mismatches (bitwise), first at ray {bad_t[:5]}"


def degenerate_rays(ort, depth):
    """310 000 rays built to hit every special case of the kernels' fast path: zero and denormal direction components
    (coef = -inf), origins on cell planes -- including coordinates of exactly 1.0f, which mirror to 2.0f on an axis
    travelled in the positive direction and leave [1,2) --, origins outside [1,2)^3, grazing rays, NaN / inf / huge / tiny components."""
    rs = np.random.RandomState(7)
    o, d = ort.harness.random_rays(200_000, seed=11)
    # degenerate directions
    dz = d[:40_000].copy()
    dz[np.arange(40_000), rs.randint(0, 3, 40_000)] = rs.choice(np.array([0.0, -0.0, 1e-42, -1e-42], np.float32), 40_000)
    d2 = d[40_000:60_000].copy()
    d2[:, :2] = 0.0                                              # two degenerate axes
    # on-plane origins: coordinates snapped to multiples of 2^-k
    op = o[:40_000].copy()
    k = rs.randint(1, depth + 1, size=op.shape)
    op = (np.floor((op - 1.0) * (1 << k)) / (1 << k) + 1.0).astype(np.float32)
    # origins outside the cube (FastWalker must hand these to the baseline walk)
    oo = (o[:20_000] + rs.choice(np.array([-1.0, 1.0, 0.0], np.float32), size=(20_000, 3))).astype(np.float32)
    # grazing rays just above the terrain
    og = o[:20_000].copy(); og[:, 2] = 1.0 + 5.0 / 16.0 + 1e-3
    dg = d[:20_000].copy(); dg[:, 2] = -np.abs(dg[:, 2]) * 1e-3
    # NaN (both signs), +-inf, huge and near-denormal components: one or two per direction, one per origin
    special = np.array([np.nan, 0.0, np.inf, -np.inf, 3e38, -3e38, 1e-38, -1e-38], np.float32)
    special[1:2] = np.array([0xFFC00000], np.uint32).view(np.float32)
    n = 10_000
    s1 = d[60_000:70_000].copy(); s1[np.arange(n), rs.randint(0, 3, n)] = rs.choice(special, n)
    s2 = d[70_000:80_000].copy(); k = rs.randint(0, 3, n)
    s2[np.arange(n), k] = rs.choice(special, n); s2[np.arange(n), (k + 1) % 3] = rs.choice(special, n)
    so = o[80_000:90_000].copy(); so[np.arange(n), rs.randint(0, 3, n)] = rs.choice(special, n)
    O = np.concatenate([o, o[:40_000], o[40_000:60_000], op, oo, og, o[60_000:80_000], so])
    D = np.concatenate([d, dz, d2, d[:40_000], d[:20_000], dg, s1, s2, d[80_000:90_000]])
    return O, D
