"""Generate the committed golden vectors from the UNMODIFIED reference.

Needs the compiled reference in oracle/_ref (`make -C oracle ref liftref
recolourref REF=<reference source tree>`):

    python tests/golden/make_golden.py

Writes tests/golden/raht_golden.npz (inputs + reference outputs for a set of
small clouds x parameter variants), tests/golden/arith_golden.npz
(known-answer vectors of the scalar helpers), the LoD, spherical and symbol
vectors, and tests/golden/reference_tape.npz (what the reference returned to
every ref_* call of the suite's comparisons, see pcc_testlib.taped).  The
comparisons read these files only: they need neither the reference sources
nor oracle/_ref."""
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from pcc_testlib import *  # noqa

VARIANTS = {
    "default": dict(),
    "nopred": dict(prediction=0),
    "nosubnode": dict(subnode=0),
    "haar": dict(haar=1),
    "noext": dict(ext=0),
    "range5": dict(search_range=5),
}


LOD_GOLDEN_CASES = [
    dict(levels=8),
    dict(levels=8, distribution=0),
    dict(levels=8, decimation=1),
    dict(levels=8, decimation=2),
    dict(levels=8, decimation=0, skip_layers=0, intra_range=64, inter_range=64, blending=1),
]


def clouds():
    rng = np.random.default_rng(2024)
    out = {}
    xyz, at = cloud_cube(3000, side=20)
    out["cube"] = (xyz, at, None)
    xyz, at = cloud_shell(3000, bits=7, seed=3)
    out["shell"] = (xyz, at, None)
    xyz, at = cloud_shell(3000, bits=6, seed=4, dups=True)
    out["shelldup"] = (xyz, at, None)
    xyz, at = cloud_lidar(3000, seed=2)
    out["lidar"] = (xyz, at[:, :1].copy(), None)
    xyz, at = cloud_random(2000, 21, seed=5, dup_frac=0.1)
    qpo = rng.integers(-5, 6, size=(2000, 2)).astype(np.int32)
    out["sparse21"] = (xyz, at, qpo)
    return out


def main():
    data = {}
    for cname, (xyz, attrs, qpo) in clouds().items():
        mort, a_s, order = sort_cloud(xyz, attrs)
        q = qpo[order] if qpo is not None else None
        data[f"{cname}/xyz"] = xyz
        data[f"{cname}/attrs"] = attrs
        if qpo is not None:
            data[f"{cname}/qpo"] = qpo
        for vname, kw in VARIANTS.items():
            for qp in (16, 34):
                p = make_params(**kw)
                qs = make_qpset(qp=qp)
                rec, coef = ref_raht(1, p, qs, mort, a_s, qpoffs=q)
                rec2, _ = ref_raht(0, p, qs, mort, a_s * 0, coeffs=coef, qpoffs=q)
                assert np.array_equal(rec, rec2)
                data[f"{cname}/{vname}/qp{qp}/coef"] = coef
                data[f"{cname}/{vname}/qp{qp}/rec"] = rec
    np.savez_compressed(os.path.join(HERE, "raht_golden.npz"), **data)

    ref = load_ref()
    rng = np.random.default_rng(99)
    xs = np.concatenate([
        np.arange(0, 5000, dtype=np.uint64),
        rng.integers(0, 1 << 62, size=5000, dtype=np.uint64) >> rng.integers(0, 62, size=5000).astype(np.uint64),
    ])
    isq = np.array([ref.tmc13ref_isqrt(int(x)) for x in xs], dtype=np.uint64)
    irs = np.array([ref.tmc13ref_irsqrt(int(x)) for x in xs], dtype=np.uint64)
    a = rng.integers(-(1 << 45), 1 << 45, size=4000, dtype=np.int64)
    b = rng.integers(-(1 << 17), 1 << 17, size=4000, dtype=np.int64)
    fx = np.array([ref.tmc13ref_fixed_mul(int(x), int(y)) for x, y in zip(a, b)], dtype=np.int64)
    qps = rng.integers(0, 100, size=4000).astype(np.int32)
    qx = rng.integers(-(1 << 30), 1 << 30, size=4000, dtype=np.int64)
    qq = np.array([ref.tmc13ref_quantize(int(q), int(x)) for q, x in zip(qps, qx)], dtype=np.int64)
    qs = np.array([ref.tmc13ref_scale(int(q), int(x)) for q, x in zip(qps, qx)], dtype=np.int64)
    pts = rng.integers(0, 1 << 21, size=(3000, 3)).astype(np.int32)
    mc = np.array([ref.tmc13ref_morton_addr(int(p[0]), int(p[1]), int(p[2])) for p in pts], dtype=np.int64)
    ma = rng.integers(0, 1 << 62, size=3000, dtype=np.uint64)
    mb = np.concatenate([np.full(1500, 0xFFFFFFFFFFFFFFFF, dtype=np.uint64),
                         rng.integers(0, 64, size=1500, dtype=np.uint64)])
    madd = np.array([ref.tmc13ref_morton3d_add(int(x), int(y)) for x, y in zip(ma, mb)], dtype=np.uint64)
    da = rng.integers(-(1 << 40), 1 << 40, size=3000, dtype=np.int64)
    db = rng.integers(1, 1 << 30, size=3000, dtype=np.uint64) >> rng.integers(0, 29, size=3000).astype(np.uint64)
    db = np.maximum(db, 1)
    dv = np.array([ref.tmc13ref_div_approx(int(x), int(y), 0) for x, y in zip(da, db)], dtype=np.int64)
    np.savez_compressed(
        os.path.join(HERE, "arith_golden.npz"), xs=xs, isqrt=isq, irsqrt=irs,
        fa=a, fb=b, fxmul=fx, qps=qps, qx=qx, quant=qq, scale=qs, pts=pts,
        morton=mc, ma=ma, mb=mb, madd=madd, da=da, db=db, divapprox=dv)
    # level-of-detail build (AttributeLods::generate)
    lod = {}
    xyz, _ = cloud_shell(4000, bits=7, seed=3)
    lod["shell/xyz"] = xyz
    xyz2, _ = cloud_random(3000, 21, seed=5, dup_frac=0.1)
    lod["sparse/xyz"] = xyz2
    for cname in ("shell", "sparse"):
        for i, kw in enumerate(LOD_GOLDEN_CASES):
            p, idx, npl = ref_lod_build(make_lod_params(**kw), lod[f"{cname}/xyz"])
            lod[f"{cname}/{i}/preds"] = p
            lod[f"{cname}/{i}/indexes"] = idx
            lod[f"{cname}/{i}/npl"] = npl
    np.savez_compressed(os.path.join(HERE, "lod_golden.npz"), **lod)
    spherical_golden()
    symbols_golden()
    record_reference_tape()
    print("golden vectors written")


# the tests whose ref_* calls the tape serves (the fuzz slices record from
# their subprocesses)
TAPED_TESTS = ["tests/test_oracle_vs_reference.py", "tests/test_recolour.py", "tests/test_fuzz_cpu.py"]


def record_reference_tape():
    """run the comparisons against the compiled reference and record its outputs"""
    root = os.path.dirname(os.path.dirname(HERE))
    if os.path.exists(TAPE_PATH):
        os.remove(TAPE_PATH)
    env = dict(os.environ, PCCB200_RECORD_REFERENCE="1")
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", *TAPED_TESTS],
                          cwd=root, env=env)


SYMBOL_GOLDEN_CASES = [("shell3", 3, 16), ("shell1", 1, 22), ("lidar3", 3, 28), ("lidar1", 1, 10)]


def symbols_golden():
    """the symbol stream the reference's RAHT attribute decoder reads from the
    payload of the reference's own encoder (oracle/_ref/libtmc13_lift.so)"""
    g = {}
    for name, a, qp in SYMBOL_GOLDEN_CASES:
        if name.startswith("shell"):
            xyz, attrs = cloud_shell(5000, bits=7, seed=5, a=a)
        else:
            xyz, attrs = cloud_lidar(5000, seed=5, a=a)
        params, qs = make_params(), make_qpset(qp=qp)
        payload, recon = ref_raht_encode_payload(params, qs, xyz, attrs)
        runs, vals, tail = ref_decode_symbol_stream(payload, len(xyz), a)
        g[f"{name}/xyz"] = xyz
        g[f"{name}/attrs"] = attrs
        g[f"{name}/runs"] = runs
        g[f"{name}/values"] = vals
        g[f"{name}/tail"] = np.int32(tail)
        g[f"{name}/recon"] = recon
        g[f"{name}/payload"] = np.frombuffer(payload, dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, "symbols_golden.npz"), **g)


def spherical_golden():
    """spherical-coordinate conversion (convertXyzToRpl + offsetAndScale of the
    compiled reference, oracle/_ref/libtmc13_lift.so)"""
    g = {}
    xyz, _ = cloud_lidar(6000, seed=9)
    rng = np.random.default_rng(17)
    wide = rng.integers(-(1 << 20), 1 << 20, size=(3000, 3)).astype(np.int32)
    wide[:200, :2] = rng.integers(-3, 4, size=(200, 2))  # around the axis, radius ~0
    cases = [("lidar", xyz, (12, -7, 30), lidar_lasers(64)),
             ("wide", wide, (0, 0, 0), lidar_lasers(16, -0.9, 0.9)),
             ("one_laser", wide[:500], (5, 5, 5), lidar_lasers(1)),
             ("two_lasers", wide[:500], (-9, 2, 0), lidar_lasers(2, -0.2, 0.3))]
    g["names"] = np.array([c[0] for c in cases])
    for name, pts, origin, theta in cases:
        rpl, bbox = ref_xyz_to_rpl(origin, theta, pts)
        w = ref_normalised_axes_weights(np.maximum(bbox[3:], 1))
        g[f"{name}/xyz"] = pts
        g[f"{name}/origin"] = np.array(origin, dtype=np.int32)
        g[f"{name}/theta"] = theta
        g[f"{name}/rpl"] = rpl
        g[f"{name}/bbox"] = bbox
        g[f"{name}/weight"] = np.array(w, dtype=np.int32)
        g[f"{name}/scaled"] = ref_offset_and_scale(bbox[:3], w, rpl)
    np.savez_compressed(os.path.join(HERE, "spherical_golden.npz"), **g)


if __name__ == "__main__":
    main()
