"""Developer tool (CPU only): randomised cross-check of the small rows either
side of the transform — spherical conversion, estimateDist2, quantisation-weight
variants — compiled reference == oracle == kernel bodies (host build).
Usage: python tools/fuzz_misc_cpu.py [cases] [seed]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
from pcc_testlib import *  # noqa: E402,F401,F403


def main():
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 100
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    rng = np.random.default_rng(seed)
    bad = 0
    for i in range(cases):
        n = int(rng.integers(1, 6000))
        bits = int(rng.integers(3, 22))
        xyz = rng.integers(-(1 << bits), 1 << bits, size=(n, 3)).astype(np.int32)
        if rng.integers(0, 3) == 0:
            xyz[: n // 3, :2] = rng.integers(-2, 3, size=(n // 3, 2))  # on / next to the axis
        # spherical conversion
        nt = int(rng.choice([1, 2, 3, 16, 64, 128]))
        theta = lidar_lasers(nt, float(rng.uniform(-1.4, -0.05)), float(rng.uniform(0.05, 1.4)))
        origin = tuple(int(x) for x in rng.integers(-1000, 1000, 3))
        r, rb = ref_xyz_to_rpl(origin, theta, xyz)
        o, ob = oracle_xyz_to_rpl(origin, theta, xyz)
        e, eb = emu_xyz_to_rpl(origin, theta, xyz)
        ok = same(r, o) and same(rb, ob) and np.array_equal(e, o) and np.array_equal(eb, ob)
        w = ref_normalised_axes_weights(np.maximum(rb[3:], 1), 0)
        mp = rb[:3] if rng.integers(0, 2) else tuple(int(x) for x in rng.integers(-500, 500, 3))
        rs = ref_offset_and_scale(mp, w, r)
        ok = ok and same(rs, oracle_offset_and_scale(mp, w, o))
        es, _ = emu_xyz_to_rpl(origin, theta, xyz, weight=w, min_pos=mp)
        ok = ok and same(es, rs)
        # estimateDist2 on the Morton-sorted cloud (non-negative coordinates)
        pos = np.abs(xyz)
        _, _, order = sort_cloud(pos, np.zeros((n, 1), dtype=np.int32))
        pos = pos[order]
        period, sr = int(rng.integers(1, 200)), int(rng.integers(1, 300))
        pct = float(rng.choice([0.0, 0.5, 0.85, 0.99]))
        d = ref_estimate_dist2(pos, period, sr, pct)
        ok = ok and oracle_estimate_dist2(pos, period, sr, pct) == d and emu_estimate_dist2(pos, period, sr, pct) == d
        # quantisation-weight variants on a synthetic LoD structure
        m = int(rng.integers(8, 4000))
        preds, npl = synth_predictors(m, int(rng.integers(2, 9)), seed=int(rng.integers(1 << 30)))
        nw = tuple(int(x) for x in rng.integers(0, 600, 3))
        qr = ref_quant_weights_fixed(preds, nw)
        ok = ok and same(qr, oracle_quant_weights_fixed(preds, nw), emu_quant_weights_fixed(preds, npl, nw))
        numpts, ml2 = int(rng.integers(m, 4 * m)), int(rng.integers(0, 3))
        sr_ = ref_quant_weights_scalable(preds, npl, numpts, ml2)
        ok = ok and same(sr_, oracle_quant_weights_scalable(npl, numpts, ml2),
                         emu_quant_weights_scalable(npl, numpts, ml2))
        if not ok:
            bad += 1
            print("MISMATCH case", i, "n", n, "bits", bits, "lasers", nt, "origin", origin, period, sr, pct, nw)
    print(f"{cases} cases, {bad} mismatches (seed {seed})")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
