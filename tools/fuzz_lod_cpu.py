"""Developer tool (CPU only): randomised cross-check of the level-of-detail
build over its parameter space — compiled reference == oracle == kernel bodies
(host build) — on small random clouds, followed by the lifting coder chain
(oracle vs kernel bodies).  Usage: python tools/fuzz_lod_cpu.py [cases] [seed]"""
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
        kind = rng.integers(0, 3)
        n = int(rng.integers(1, 5000))
        if kind == 0:
            xyz, attrs = cloud_shell(n, bits=int(rng.integers(4, 11)), seed=int(rng.integers(1 << 30)),
                                     dups=bool(rng.integers(0, 2)))
        elif kind == 1:
            xyz, attrs = cloud_lidar(max(n, 50), seed=int(rng.integers(1 << 30)))
        else:
            xyz, attrs = cloud_random(n, int(rng.integers(2, 22)), seed=int(rng.integers(1 << 30)),
                                      dup_frac=float(rng.choice([0.0, 0.2])))
        levels = int(rng.integers(1, 14))
        lifting = bool(rng.integers(0, 2))
        kw = dict(levels=levels, decimation=int(rng.integers(0, 3)), period=int(rng.integers(2, 9)),
                  dist2=int(rng.integers(0, 4)), k=int(rng.integers(1, 4)),
                  inter_range=int(rng.choice([1, 8, 128, 1100000])),
                  distribution=int(rng.integers(0, 2)),
                  bias=tuple(int(x) for x in rng.integers(1, 4, 3)))
        if not lifting:  # predicting transform: intra-LoD prediction and blending allowed
            kw.update(intra_range=int(rng.choice([0, 4, 128])), skip_layers=int(rng.integers(0, levels + 1)),
                      blending=int(rng.integers(0, 2)))
        lp = make_lod_params(**kw)
        rp, ri, rn = ref_lod_build(lp, xyz)
        op, oi, on = oracle_lod_build(lp, xyz)
        ep, ei, en = emu_lod_build(lp, xyz)
        ok = (same(rn, on) and same(ri, oi) and same(rp, op)
              and np.array_equal(en, on) and np.array_equal(ei, oi) and np.array_equal(ep, op))
        if ok and lifting and len(xyz) > 1:
            a = int(rng.choice([1, 3]))
            at = attrs[:, :a].copy()
            lcp = int(rng.integers(0, 2))
            qs = make_qpset(qp=int(rng.integers(4, 52)), chroma_offset=int(rng.integers(-4, 5)) if a == 3 else 0,
                            fixed_point_qp_offset=24)
            ov, orr, ol = oracle_lift_encode(lp, qs, lcp, xyz, at)
            ev, er, el = emu_attr_lift(1, lp, qs, lcp, xyz, at)
            ok = np.array_equal(ev, ov) and np.array_equal(er, orr) and (not (a == 3 and lcp) or np.array_equal(el, ol))
            if ok:  # the reference's own lifting encoder bodies
                rv, rrec, rl = ref_lift_encode(lp, qs, lcp, xyz, at)
                ok = same(rv, ov) and same(rrec, orr) and (not (a == 3 and lcp) or same(rl, ol))
        if not ok:
            bad += 1
            print("MISMATCH case", i, "n", len(xyz), kw, "lifting", lifting)
    print(f"{cases} cases, {bad} mismatches (seed {seed})")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
