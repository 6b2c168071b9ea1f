"""Developer tool (CPU only): randomised cross-check of the three CPU-side
implementations of the RAHT path over the parameter space —
    compiled reference  ==  oracle (C restatement)  ==  kernel bodies (host build)
on small random clouds.  Usage: python tools/fuzz_cpu.py [cases] [seed]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
from pcc_testlib import *  # noqa: E402,F401,F403


def random_case(rng):
    kind = rng.integers(0, 4)
    n = int(rng.integers(1, 4000))
    a = int(rng.choice([1, 3]))
    if kind == 0:
        xyz, attrs = cloud_shell(n, bits=int(rng.integers(4, 10)), seed=int(rng.integers(1 << 30)), a=a,
                                 dups=bool(rng.integers(0, 2)))
    elif kind == 1:
        xyz, attrs = cloud_lidar(max(n, 50), seed=int(rng.integers(1 << 30)), a=a)
    elif kind == 2:
        xyz, attrs = cloud_random(n, int(rng.integers(2, 21)), seed=int(rng.integers(1 << 30)), a=a,
                                  dup_frac=float(rng.choice([0.0, 0.3])))
    else:
        xyz, attrs = cloud_cube(n, seed=int(rng.integers(1 << 30)), a=a)
    bitdepth = int(rng.choice([8, 8, 10, 16]))
    if bitdepth != 8:
        attrs = (attrs.astype(np.int64) * ((1 << bitdepth) - 1) // 255).astype(np.int32)
    # prediction weights: the reference normalises with a 64-entry reciprocal table
    # indexed by the weight sum (RAHT.cpp:445-451,567-570); sets whose largest
    # possible sum exceeds it read past the table there, so stay inside
    while True:
        w = tuple(int(x) for x in rng.integers(1, 12, 5))
        if w[0] + 3 * max(w[1], w[3]) + 3 * max(w[2], w[4]) <= 64:
            break
    pkw = dict(prediction=int(rng.integers(0, 2)), haar=int(rng.integers(0, 4) == 0),
               thr0=int(rng.integers(0, 20)), thr1=int(rng.integers(0, 20)),
               subnode=int(rng.integers(0, 2)), search_range=int(rng.choice([1, 7, 100, 50000])),
               weights=w, ext=int(rng.integers(0, 4) != 0))
    nl = int(rng.integers(1, 5))
    layers = [(int(rng.integers(4, 52)), int(rng.integers(-6, 7))) for _ in range(nl)]
    ac = None
    if rng.integers(0, 4) == 0:
        ac = [[(int(rng.integers(-4, 5)), int(rng.integers(-4, 5))) for _ in range(7)]
              for _ in range(int(rng.integers(1, 4)))]
    qkw = dict(layers=layers, bitdepth=bitdepth, fixed_point_qp_offset=int(rng.choice([0, 0, 8, 24])), ac_qps=ac)
    qpo = None
    if rng.integers(0, 3) == 0:
        qpo = np.zeros((len(xyz), 2), dtype=np.int32)
        sel = rng.random(len(xyz)) < 0.4
        qpo[sel] = (int(rng.integers(-6, 7)), int(rng.integers(-6, 7)))
    return xyz, attrs, pkw, qkw, qpo


def main():
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    rng = np.random.default_rng(seed)
    bad = 0
    for i in range(cases):
        xyz, attrs, pkw, qkw, qpo = random_case(rng)
        params, qs = make_params(**pkw), make_qpset(**qkw)
        mort, a_s, order = sort_cloud(xyz, attrs)
        q = qpo[order] if qpo is not None else None
        rr, rc = ref_raht(1, params, qs, mort, a_s, qpoffs=q)
        orc, oc = oracle_raht(1, params, qs, mort, a_s, qpoffs=q)
        er, ec = emu_raht(1, params, qs, mort, a_s, qpoffs=q)
        ok = same(rr, orc) and same(rc, oc) and np.array_equal(er, orc) and np.array_equal(ec, oc)
        if ok:  # decoders from the encoder's coefficients
            dr, _ = ref_raht(0, params, qs, mort, a_s * 0, coeffs=rc, qpoffs=q)
            do, _ = oracle_raht(0, params, qs, mort, a_s * 0, coeffs=oc, qpoffs=q)
            de, _ = emu_raht(0, params, qs, mort, a_s * 0, coeffs=oc, qpoffs=q)
            ok = same(dr, do) and np.array_equal(de, do) and same(dr, rr)
        if ok and qpo is None and qkw["bitdepth"] <= 10:
            # attribute level: the reference encoder's bitstream from the oracle's symbols
            payload, recon = ref_raht_encode_payload(params, qs, xyz, attrs, bitdepth=qkw["bitdepth"])
            runs, vals, ctx, tail = oracle_coeff_symbols(oc)
            out = np.empty_like(orc)
            out[order] = np.clip(orc, 0, (1 << qkw["bitdepth"]) - 1)
            ok = (same(out, recon)
                  and same(ref_symbols_payload(0, runs, vals, ctx, tail, len(xyz)), payload)
                  and same(ref_symbols_payload(1, runs, vals, ctx, tail, len(xyz)), payload))
            es = emu_coeff_symbols(ec)
            ok = ok and np.array_equal(es[0], runs) and np.array_equal(es[1], vals) and es[3] == tail
        if not ok:
            bad += 1
            print("MISMATCH case", i, "n", len(xyz), "A", attrs.shape[1], pkw, qkw, "qpo", qpo is not None)
    print(f"{cases} cases, {bad} mismatches (seed {seed})")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
