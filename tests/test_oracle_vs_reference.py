"""CPU tests: the oracle (oracle/raht_oracle.c) against (a) the committed
golden vectors produced by the unmodified reference and (b) the outputs of
the compiled reference on a wider set of clouds and flag combinations, as
recorded in tests/golden/reference_tape.npz (pcc_testlib: `taped`)."""
import os

import numpy as np
import pytest

from pcc_testlib import *  # noqa

GOLD = os.path.join(os.path.dirname(__file__), "golden")
from golden.make_golden import VARIANTS  # noqa


@pytest.fixture(scope="module")
def raht_gold():
    return np.load(os.path.join(GOLD, "raht_golden.npz"))


@pytest.fixture(scope="module")
def arith_gold():
    return np.load(os.path.join(GOLD, "arith_golden.npz"))


def test_arith_golden(arith_gold):
    g = arith_gold
    o = load_oracle()
    assert [o.oracle_isqrt(int(x)) for x in g["xs"]] == g["isqrt"].tolist()
    assert [o.oracle_irsqrt(int(x)) for x in g["xs"]] == g["irsqrt"].tolist()
    assert [o.oracle_fixed_mul(int(a), int(b)) for a, b in zip(g["fa"], g["fb"])] == g["fxmul"].tolist()
    assert [o.oracle_quantize(int(q), int(x)) for q, x in zip(g["qps"], g["qx"])] == g["quant"].tolist()
    assert [o.oracle_scale(int(q), int(x)) for q, x in zip(g["qps"], g["qx"])] == g["scale"].tolist()
    assert [o.oracle_morton_addr(*map(int, p)) for p in g["pts"]] == g["morton"].tolist()
    assert [o.oracle_morton3d_add(int(a), int(b)) for a, b in zip(g["ma"], g["mb"])] == g["madd"].tolist()
    assert [o.oracle_div_approx(int(a), int(b), 0) for a, b in zip(g["da"], g["db"])] == g["divapprox"].tolist()
    assert np.array_equal(np_morton(g["pts"]), g["morton"])


@pytest.mark.parametrize("cname", ["cube", "shell", "shelldup", "lidar", "sparse21"])
def test_raht_golden(raht_gold, cname):
    g = raht_gold
    xyz, attrs = g[f"{cname}/xyz"], g[f"{cname}/attrs"]
    qpo = g[f"{cname}/qpo"] if f"{cname}/qpo" in g else None
    mort, a_s, order = sort_cloud(xyz, attrs)
    k2, o2 = oracle_morton_sort(xyz)
    assert np.array_equal(k2, mort) and np.array_equal(o2, order)
    q = qpo[order] if qpo is not None else None
    for vname, kw in VARIANTS.items():
        for qp in (16, 34):
            p, qs = make_params(**kw), make_qpset(qp=qp)
            rec, coef = oracle_raht(1, p, qs, mort, a_s, qpoffs=q)
            assert np.array_equal(coef, g[f"{cname}/{vname}/qp{qp}/coef"]), (vname, qp)
            assert np.array_equal(rec, g[f"{cname}/{vname}/qp{qp}/rec"]), (vname, qp)
            rec2, _ = oracle_raht(0, p, qs, mort, a_s * 0, coeffs=coef, qpoffs=q)
            assert np.array_equal(rec2, rec), (vname, qp)


def _cmp(xyz, attrs, p, qs, qpo=None):
    mort, a_s, order = sort_cloud(xyz, attrs)
    q = qpo[order] if qpo is not None else None
    rr, rc = ref_raht(1, p, qs, mort, a_s, qpoffs=q)
    orr, oc = oracle_raht(1, p, qs, mort, a_s, qpoffs=q)
    assert same(rc, oc)
    assert same(rr, orr)
    r2, _ = ref_raht(0, p, qs, mort, a_s * 0, coeffs=rc, qpoffs=q)
    o2, _ = oracle_raht(0, p, qs, mort, a_s * 0, coeffs=oc, qpoffs=q)
    assert same(r2, o2)
    assert same(r2, rr)  # decoder reproduces the encoder's reconstruction


@pytest.mark.parametrize("kw", [dict(), dict(prediction=0), dict(subnode=0), dict(haar=1),
                                dict(ext=0), dict(ext=0, subnode=0), dict(thr0=0, thr1=1)])
@pytest.mark.parametrize("qp", [10, 34, 46])
def test_live_shell(kw, qp):
    xyz, attrs = cloud_shell(30000, bits=8, seed=qp)
    _cmp(xyz, attrs, make_params(**kw), make_qpset(qp=qp))


@pytest.mark.parametrize("a", [1, 3])
def test_live_dups_and_lidar(a):
    xyz, attrs = cloud_shell(30000, bits=7, seed=4, a=a, dups=True)
    for kw in (dict(), dict(haar=1), dict(ext=0)):
        _cmp(xyz, attrs, make_params(**kw), make_qpset(qp=28))
    xyz, attrs = cloud_lidar(40000, seed=2, a=a)
    _cmp(xyz, attrs, make_params(search_range=2500), make_qpset(qp=34))
    xyz, attrs = cloud_random(20000, 3, seed=12, a=a)  # weights > 1024
    _cmp(xyz, attrs, make_params(), make_qpset(qp=34))


def test_live_qp_structures():
    rng = np.random.default_rng(7)
    xyz, attrs = cloud_shell(30000, bits=8, seed=5)
    qpo = rng.integers(-6, 7, size=(xyz.shape[0], 2)).astype(np.int32)
    _cmp(xyz, attrs, make_params(), make_qpset(qp=30), qpo)
    _cmp(xyz, attrs, make_params(), make_qpset(layers=[(40, -2), (36, -1), (32, 0), (28, 1), (26, 2)]))
    ac = [[(l - c, c - l) for c in range(7)] for l in range(4)]
    _cmp(xyz, attrs, make_params(), make_qpset(qp=30, ac_qps=ac), qpo)
    xyz, a16 = cloud_random(20000, 8, seed=11, bitdepth=16)
    _cmp(xyz, a16, make_params(), make_qpset(qp=40, bitdepth=16))


def test_live_edge_cases():
    rng = np.random.default_rng(3)
    for n in (1, 2, 3, 9, 17):
        xyz, attrs = cloud_random(n, 3, seed=n)
        _cmp(xyz, attrs, make_params(), make_qpset(qp=20))
    xyz = np.tile(np.array([[5, 6, 7]], dtype=np.int32), (6, 1))
    attrs = rng.integers(0, 256, size=(6, 3)).astype(np.int32)
    _cmp(xyz, attrs, make_params(), make_qpset(qp=20))  # every point identical
    xyz = np.array([[0, 0, 0], [2**20, 2**20, 2**20], [2**20 + 1, 2**20, 2**20]], dtype=np.int32)
    _cmp(xyz, attrs[:3], make_params(thr0=0, thr1=0), make_qpset(qp=20))  # skipped stages
    for bits in (4, 12, 21):
        xyz, attrs = cloud_random(10000, bits, seed=bits, dup_frac=0.2)
        _cmp(xyz, attrs, make_params(thr0=0, thr1=1), make_qpset(qp=30))


def test_live_scalar_helpers():
    o = load_oracle()
    rng = np.random.default_rng(5)
    xs = np.concatenate([np.arange(0, 3000, dtype=np.uint64), rng.integers(0, 1 << 62, size=3000, dtype=np.uint64)])
    assert same(ref_elementwise("isqrt", "uint64", xs),
                np.array([o.oracle_isqrt(int(x)) for x in xs], dtype=np.uint64))
    assert same(ref_elementwise("irsqrt", "uint64", xs),
                np.array([o.oracle_irsqrt(int(x)) for x in xs], dtype=np.uint64))
    # kDivApproxDivisor[i] + 1 == 65536 // (i + 1) for every index the LUT serves
    b = np.arange(1, 257)
    assert same(ref_elementwise("div_approx", "int64", np.full(256, 1 << 20), b, np.zeros(256, dtype=np.int64)),
                np.array([o.oracle_div_approx(1 << 20, int(v), 0) for v in b], dtype=np.int64))


@pytest.mark.parametrize("a", [1, 3])
def test_live_lifting(a):
    """lift_oracle.c against PCCComputeQuantizationWeights / PCCLiftPredict /
    PCCLiftUpdate of the compiled reference, on synthetic LoD structures."""
    rng = np.random.default_rng(17)
    for n, lods in ((5000, 6), (60000, 10), (37, 3)):
        preds, npl = synth_predictors(n, lods, seed=n)
        qw_r = ref_quant_weights(preds)
        qw_o = oracle_quant_weights(preds)
        assert same(qw_r, qw_o)
        attrs = (rng.integers(0, 256, size=(n, a)).astype(np.int64)) << 8
        fr = ref_lift(1, preds, qw_r, npl, attrs)
        fo = oracle_lift(1, preds, qw_o, npl, attrs)
        assert same(fr, fo)
        ir = ref_lift(0, preds, qw_r, npl, fr)
        io = oracle_lift(0, preds, qw_o, npl, fo)
        assert same(ir, io)


LOD_CASES = [
    dict(),
    dict(distribution=0),
    dict(decimation=1),
    dict(decimation=2),
    dict(decimation=0, skip_layers=0, intra_range=128, inter_range=128, blending=1),
    dict(decimation=1, skip_layers=0, intra_range=16, inter_range=16, blending=1, period=3),
    dict(decimation=2, k=1, inter_range=8),
    dict(decimation=0, bias=(1, 2, 3), levels=6, dist2=1),
]


def _cmp_lod(xyz, kw):
    lp = make_lod_params(**kw)
    rp, ri, rn = ref_lod_build(lp, xyz)
    op, oi, on = oracle_lod_build(lp, xyz)
    assert same(rn, on), kw
    assert same(ri, oi), kw
    assert same(rp, op), kw


@pytest.mark.parametrize("kw", LOD_CASES)
def test_live_lod(kw):
    """lod_oracle.c against AttributeLods::generate of the compiled reference:
    numPointsInLod, indexes and every predictor (count, indices, weights)."""
    xyz, _ = cloud_shell(40000, bits=9, seed=3)
    _cmp_lod(xyz, kw)
    xyz, _ = cloud_lidar(40000, seed=2)
    _cmp_lod(xyz, dict(kw, levels=8))


def test_live_lod_edge_cases():
    xyz, _ = cloud_random(20000, 21, seed=5, dup_frac=0.1)   # many atlases, stalled fill cursor
    _cmp_lod(xyz, dict(levels=14))
    _cmp_lod(xyz, dict(decimation=1))
    xyz, _ = cloud_random(20000, 5, seed=6)                  # heavy duplicates
    for dec in (0, 1, 2):
        _cmp_lod(xyz, dict(decimation=dec, levels=5))
    for n in (1, 2, 5, 40):
        xyz, _ = cloud_random(n, 4, seed=n)
        _cmp_lod(xyz, dict())


def test_lod_golden():
    from golden.make_golden import LOD_GOLDEN_CASES

    g = np.load(os.path.join(GOLD, "lod_golden.npz"))
    for cname in ("shell", "sparse"):
        for i, kw in enumerate(LOD_GOLDEN_CASES):
            p, idx, npl = oracle_lod_build(make_lod_params(**kw), g[f"{cname}/xyz"])
            assert np.array_equal(npl, g[f"{cname}/{i}/npl"])
            assert np.array_equal(idx, g[f"{cname}/{i}/indexes"])
            assert np.array_equal(p, g[f"{cname}/{i}/preds"])


@pytest.mark.parametrize("a", [1, 3])
def test_live_lifting_encoder(a):
    """The oracle chain (LoD build, weights, lifting, LCP, quantisation,
    reconstruction) against the reference's own lifting encoder bodies
    (encodeColorsLift / encodeReflectancesLift): quantised values as decoded
    from the reference's arithmetic-coded payload, the reconstruction written
    back into the point cloud, and the LCP coefficients."""
    for cloud in (cloud_shell(20000, bits=9, seed=3, a=a), cloud_lidar(20000, seed=2, a=a)):
        xyz, attrs = cloud
        for qp in (34, 16):
            for lcp in (0, 1):
                for dec in (0, 1, 2):
                    lp = make_lod_params(levels=10, decimation=dec)
                    qs = make_qpset(qp=qp, chroma_offset=-2 if a == 3 else 0, fixed_point_qp_offset=24)
                    rv, rr, rl = ref_lift_encode(lp, qs, lcp, xyz, attrs)
                    ov, orr, ol = oracle_lift_encode(lp, qs, lcp, xyz, attrs)
                    assert same(rv, ov) and same(rr, orr)
                    if a == 3 and lcp:
                        assert same(rl, ol)


# --------------------------------------------------------------------------
# spherical coordinates for attribute coding (row N2)

def test_spherical_golden():
    """oracle against the committed outputs of the compiled reference"""
    g = np.load(os.path.join(GOLD, "spherical_golden.npz"))
    for name in g["names"]:
        rpl, bbox = oracle_xyz_to_rpl(g[f"{name}/origin"], g[f"{name}/theta"], g[f"{name}/xyz"])
        assert np.array_equal(rpl, g[f"{name}/rpl"]) and np.array_equal(bbox, g[f"{name}/bbox"])
        sc = oracle_offset_and_scale(bbox[:3], g[f"{name}/weight"], rpl)
        assert np.array_equal(sc, g[f"{name}/scaled"])


def test_live_spherical():
    orc = load_oracle()
    rng = np.random.default_rng(5)
    # the fixed-point arc tangent, all quadrants, axes, tiny and large arguments
    ys = np.concatenate([rng.integers(-(1 << 30), 1 << 30, 4000), rng.integers(-300, 300, 2000),
                         [0, 0, 1, -1, 5, -5, 0, (1 << 30), -(1 << 30)]])
    xs = np.concatenate([rng.integers(-(1 << 30), 1 << 30, 4000), rng.integers(-300, 300, 2000),
                         [0, 7, 0, 0, 5, 5, -9, (1 << 30), (1 << 30)]])
    assert same(ref_elementwise("iatan2", "int64", ys, xs),
                np.array([orc.oracle_iatan2(int(y), int(x)) for y, x in zip(ys, xs)], dtype=np.int64))
    # whole conversion on LiDAR-shaped and uniformly random clouds
    xyz, _ = cloud_lidar(30000, seed=4)
    wide = rng.integers(-(1 << 21), 1 << 21, size=(20000, 3)).astype(np.int32)
    for pts, origin, theta in ((xyz, (3, -4, 20), lidar_lasers(64)),
                               (xyz, (0, 0, 0), lidar_lasers(32, -0.3, 0.1)),
                               (wide, (100, -100, 7), lidar_lasers(40, -1.2, 1.2)),
                               (wide[:100], (0, 0, 0), lidar_lasers(1)),
                               (wide[:100], (0, 0, 0), lidar_lasers(2)),
                               (wide[:1], (1, 2, 3), lidar_lasers(5))):
        r, rb = ref_xyz_to_rpl(origin, theta, pts)
        o, ob = oracle_xyz_to_rpl(origin, theta, pts)
        assert same(r, o) and same(rb, ob)
        w = ref_normalised_axes_weights(np.maximum(rb[3:], 1))
        for mp in (rb[:3], (0, 0, 0), (-50, 7, 1)):
            assert same(ref_offset_and_scale(mp, w, r), oracle_offset_and_scale(mp, w, o))


# --------------------------------------------------------------------------
# symbol preparation for the entropy coder (row N1)

def _oracle_symbols_for(xyz, attrs, params, qs):
    mort, a_s, order = sort_cloud(xyz, attrs)
    orec, ocoef = oracle_raht(1, params, qs, mort, a_s)
    out = np.empty_like(orec)
    out[order] = np.clip(orec, 0, 255)
    return out, oracle_coeff_symbols(ocoef)


def test_symbols_golden():
    """oracle (RAHT + coefficient walk) against the symbol stream decoded from
    the reference encoder's payload (committed)"""
    from golden.make_golden import SYMBOL_GOLDEN_CASES

    g = np.load(os.path.join(GOLD, "symbols_golden.npz"))
    for name, a, qp in SYMBOL_GOLDEN_CASES:
        rec, (runs, vals, ctx, tail) = _oracle_symbols_for(
            g[f"{name}/xyz"], g[f"{name}/attrs"], make_params(), make_qpset(qp=qp))
        assert np.array_equal(runs, g[f"{name}/runs"]) and np.array_equal(vals, g[f"{name}/values"])
        assert tail == int(g[f"{name}/tail"]) and np.array_equal(rec, g[f"{name}/recon"])
        assert (ctx is None) == (a == 1)


@pytest.mark.parametrize("a", [1, 3])
def test_live_symbols(a):
    """the oracle's symbol stream, pushed through the reference's own
    PCCResidualsEncoder, must give the reference encoder's bitstream byte for
    byte — through encode() (runs + values) and through encodeSymbol with the
    oracle's context selectors; and it must be what the reference decoder reads"""
    for xyz, attrs in (cloud_shell(15000, bits=8, seed=3, a=a), cloud_lidar(15000, seed=2, a=a),
                       cloud_random(3000, 12, seed=7, a=a, dup_frac=0.2)):
        for qp, kw in ((34, {}), (10, {}), (46, dict(prediction=0)), (22, dict(haar=1))):
            params, qs = make_params(**kw), make_qpset(qp=qp)
            payload, recon = ref_raht_encode_payload(params, qs, xyz, attrs)
            rec, (runs, vals, ctx, tail) = _oracle_symbols_for(xyz, attrs, params, qs)
            assert same(rec, recon)
            n = len(xyz)
            assert same(ref_symbols_payload(0, runs, vals, ctx, tail, n), payload)
            assert same(ref_symbols_payload(1, runs, vals, ctx, tail, n), payload)
            rr, rv, rt = ref_decode_symbol_stream(payload, n, a)
            assert same(rr, runs) and same(rv, vals) and rt == tail


# --------------------------------------------------------------------------
# estimateDist2 (row N3, first half)

def _dist2_cases():
    rng = np.random.default_rng(21)
    cases = []
    for n, bits in ((30000, 8), (30000, 12), (5000, 18), (150, 6), (2, 4), (3, 20)):
        xyz, _ = cloud_random(n, bits, seed=n + bits)
        mort, _, order = sort_cloud(xyz, np.zeros((len(xyz), 1), dtype=np.int32))
        cases.append(xyz[order])  # coding order is Morton order after geometry coding
    cases.append(cloud_lidar(40000, seed=3)[0])
    cases.append(cloud_shell(40000, bits=10, seed=3)[0])
    cases.append(np.zeros((500, 3), dtype=np.int32))  # all points coincide
    cases.append((rng.integers(0, 1 << 20, size=(4000, 3))).astype(np.int32))  # unsorted, far apart
    return cases


DIST2_PARAMS = [(100, 128, 0.85), (1, 4, 0.5), (7, 1, 0.0), (10, 300, 0.99), (1000, 128, 0.85)]


def test_live_estimate_dist2():
    for xyz in _dist2_cases():
        for period, rng_, pct in DIST2_PARAMS:
            r = ref_estimate_dist2(xyz, period, rng_, pct)
            assert oracle_estimate_dist2(xyz, period, rng_, pct) == r, (len(xyz), period, rng_, pct)


# --------------------------------------------------------------------------
# quantisation weights of the predicting transform and of scalable lifting (row L5)

def _qw_structures():
    out = [synth_predictors(n, lods, seed=n) for n, lods in ((5000, 6), (40000, 9), (37, 3))]
    # real LoD builds, with predictors that reference their own level of detail
    for kw in (dict(decimation=0, skip_layers=0, intra_range=128, inter_range=128, blending=1),
               dict(decimation=1, skip_layers=0, intra_range=16, inter_range=16, period=3),
               dict()):
        xyz, _ = cloud_shell(15000, bits=8, seed=9)
        p, idx, npl = oracle_lod_build(make_lod_params(**dict(kw, levels=8)), xyz)
        out.append((p, npl))
    return out


def test_live_quant_weight_variants():
    for preds, npl in _qw_structures():
        for nw in ((256, 128, 64), (1, 1, 1), (8192, 0, 5)):
            assert same(ref_quant_weights_fixed(preds, nw), oracle_quant_weights_fixed(preds, nw))
        n = len(preds)
        for num_points, min_log2 in ((n, 0), (n, 2), (3 * n + 7, 1)):
            assert same(ref_quant_weights_scalable(preds, npl, num_points, min_log2),
                        oracle_quant_weights_scalable(npl, num_points, min_log2))
