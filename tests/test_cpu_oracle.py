"""CPU tests (run with -m "not gpu"): the oracle is pinned against the golden vectors, the
host build of the device geometry agrees with the reference's Clipper, the C-ABI library loads
and exports everything include/stardist_b200.h declares.  No compute call needs a GPU here."""
import ctypes, json, os, re, subprocess, sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases
from oracle import ref_ext, geom2d_np, nms_np

needs_ref = pytest.mark.skipif(not ref_ext.available(), reason="oracle/_ref not built (make -C oracle ref)")


@needs_ref
@pytest.mark.parametrize("name", list(cases.NMS2D_CASES))
def test_ref_nms2d_matches_golden(name, golden_dir):
    """the compiled reference reproduces the committed golden keep masks (pins oracle/_ref)"""
    g = np.load(os.path.join(golden_dir, "nms2d.npz"))
    d, p, s, thr = cases.nms2d_inputs(name)
    assert len(d) == int(g[name + "/n"])
    for kd in (1, 0):
        keep = ref_ext.stardist2d().c_non_max_suppression_inds(d, p, kd, 1, 0, thr)
        want = np.unpackbits(g["%s/keep_kd%d" % (name, kd)])[:len(d)].astype(bool)
        assert np.array_equal(keep, want)


@needs_ref
def test_kdtree_changes_result_only_at_exact_touching_distance(golden_dir):
    """reference property (tests/test_nms3D.py:46 analogue in 2D): kd-tree on/off -> same survivors,
    EXCEPT when centres sit exactly at the strict radius (noise 0, thresh 0: circles at distance
    2r are skipped by the kd-tree's `d2 < r2` but overlap after integer truncation)."""
    g = np.load(os.path.join(golden_dir, "nms2d.npz"))
    for name in cases.NMS2D_CASES:
        same = np.array_equal(g[name + "/keep_kd1"], g[name + "/keep_kd0"])
        assert same == (name != "r32_noise0_thr0")


def _hostcheck():
    path = os.path.join(ROOT, "tests", "hostcheck", "_build", "libhostcheck.so")
    subprocess.run(["make", "-C", os.path.join(ROOT, "tests", "hostcheck")], check=True, stdout=subprocess.DEVNULL)
    return ctypes.CDLL(path)


CLIP_CASES = [(32, 10, .1, 0), (32, 3, .5, 1), (11, 8, .1, 2), (64, 20, .4, 3), (32, 30, .9, 4)]
CLIP_PAIRS = 40000


@pytest.mark.parametrize("n_rays,radius,noise,seed", CLIP_CASES)
def test_clip_sweep_bit_exact_vs_reference_clipper(n_rays, radius, noise, seed, golden_dir):
    """clip2d.cuh (host build) == vendored Clipper 6.4.2 on fuzzed polygon pairs, float-bit exact on every pair (where
    oracle/_ref is not built: against the sha256 of the reference's float32 areas, tests/golden/refshim.npz, make_refshim.py)"""
    import hashlib
    sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))
    import clip_fuzz as cf
    cf.hc = _hostcheck()
    a, b = cf.make_pairs(CLIP_PAIRS, n_rays, radius, noise, seed)
    h, st = cf.host(a, b)
    assert np.count_nonzero(st == 2) == 0
    if cf.ref is not None:          # the reference's Clipper built in oracle/_ref
        r, _, _ = cf.run(a, b)
        assert np.array_equal(r.view(np.int32), h.view(np.int32))
    else:
        want = np.load(os.path.join(golden_dir, "refshim.npz"))["clip/%d/sha256" % seed].tobytes().decode()
        assert hashlib.sha256(np.ascontiguousarray(h, "<f4").tobytes()).hexdigest() == want
    assert np.count_nonzero(h) > 1000


def test_capi_exports_every_declared_symbol():
    lib_path = os.path.join(ROOT, "stardist_b200", "libstardist_b200.so")
    if not os.path.exists(lib_path):
        pytest.skip("libstardist_b200.so not built (python -c 'import __graft_entry__ as g; g.build()')")
    hdr = open(os.path.join(ROOT, "include", "stardist_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = re.findall(r"\b((?:sdb_|_LIB_)\w+)\s*\(", hdr)
    assert len(names) >= 10
    lib = ctypes.CDLL(lib_path)
    missing = [n for n in sorted(set(names)) if not hasattr(lib, n)]
    assert not missing, "declared in include/stardist_b200.h but not exported: %s" % missing


def test_product_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from stardist_b200 import _lib
    from stardist_b200.lib.stardist2d import c_non_max_suppression_inds
    with pytest.raises(_lib.StarDistB200Error):
        c_non_max_suppression_inds(np.ones((3, 32), np.float32), np.zeros((3, 2), np.float32), 1, 1, 0, np.float32(.4))


# ---- polygon rule restatement (skimage is not installed: property tests only) -------------
def test_polygon_rule_convex_matches_halfplanes():
    rng = np.random.default_rng(0)
    for _ in range(20):
        R = 16
        phi = np.linspace(0, 2 * np.pi, R, endpoint=False)
        c = rng.uniform(20, 40, 2); rad = rng.uniform(5, 15)
        r = (c[0] + rad * np.sin(phi)).astype(np.float32); cc = (c[1] + rad * np.cos(phi)).astype(np.float32)
        rr, cx = geom2d_np.polygon(r, cc, (64, 64))
        img = np.zeros((64, 64), bool); img[rr, cx] = True
        # strict interior by half-plane test must be painted, strict exterior must not
        Y, X = np.mgrid[0:64, 0:64].astype(np.float64)
        inside = np.ones((64, 64), bool); outside = np.zeros((64, 64), bool)
        for k in range(R):
            y0, x0, y1, x1 = float(r[k]), float(cc[k]), float(r[(k + 1) % R]), float(cc[(k + 1) % R])
            cr = (x1 - x0) * (Y - y0) - (y1 - y0) * (X - x0)
            sgn = np.sign((x1 - x0) * (c[0] - y0) - (y1 - y0) * (c[1] - x0))     # side of the centre
            inside &= sgn * cr > 1e-9; outside |= sgn * cr < -1e-9
        assert inside.sum() > 50
        assert img[inside].all() and not img[outside].any()


def test_polygon_integer_vertices_are_painted():
    # n_rays=32: rays 0/16 land on integer rows, 8/24 on integer columns for integer centres (SURVEY A.4)
    d = np.full((1, 32), 5.0, np.float32); p = np.array([[20, 20]])
    lbl = geom2d_np.polygons_to_label(d, p, (40, 40))
    assert lbl[20, 25] == 1 and lbl[20, 15] == 1 and lbl[25, 20] == 1 and lbl[15, 20] == 1
    assert lbl[20, 26] == 0 and lbl[14, 20] == 0


def test_paint_order_highest_prob_wins():
    d = np.full((2, 32), 6.0, np.float32); p = np.array([[20, 20], [20, 24]])
    lbl = geom2d_np.polygons_to_label(d, p, (40, 48), prob=np.array([0.9, 0.8]))
    assert lbl[20, 22] == 1          # overlap region belongs to the higher prob polygon (painted last)
    lbl = geom2d_np.polygons_to_label(d, p, (40, 48), prob=np.array([0.8, 0.8]))
    assert lbl[20, 22] == 2          # ties: stable ascending sort paints index 1 last


def test_stable_score_order_definition():
    s = np.array([.5, .9, .5, .9, .1], np.float32)
    assert nms_np.argsort_desc(s).tolist() == [3, 1, 2, 0, 4]


def test_unet_topology_param_counts():
    from stardist_b200.models.config import Config2D
    from stardist_b200.models.weights import glorot_uniform_weights, count_params
    assert count_params(glorot_uniform_weights(Config2D())) == 1406689            # SURVEY section 8
    assert count_params(glorot_uniform_weights(Config2D(grid=(2, 2)))) == 1425185  # == 2D_demo weights file


def test_oracle_reproduces_reference_2d_demo_test():
    """The reference pins its shipped 2D_demo model on its test image to matching(...) == (fp 5, tp 114, fn 11)
    (stardist tests/test_model2D.py:92-106).  The oracle (torch-CPU U-Net restatement + reference C++ NMS + numpy label
    painting) with those weights must reproduce exactly that: this pins the network restatement to a reference test."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import demo2d
    from oracle import pipeline2d, ref_ext
    if not ref_ext.available():
        pytest.skip("oracle/_ref not built")
    import stardist_b200 as sd
    from stardist_b200.utils import normalize
    from stardist_b200.matching import matching
    kwargs, weights, thr, img, mask = demo2d.load()
    cfg = sd.Config2D(**kwargs)
    assert sum(k.size + b.size for k, b in weights.values()) == 1425185
    x = normalize(img, 1, 99.8)
    labels, res = pipeline2d.predict_instances(cfg, weights, x, thr['prob'], thr['nms'])
    assert labels.shape == img.shape and labels.max() == len(res['prob']) == len(res['points'])
    st = matching(mask, labels, thresh=0.5)
    assert (st.fp, st.tp, st.fn) == demo2d.REFERENCE_TEST_STATS


@pytest.fixture(scope="module")
def demo_models(tmp_path_factory):
    """the reference's models/examples/{2D_demo,3D_demo}, rebuilt byte for byte from tests/golden (demo_models.py)"""
    import demo_models
    return demo_models.rebuild(str(tmp_path_factory.mktemp("examples")))


def test_h5lite_reads_the_reference_weight_file(demo_models):
    """pure-Python HDF5 subset reader on the reference's 2D_demo weights_best.h5 == the frozen fixture"""
    import sys, os
    path = os.path.join(demo_models, "2D_demo", "weights_best.h5")
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import demo2d
    from stardist_b200.io import h5lite
    w = h5lite.read_keras_weights(path)
    _, weights, _, _, _ = demo2d.load()
    assert sorted(w) == sorted(weights)
    for n in w:
        assert np.array_equal(w[n][0], weights[n][0]) and np.array_equal(w[n][1], weights[n][1])
    with pytest.raises(h5lite.H5Error):
        h5lite.read_datasets(os.path.abspath(__file__))


def test_matching_metrics():
    from stardist_b200.matching import matching
    y = np.zeros((100, 100), np.uint16); y[10:20, 10:20] = 1
    st = matching(y, np.roll(y, 5, axis=0))
    assert (st.fp, st.tp, st.fn) == (1, 0, 1) and st.n_true == 1 and st.n_pred == 1
    st = matching(y, np.roll(y, 2, axis=0))
    assert (st.fp, st.tp, st.fn) == (0, 1, 0) and abs(st.mean_matched_score - 80 / 120) < 1e-6


def test_model_folder_with_keras_checkpoint_loads(demo_models):
    """StarDist2D(None, name, basedir) on a reference model folder: config.json + thresholds.json + weights_best.h5"""
    import stardist_b200 as sd
    m = sd.StarDist2D(None, name='2D_demo', basedir=demo_models)
    assert tuple(m.config.grid) == (2, 2) and m.config.n_rays == 32
    assert abs(m.thresholds.prob - 0.4861655269131771) < 1e-12 and m.thresholds.nms == 0.5
    assert m.weights['conv2d_1'][0].shape == (3, 3, 1, 32) and m.weights['dist'][0].shape == (1, 1, 128, 32)
    with pytest.raises(ValueError):
        sd.StarDist2D(sd.Config2D(n_rays=16), name=None, basedir=None, weights=m.weights)
    m3 = sd.StarDist3D(None, name='3D_demo', basedir=demo_models)
    assert m3.config.backbone == 'resnet' and tuple(m3.config.grid) == (1, 2, 2) and m3.config.n_rays == 96
    assert m3._axes_div_by('ZYX') == (1, 2, 2) and m3.weights['conv3d_1'][0].shape == (7, 7, 7, 1, 32)


def test_oracle_reproduces_reference_3d_demo_test():
    """3D_demo (ResNet backbone, 96 anisotropic rays, grid (1,2,2)) on the reference's test volume: the reference pins
    matching(...) == (fp 0, tp 30, fn 21) (stardist tests/test_model3D.py:85-96); the oracle (torch-CPU ResNet restatement +
    reference C++ NMS / polyhedron_to_label) must reproduce it."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import demo3d
    from oracle import pipeline3d, ref_ext
    if not ref_ext.available():
        pytest.skip("oracle/_ref not built")
    import stardist_b200 as sd
    from stardist_b200.utils import normalize
    from stardist_b200.matching import matching
    from stardist_b200.rays3d import rays_from_json
    rays_json, kwargs, weights, thr, img, mask = demo3d.load()
    rays = rays_from_json(rays_json)
    cfg = sd.Config3D(rays=rays, **kwargs)
    assert cfg.backbone == 'resnet' and sum(k.size + b.size for k, b in weights.values()) == 1547201
    old = os.environ.get("OMP_NUM_THREADS")
    os.environ["OMP_NUM_THREADS"] = "1"          # the reference's 3D NMS has a racy anisotropy sum
    try:
        labels, res = pipeline3d.predict_instances(cfg, rays, normalize(img, 1, 99.8), thr['prob'], thr['nms'], weights=weights)
    finally:
        if old is None: os.environ.pop("OMP_NUM_THREADS", None)
        else: os.environ["OMP_NUM_THREADS"] = old
    st = matching(mask, labels, thresh=0.5)
    assert labels.shape == img.shape and (st.fp, st.tp, st.fn) == demo3d.REFERENCE_TEST_STATS



def test_relabel_sequential_reference_docstring_vectors():
    """the known answers in the reference's docstring (stardist/matching.py:363-381)"""
    from stardist_b200.matching import relabel_sequential
    lf = np.array([1, 1, 5, 5, 8, 99, 42])
    relab, fw, inv = relabel_sequential(lf)
    assert relab.tolist() == [1, 1, 2, 2, 3, 5, 4]
    assert np.flatnonzero(fw).tolist() == [1, 5, 8, 42, 99] and fw[[1, 5, 8, 42, 99]].tolist() == [1, 2, 3, 4, 5] and len(fw) == 100
    assert inv.tolist() == [0, 1, 5, 8, 42, 99]
    assert (fw[lf] == relab).all() and (inv[relab] == lf).all()
    assert relabel_sequential(lf, offset=5)[0].tolist() == [5, 5, 6, 6, 7, 9, 8]
    with pytest.raises(ValueError):
        relabel_sequential(lf, offset=0)
    with pytest.raises(ValueError):
        relabel_sequential(np.array([1, -1]))


@pytest.mark.parametrize("noise,n_rays", cases.NMS3D_ACCURACY_CASES)
def test_oracle_reproduces_reference_nms_accuracy_test(noise, n_rays):
    """the reference's own property test (tests/test_nms3D.py:60-83) through the oracle (= the reference C++ + restated glue):
    two overlapping polyhedra, rendered IoU; NMS at 0.95*iou suppresses one, at 1.05*iou keeps both"""
    if not ref_ext.available(): pytest.skip("oracle/_ref not present")
    from oracle import pipeline3d
    dist, points, prob, rays, shape = cases.nms3d_accuracy_inputs(noise, n_rays)
    m1 = pipeline3d.polyhedron_to_label(dist[:1], points[:1], rays, shape, prob[:1])
    m2 = pipeline3d.polyhedron_to_label(dist[1:], points[1:], rays, shape, prob[1:])
    iou = np.count_nonzero(m1 * m2) / min(np.count_nonzero(m1), np.count_nonzero(m2) + 1e-10)
    assert 0 < iou < 1
    sup1 = nms_np.non_maximum_suppression_3d_sparse(dist, prob, points, rays, nms_thresh=0.95 * iou)[0]
    sup2 = nms_np.non_maximum_suppression_3d_sparse(dist, prob, points, rays, nms_thresh=1.05 * iou)[0]
    assert len(sup1) == 1 and len(sup2) == 2


def _hc_paint3d(hc, dist, point, rays, shape):
    hc.hc_paint3d.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int] * 5 + [ctypes.c_void_p]
    v = np.ascontiguousarray(rays.vertices, np.float32); f = np.ascontiguousarray(rays.faces, np.int32)
    d = np.ascontiguousarray(dist, np.float32); c = np.ascontiguousarray(point, np.float32)
    out = np.zeros(shape, np.uint8)
    hc.hc_paint3d(d.ctypes.data, c.ctypes.data, v.ctypes.data, f.ctypes.data, len(v), len(f), shape[0], shape[1], shape[2], out.ctypes.data)
    return out


@needs_ref
@pytest.mark.parametrize("noise,n_rays", cases.NMS3D_ACCURACY_CASES)
def test_device_render_rule_vs_reference_on_lattice_aligned_vertices(noise, n_rays):
    """k_paint3d's rule (host build of the same header code: f64 kernel half-spaces OR float inside_polyhedron, the Qhull hull
    test dropped) against the reference's c_polyhedron_to_label on the reference's test_nms_accuracy polyhedra, whose polar
    vertices lie exactly on the voxel lattice: the masks differ in at most 2 voxels, each one AT such a vertex (labelled here,
    left out by the reference whenever Qhull's plane rounding says so) -- DESIGN.md 5, 3D labels.  The B200 run shows the same
    counts (tests/test_gpu_3d.py::test_reference_nms_accuracy_property)."""
    from oracle import pipeline3d
    hc = _hostcheck()
    dist, points, prob, rays, shape = cases.nms3d_accuracy_inputs(noise, n_rays)
    for k in range(2):
        ours = _hc_paint3d(hc, dist[k], points[k], rays, shape)
        ref = pipeline3d.polyhedron_to_label(dist[k:k + 1], points[k:k + 1], rays, shape, prob[k:k + 1])
        diff = np.argwhere((ours > 0) != (ref > 0))
        assert len(diff) <= 2
        poles = {(int(points[k][0]) - 10, int(points[k][1]), int(points[k][2])), (int(points[k][0]) + 10, int(points[k][1]), int(points[k][2]))}
        for vox in diff:
            assert tuple(int(t) for t in vox) in poles and ours[tuple(vox)] == 1


@needs_ref
def test_device_render_rule_equals_reference_off_lattice():
    """same comparison on polyhedra without lattice-aligned vertices (random centres' fractional distances): identical masks"""
    from oracle import pipeline3d
    hc = _hostcheck()
    rng = np.random.default_rng(5)
    for n_rays in (24, 65, 96):
        rays = cases.rays_golden_spiral(n_rays, (2, 1, 1) if n_rays == 96 else None)
        shape = (36, 40, 44)
        for _ in range(6):
            dist = rng.uniform(3.3, 12.7, n_rays).astype(np.float32)
            point = np.array([rng.integers(12, 24), rng.integers(14, 26), rng.integers(14, 30)])
            ours = _hc_paint3d(hc, dist, point, rays, shape)
            ref = pipeline3d.polyhedron_to_label(dist[None], point[None], rays, shape, np.ones(1))
            assert np.count_nonzero(ref) > 100 and np.array_equal(ours > 0, ref > 0)


def test_face_cone_volume_n_bit_identical_to_face_cone_volume():
    """geom3d.cuh: the S3 / S4 volume stages on pre-normalised planes (face_cone_volume_n: planes scaled once, squared
    parallel test, non-cutting planes skipped) against the GPU-validated formulation, host build: identical float bits of both
    stages and identical raw double sums, on star polyhedra incl. integer centres, equal shapes and coincident centres"""
    import math
    hc = _hostcheck()
    for f in (hc.hc_overlap_kernel, hc.hc_overlap_convex, hc.hc_overlap_kernel_n, hc.hc_overlap_convex_n): f.restype = ctypes.c_float
    P = ctypes.c_void_p
    # sqrt(s) < 1e-12  <=>  s < 1e-24 for correctly rounded sqrt: check the doubles around the threshold
    x = np.float64(1e-24)
    assert math.sqrt(float(x)) >= 1e-12 and math.sqrt(float(np.nextafter(x, 0))) < 1e-12
    n_pos = 0; tot = 0
    for n_rays, aniso in ((96, None), (96, (2, 1, 1)), (32, None), (65, None)):
        r = cases.rays_golden_spiral(n_rays, aniso)
        verts = np.ascontiguousarray(r.vertices, np.float32); faces = np.ascontiguousarray(r.faces, np.int32)
        for radius, noise, sep, seed in ((10, .2, 12, 0), (10, .6, 8, 1), (5, .05, 3, 2), (20, .9, 25, 3)):
            rng = np.random.default_rng(seed * 7 + n_rays)
            for it in range(60):
                c1 = rng.uniform(20, 60, 3).astype(np.float32); c2 = (c1 + rng.uniform(-sep, sep, 3)).astype(np.float32)
                if it % 5 == 0: c1 = np.round(c1); c2 = np.round(c2)
                d1 = (radius * (1 + noise * rng.uniform(-1, 1, n_rays))).astype(np.float32)
                d2 = (radius * (1 + noise * rng.uniform(-1, 1, n_rays))).astype(np.float32)
                if it % 7 == 0: d2 = d1.copy()
                if it % 11 == 0: c2 = c1.copy()
                pv1 = (c1[None] + d1[:, None] * verts).astype(np.float32); pv2 = (c2[None] + d2[:, None] * verts).astype(np.float32)
                a = (P(pv1.ctypes.data), P(c1.ctypes.data), P(pv2.ctypes.data), P(c2.ctypes.data), P(faces.ctypes.data), n_rays, len(faces))
                k0, k1 = hc.hc_overlap_kernel(*a), hc.hc_overlap_kernel_n(*a)
                v0, v1 = hc.hc_overlap_convex(*a[:4], n_rays), hc.hc_overlap_convex_n(*a[:4], n_rays)
                out = np.zeros(2); hc.hc_overlap_kernel_pair(*a, P(out.ctypes.data))
                assert np.float32(k0).view(np.int32) == np.float32(k1).view(np.int32)
                assert np.float32(v0).view(np.int32) == np.float32(v1).view(np.int32)
                assert out[0] == out[1] or (np.isnan(out[0]) and np.isnan(out[1]))
                tot += 1; n_pos += k0 > 0
    assert n_pos > tot // 10


def test_stage_fill_matches_numpy_cast():
    """StarDistBase._stage_fill (host image -> float32 staging buffer): torch's parallel copy and the numpy fallback give the
    same float32 values as x.astype(np.float32) for contiguous / strided / float64 / integer / byte-swapped inputs"""
    import torch
    from stardist_b200.models.base import StarDistBase
    rng = np.random.default_rng(0)
    base = rng.uniform(-3, 3, (70, 300, 40))
    big = rng.uniform(-3, 3, (1 << 23) + 5).astype(np.float32)      # above the threshold of the torch path
    inputs = [base.astype(np.float32), base, base.astype(np.float32)[::-1, ::2], base[:, :, ::-1], np.asfortranarray(base.astype(np.float32)),
              big, big.astype(np.float64)[::-1], (base * 1000).astype(np.uint16), (base * 10).astype(np.int8), base.astype('>f4'), base.astype(np.float16), base[:3, :5, :7].astype(np.float32)]
    for x in inputs:
        stage = torch.full((1,) + x.shape, np.nan, dtype=torch.float32)
        StarDistBase._stage_fill(stage, x)
        assert np.array_equal(stage.numpy()[0], x.astype(np.float32)), (x.dtype, x.strides)


@needs_ref
def test_serial_host_nms3d_equals_reference_beyond_the_goldens():
    """tests/tools/nms3d_serial_fuzz.py (mini set; the full set -- 10 clouds, 10 935 candidates, 65 / 100 / 187 rays, anisotropic
    rays, use_bbox = 0, use_kdtree = 0, 69 k S3 / 66 k S4 / 26 k S5 evaluations -- gave 0 differing decisions, profiles/r01z):
    the arithmetic of geom3d.cuh / nms3d_pair.cuh in the reference's greedy order == the reference's c_non_max_suppression_inds,
    for both formulations of the volume stages.  Separate process with OMP_NUM_THREADS=1 (racy anisotropy sum in the reference)."""
    import json
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "tools", "nms3d_serial_fuzz.py"), "mini"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["cases"] == 4 and out["candidates"] > 400 and out["mismatches"] == 0
    assert all(c > 50 for c in out["stage_counts"])           # every stage of the cascade is exercised


def test_ray_classes_equal_reference(golden_dir):
    """stardist_b200.rays3d vs tests/golden/rays3d.npz (the reference's stardist/rays3d.py, imported standalone by
    make_rays3d.py): vertices bit-equal (float32), faces equal, volume / surface / dist_loss_weights / copy(scale) to 1e-12,
    for every ray class rays_from_json can name"""
    import json
    import stardist_b200 as sd
    g = np.load(os.path.join(golden_dir, "rays3d.npz"))
    specs = json.loads(bytes(g["specs"]).decode())
    assert len(specs) == 42
    for i, (name, kw) in enumerate(specs):
        kw = {k: (tuple(v) if isinstance(v, list) else v) for k, v in kw.items()}
        r = getattr(sd, name)(**kw)
        assert r.vertices.dtype == np.float32 and np.array_equal(r.vertices, g["%d/vertices" % i]), (name, kw)
        assert np.array_equal(r.faces, g["%d/faces" % i]), (name, kw)
        d = g["%d/dist" % i]
        assert np.allclose(r.volume(d), g["%d/volume" % i], rtol=1e-12, atol=0) and np.allclose(r.surface(d), g["%d/surface" % i], rtol=1e-12, atol=0)
        assert np.allclose(r.dist_loss_weights((2, 1, 1)), g["%d/weights" % i], rtol=1e-12, atol=0)
        assert np.array_equal(r.copy(scale=(.5, 1, 2)).vertices, g["%d/scaled" % i])
        r2 = sd.rays_from_json(json.loads(json.dumps(r.to_json())))               # config.json round trip
        assert type(r2) is type(r) and np.array_equal(r2.vertices, r.vertices) and np.array_equal(r2.faces, r.faces)


HOSTFUNC_NMS2D = ["r32_356x299", "r11_114x217", "r32_grid16", "r64_small"]
HOSTFUNC_NMS3D = ["r14_thr02", "r32_noise01_thr01", "r96_aniso_thr03"]


@needs_ref
@pytest.mark.parametrize("name", HOSTFUNC_NMS2D)
def test_oracle_host_glue_2d_equals_reference_modules(golden_dir, name):
    """oracle/nms_np.py and oracle/geom2d_np.py against the outputs of the reference's OWN nms.py / geom2d.py
    (tests/golden/hostfuncs.npz, produced by make_hostfuncs.py from the reference's sources): dense and sparse 2-D NMS front-ends
    (points, prob, dist, original indices) bit-equal, dist_to_coord bit-equal (float32)"""
    g = np.load(os.path.join(golden_dir, "hostfuncs.npz"))
    shape, radius, noise, n_rays, grid, pthr, nthr, seed = cases.NMS2D_CASES[name]
    prob, dist = cases.create_random_data_2d(shape, radius, noise, n_rays, seed)
    prob = prob[::grid[0], ::grid[1]]; dist = dist[::grid[0], ::grid[1]]
    p, pr, d = nms_np.non_maximum_suppression(dist, prob, grid=grid, b=2, nms_thresh=nthr, prob_thresh=pthr)
    k = "nms2d/%s/" % name
    assert np.array_equal(p, g[k + "points"]) and np.array_equal(pr, g[k + "prob"]) and np.array_equal(d, g[k + "dist"])
    mask = nms_np._ind_prob_thresh(prob, pthr, b=2)
    pts = np.stack(np.where(mask), 1) * np.array(grid).reshape(1, 2)
    ps, prs, ds, inds = nms_np.non_maximum_suppression_sparse(dist[mask], prob[mask], pts, nms_thresh=nthr)
    assert np.array_equal(ps, g[k + "sparse_points"]) and np.array_equal(inds, g[k + "sparse_inds"])
    for key, sc in (("coord", (1, 1)), ("coord_scaled", (2, .5))):
        c = geom2d_np.dist_to_coord(d, p, scale_dist=sc)
        assert c.dtype == g[k + key].dtype and np.array_equal(c, g[k + key])


@needs_ref
@pytest.mark.parametrize("name", HOSTFUNC_NMS3D)
def test_oracle_host_glue_3d_equals_reference_modules(golden_dir, name):
    """3-D: sparse NMS front-end (nms.py:285-384) and polyhedron_to_label (geom3d.py:100-198) of the reference vs the oracle"""
    from oracle import pipeline3d
    g = np.load(os.path.join(golden_dir, "hostfuncs.npz"))
    shape, noise, n_rays, pthr, nthr, seed, aniso = cases.NMS3D_CASES[name]
    prob, dist = cases.create_random_data_3d(shape, noise, n_rays, seed)
    rays = cases.rays_golden_spiral(n_rays, aniso)
    mask = nms_np._ind_prob_thresh(prob, pthr, b=2)
    pts = np.stack(np.where(mask), 1)
    ps, prs, ds, inds = nms_np.non_maximum_suppression_3d_sparse(dist[mask], prob[mask], pts, rays, nms_thresh=nthr)
    k = "nms3d/%s/" % name
    assert np.array_equal(ps, g[k + "sparse_points"]) and np.array_equal(inds, g[k + "sparse_inds"])
    assert np.array_equal(ps, g[k + "points"]) and np.array_equal(prs, g[k + "prob"]) and np.array_equal(ds, g[k + "dist"])   # dense == sparse
    lab = pipeline3d.polyhedron_to_label(ds, ps, rays, shape, prs)
    assert np.array_equal(lab, g[k + "labels"])


def test_matching_and_relabel_equal_reference_modules(golden_dir):
    """stardist_b200.matching (matching, relabel_sequential) and utils._normalize_grid against the reference's matching.py /
    utils.py outputs on three label-image pairs x 3 criteria x 3 thresholds"""
    from stardist_b200.matching import matching, relabel_sequential
    from stardist_b200.utils import _normalize_grid
    g = np.load(os.path.join(golden_dir, "hostfuncs.npz"))
    for seed in (0, 1, 2):
        a, b = g["match/%d/a" % seed], g["match/%d/b" % seed]
        for crit in ("iou", "iot", "iop"):
            for thr in (0.3, 0.5, 0.9):
                m = matching(a, b, thresh=thr, criterion=crit)
                got = np.array([m.fp, m.tp, m.fn, m.precision, m.recall, m.accuracy, m.f1, m.n_true, m.n_pred,
                                m.mean_true_score, m.mean_matched_score, m.panoptic_quality], np.float64)
                assert np.array_equal(got, g["match/%d/%s/%.1f" % (seed, crit, thr)]), (seed, crit, thr)
        rl, fw, inv = relabel_sequential(b, offset=3)
        assert np.array_equal(rl, g["relabel/%d/out" % seed]) and np.array_equal(fw, g["relabel/%d/fw" % seed]) and np.array_equal(inv, g["relabel/%d/inv" % seed])
    assert np.array_equal(np.array([_normalize_grid((2, 2, 2), 3), _normalize_grid([1, 2, 4], 3)]), g["normalize_grid"])


@needs_ref
def test_product_nms_front_end_equals_reference_modules(golden_dir, monkeypatch):
    """stardist_b200/nms.py (the host glue in front of the device kernels) with its two C entry points replaced by the
    reference's compiled extensions: dense and sparse, 2-D and 3-D front-ends return what the reference's own nms.py returned
    (tests/golden/hostfuncs.npz) -- the host logic is device independent, so this pins it on the CPU"""
    import stardist_b200.lib.stardist2d as l2, stardist_b200.lib.stardist3d as l3
    from stardist_b200 import nms
    monkeypatch.setattr(l2, "c_non_max_suppression_inds", ref_ext.stardist2d().c_non_max_suppression_inds)
    monkeypatch.setattr(l3, "c_non_max_suppression_inds", ref_ext.stardist3d().c_non_max_suppression_inds)
    g = np.load(os.path.join(golden_dir, "hostfuncs.npz"))
    for name in HOSTFUNC_NMS2D:
        shape, radius, noise, n_rays, grid, pthr, nthr, seed = cases.NMS2D_CASES[name]
        prob, dist = cases.create_random_data_2d(shape, radius, noise, n_rays, seed)
        prob = prob[::grid[0], ::grid[1]]; dist = dist[::grid[0], ::grid[1]]
        k = "nms2d/%s/" % name
        p, pr, d = nms.non_maximum_suppression(dist, prob, grid=grid, b=2, nms_thresh=nthr, prob_thresh=pthr)
        assert p.dtype == g[k + "points"].dtype and np.array_equal(p, g[k + "points"]) and np.array_equal(pr, g[k + "prob"]) and np.array_equal(d, g[k + "dist"])
        mask = nms._ind_prob_thresh(prob, pthr, b=2)
        pts = np.stack(np.where(mask), 1) * np.array(grid).reshape(1, 2)
        ps, prs, ds, inds = nms.non_maximum_suppression_sparse(dist[mask], prob[mask], pts, nms_thresh=nthr)
        assert np.array_equal(ps, g[k + "sparse_points"]) and np.array_equal(inds, g[k + "sparse_inds"]) and np.array_equal(ds, g[k + "dist"])
    for name in HOSTFUNC_NMS3D[:2]:
        shape, noise, n_rays, pthr, nthr, seed, aniso = cases.NMS3D_CASES[name]
        prob, dist = cases.create_random_data_3d(shape, noise, n_rays, seed)
        rays = cases.rays_golden_spiral(n_rays, aniso)
        k = "nms3d/%s/" % name
        p, pr, d = nms.non_maximum_suppression_3d(dist, prob, rays, grid=(1, 1, 1), b=2, nms_thresh=nthr, prob_thresh=pthr)
        assert p.dtype == g[k + "points"].dtype and np.array_equal(p, g[k + "points"]) and np.array_equal(pr, g[k + "prob"]) and np.array_equal(d, g[k + "dist"])
        mask = nms._ind_prob_thresh(prob, pthr, b=2)
        pts = np.stack(np.where(mask), 1)
        ps, prs, ds, inds = nms.non_maximum_suppression_3d_sparse(dist[mask], prob[mask], pts, rays, nms_thresh=nthr)
        assert np.array_equal(ps, g[k + "sparse_points"]) and np.array_equal(inds, g[k + "sparse_inds"]) and np.array_equal(prs, g[k + "prob"])
    # border handling of _ind_prob_thresh (nms.py:6-17): scalar, per-axis pairs, zero margins, None
    prob = np.random.default_rng(0).uniform(size=(9, 11))
    for b in (2, ((1, 0), (0, 3)), 0, None, ((0, 0), (2, 2))):
        want = prob > .3
        if b is not None:
            bb = ((b, b),) * 2 if np.isscalar(b) else b
            inner = np.zeros_like(want); inner[tuple(slice(lo if lo > 0 else None, -hi if hi > 0 else None) for lo, hi in bb)] = True
            want &= inner
        assert np.array_equal(nms._ind_prob_thresh(prob, .3, b=b), want)


def _jsonable(v):
    if isinstance(v, (tuple, list)): return [_jsonable(x) for x in v]
    if isinstance(v, dict): return {str(k): _jsonable(x) for k, x in v.items()}
    if isinstance(v, np.integer): return int(v)
    if isinstance(v, np.floating): return float(v)
    if isinstance(v, np.ndarray): return _jsonable(v.tolist())
    return v


def test_config_classes_equal_reference(golden_dir):
    """Config2D / Config3D: every attribute (names and values, incl. the derived ones -- n_channel_out, rays_json, net_input_shape,
    train_* defaults) equals the reference classes' for 4 + 4 keyword sets (tests/golden/models_host.json, produced by importing
    stardist/models/model2d.py / model3d.py with keras / csbdeep stubbed); _axes_div_by too"""
    import json, types
    import stardist_b200 as sd
    meta = json.load(open(os.path.join(golden_dir, "models_host.json")))
    tup = lambda kw: {k: (tuple(v) if isinstance(v, list) else v) for k, v in kw.items()}
    for i, (kw, want) in enumerate(meta["cfg2d"]):
        cfg = sd.Config2D(**tup(kw))
        assert _jsonable(vars(cfg)) == want, (kw, {k: (v, want.get(k)) for k, v in _jsonable(vars(cfg)).items() if want.get(k) != v})
        assert _jsonable(sd.StarDist2D._axes_div_by(types.SimpleNamespace(config=cfg), "YXC")) == meta["div_by"]["2d/%d" % i]
    for i, (kw, want) in enumerate(meta["cfg3d"]):
        k = tup(kw); n = k.pop("n_rays", 96)
        cfg = sd.Config3D(rays=sd.Rays_GoldenSpiral(n, anisotropy=k.get("anisotropy")), **k)
        assert _jsonable(vars(cfg)) == want, (kw, {a: (v, want.get(a)) for a, v in _jsonable(vars(cfg)).items() if want.get(a) != v})
        assert _jsonable(sd.StarDist3D._axes_div_by(types.SimpleNamespace(config=cfg), "ZYXC")) == meta["div_by"]["3d/%d" % i]


@needs_ref
def test_instances_from_prediction_glue_equals_reference_classes(golden_dir, monkeypatch):
    """StarDist2D / StarDist3D._instances_from_prediction (numpy-level glue: dense / sparse, grid, scale, multi-class) against
    the reference classes' own methods (tests/golden/models_host.npz).  The device-backed leaves are replaced by their pinned
    CPU equivalents: the C entry points by the reference extensions, dist_to_coord by the oracle's (== reference, hostfuncs.npz)."""
    import types
    import stardist_b200 as sd
    import stardist_b200.lib.stardist2d as l2, stardist_b200.lib.stardist3d as l3
    from stardist_b200.models import model2d as pm2
    monkeypatch.setattr(l2, "c_non_max_suppression_inds", ref_ext.stardist2d().c_non_max_suppression_inds)
    monkeypatch.setattr(l3, "c_non_max_suppression_inds", ref_ext.stardist3d().c_non_max_suppression_inds)
    monkeypatch.setattr(l3, "c_polyhedron_to_label", ref_ext.stardist3d().c_polyhedron_to_label)
    monkeypatch.setattr(pm2, "dist_to_coord", geom2d_np.dist_to_coord)
    g = np.load(os.path.join(golden_dir, "models_host.npz"))
    thr = types.SimpleNamespace(prob=0.9, nms=0.3)

    def same(res, prefix, keys):
        for k in keys:
            a, b = np.asarray(res[k]), g[prefix + k]
            assert a.shape == b.shape and np.array_equal(a, b), (prefix, k)

    shape, radius, noise, n_rays, grid, pthr, nthr, seed = cases.NMS2D_CASES["r32_356x299"]
    prob, dist = cases.create_random_data_2d(shape, radius, noise, n_rays, seed)
    fake = types.SimpleNamespace(config=types.SimpleNamespace(grid=(1, 1)), thresholds=thr)
    _, res = sd.StarDist2D._instances_from_prediction(fake, shape, prob, dist, return_labels=False)
    same(res, "2d/dense/", ("coord", "points", "prob"))
    fake2 = types.SimpleNamespace(config=types.SimpleNamespace(grid=(2, 2)), thresholds=thr)
    _, res = sd.StarDist2D._instances_from_prediction(fake2, shape, prob[::2, ::2], dist[::2, ::2], prob_class=g["2d/grid_scale_class/prob_class_in"],
                                                      return_labels=False, scale=dict(X=.5, Y=2.))
    same(res, "2d/grid_scale_class/", ("coord", "points", "prob", "class_prob", "class_id"))
    mask = prob > 0.92
    _, res = sd.StarDist2D._instances_from_prediction(fake, shape, prob[mask], dist[mask], points=np.stack(np.where(mask), 1),
                                                      prob_class=g["2d/sparse_class/prob_class_in"], nms_thresh=0.4, return_labels=False)
    same(res, "2d/sparse_class/", ("coord", "points", "prob", "class_prob", "class_id"))

    shape, noise, n_rays, pthr, nthr, seed, aniso = cases.NMS3D_CASES["r32_noise01_thr01"]
    prob, dist = cases.create_random_data_3d(shape, noise, n_rays, seed)
    rays = sd.Rays_GoldenSpiral(n_rays)
    fake3 = sd.StarDist3D.__new__(sd.StarDist3D)
    fake3.config = types.SimpleNamespace(grid=(1, 1, 1), rays_json=rays.to_json()); fake3.thresholds = dict(prob=float(pthr), nms=float(nthr))
    labels, res = sd.StarDist3D._instances_from_prediction(fake3, shape, prob, dist)
    assert labels.dtype == g["3d/dense/labels"].dtype and np.array_equal(labels, g["3d/dense/labels"])
    same(res, "3d/dense/", ("dist", "points", "prob"))
    mask = prob > pthr
    mask[:2] = mask[-2:] = False; mask[:, :2] = mask[:, -2:] = False; mask[:, :, :2] = mask[:, :, -2:] = False
    pts = np.stack(np.where(mask), 1).astype(np.float64)       # float points: the numpy-level path (integer points go to the device path)
    labels, res = sd.StarDist3D._instances_from_prediction(fake3, shape, prob[mask], dist[mask], points=pts, nms_thresh=0.2, scale=dict(Z=1., Y=.5, X=2.))
    assert np.array_equal(labels, g["3d/sparse_scale/labels"])
    same(res, "3d/sparse_scale/", ("dist", "points", "prob", "rays_vertices"))


def test_render_rule_differs_from_reference_only_on_exact_hull_facets():
    """DESIGN 5 (3-D labels): the product's rule kernel || polyhedron (host build of k_paint3d's rule) vs the reference's
    kernel || (hull && polyhedron) on lattice-aligned polyhedra: every differing voxel lies EXACTLY (rational arithmetic,
    tests/hullcheck.py) on a facet of the convex hull and is labelled by the product only -- no tolerance"""
    import ctypes, hullcheck
    from oracle import pipeline3d, ref_ext
    if not ref_ext.available():
        pytest.skip("oracle/_ref not built")
    so = os.path.join(ROOT, "tests", "hostcheck", "_build", "libhostcheck.so")
    if not os.path.exists(so):
        pytest.skip("hostcheck library not built")
    hc = ctypes.CDLL(so)
    hc.hc_paint3d.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int] * 5 + [ctypes.c_void_p]
    rng = np.random.default_rng(1)
    shape = (40, 44, 48)
    n_diff = 0
    for gen in (lambda n: np.full(n, rng.integers(4, 14)).astype(np.float32), lambda n: rng.integers(4, 14, n).astype(np.float32),
                lambda n: (rng.integers(8, 28, n) / 2).astype(np.float32)):
        for n_rays, aniso in ((32, None), (64, (2, 1, 1)), (96, None)):
            rays = cases.rays_golden_spiral(n_rays, aniso)
            v = np.ascontiguousarray(rays.vertices, np.float32); f = np.ascontiguousarray(rays.faces, np.int32)
            for _ in range(3):
                dist = gen(n_rays); point = np.array([rng.integers(14, 26), rng.integers(14, 30), rng.integers(14, 34)])
                d = np.ascontiguousarray(dist, np.float32); c = np.ascontiguousarray(point, np.float32); ours = np.zeros(shape, np.uint8)
                hc.hc_paint3d(d.ctypes.data, c.ctypes.data, v.ctypes.data, f.ctypes.data, len(v), len(f), shape[0], shape[1], shape[2], ours.ctypes.data)
                ref = pipeline3d.polyhedron_to_label(dist[None], point[None], rays, shape, np.ones(1))
                n_diff += hullcheck.assert_only_exact_hull_boundary_voxels_differ((ours > 0).astype(np.int32), (ref > 0).astype(np.int32), dist[None],
                                                                                  point[None].astype(np.float32), rays.vertices)
    assert n_diff > 0        # the lattice-aligned families do hit the caveat


def test_auto_named_keras_layers_are_bound_positionally():
    """tf.keras 2.x names un-named convolutions conv2d, conv2d_1, ... (session counter); checkpoints bind by order"""
    from stardist_b200 import Config2D, Config3D
    from stardist_b200.models.weights import glorot_uniform_weights, canonicalize_auto_names
    for cfg, pre in ((Config2D(grid=(2, 2)), 'conv2d'), (Config3D(backbone='resnet', grid=(1, 2, 2)), 'conv3d')):
        w = glorot_uniform_weights(cfg, seed=0)
        names = sorted([k for k in w if k.startswith(pre)], key=lambda s: int(s.split('_')[1]))
        for start in (0, 7):
            w2 = {k: v for k, v in w.items() if not k.startswith(pre)}
            for i, old in enumerate(names):
                w2[pre if (start + i) == 0 else '%s_%d' % (pre, start + i)] = w[old]
            c = canonicalize_auto_names(cfg, w2)
            assert all(np.array_equal(c[k][0], w[k][0]) for k in names)
        w3 = dict(w); w3.pop(names[0])
        with pytest.raises(ValueError):
            canonicalize_auto_names(cfg, w3)


def test_fan_bounds_bracket_the_volumes_they_replace():
    """the ray-fan bounds that decide the S3 / S4 comparisons of the 3-D NMS without the exact volume (nms3d.cu fan_bounds,
    serial definition in nms3d_pair.cuh): lower <= volume <= upper for kernel and hull intersections of random polyhedron
    pairs -- 16 ... 187 rays, anisotropic rays, noise up to 0.6 -- on the coarse and on the refined fan"""
    so = os.path.join(ROOT, "tests", "hostcheck", "_build", "libhostcheck.so")
    if not os.path.exists(so):
        pytest.skip("hostcheck library not built")
    hc = ctypes.CDLL(so)
    P = ctypes.c_void_p
    hc.hc_fan_bounds_pair.argtypes = [P, P, P, P, P, P, ctypes.c_int, ctypes.c_int, P]
    rng = np.random.default_rng(0)
    n_poly, n_incl, ratios = 0, 0, []
    for n_rays, aniso in ((32, None), (96, (2, 1, 1)), (64, (1, 1.5, 3)), (187, None), (16, None)):
        rays = cases.rays_golden_spiral(n_rays, aniso)
        v = np.ascontiguousarray(rays.vertices, np.float32); f = np.ascontiguousarray(rays.faces, np.int32)
        for _ in range(40):
            r = rng.uniform(4, 12); noise = rng.choice([0.0, 0.1, 0.3, 0.6])
            d1 = (r * (1 + noise * rng.uniform(-1, 1, n_rays))).astype(np.float32)
            d2 = (r * rng.uniform(0.7, 1.3) * (1 + noise * rng.uniform(-1, 1, n_rays))).astype(np.float32)
            c1 = rng.integers(10, 40, 3).astype(np.float32); c2 = (c1 + rng.integers(-6, 7, 3)).astype(np.float32)
            pv1 = (c1[None] + d1[:, None] * v).astype(np.float32); pv2 = (c2[None] + d2[:, None] * v).astype(np.float32)
            out = np.zeros(12)
            hc.hc_fan_bounds_pair(pv1.ctypes.data, c1.ctypes.data, pv2.ctypes.data, c2.ctypes.data, v.ctypes.data, f.ctypes.data, n_rays, len(f), out.ctypes.data)
            if out[0] == 1 and out[6] == 1:
                # the stage order of the device cascade (S4 before S3) rests on kernel_1 ∩ kernel_2 ⊂ hull_1 ∩ hull_2; the two
                # volumes are rounded independently, the device allows 1e-4 relative between them
                n_incl += 1
                assert out[1] <= out[7] * (1 + 1e-6) + 1e-9, (n_rays, out[1], out[7])
            for base in (0, 6):
                if out[base] != 1: continue
                n_poly += 1
                V, lo, up, lo2, up2 = out[base + 1:base + 6]
                for L_, U_ in ((lo, up), (lo2, up2)):
                    assert L_ <= V * (1 + 1e-9) + 1e-12, (n_rays, base, L_, V)
                    assert U_ >= V * (1 - 1e-9) - 1e-12, (n_rays, base, U_, V)
                assert lo2 >= lo * (1 - 1e-9)                      # the refined fan contains the coarse one
                if up2 < 1e299 and V > 0: ratios.append((lo2 / V, up2 / V))
    assert n_poly > 250 and n_incl > 50
    r = np.array(ratios)
    assert np.median(r[:, 0]) > 0.85 and np.median(r[:, 1]) < 1.15      # and they are tight enough to decide most pairs


def test_direction_bins_list_every_face_that_can_contain_the_direction():
    """the direction bins of the 3-D rendering and of the S5 rule (bins3d.cuh; k_build_bins calls the same bin_takes_face,
    the voxel loop the same bin_of): for any direction u from the centre, every face whose cone contains u -- with a slack of
    1e-3 in the barycentric coordinates, ~1000 x what float rounding of inside_tetrahedron can move -- is in the list of u's bin,
    so the binned OR over tetrahedra is the OR over all of them.  Random directions plus the degenerate ones: the axes, the
    cube-map cell borders and diagonals, the ray directions themselves and their edge midpoints."""
    so = os.path.join(ROOT, "tests", "hostcheck", "_build", "libhostcheck.so")
    if not os.path.exists(so):
        pytest.skip("hostcheck library not built")
    hc = ctypes.CDLL(so)
    if not hasattr(hc, "hc_bin_takes_face"):
        pytest.skip("hostcheck library predates the bins check")
    P = ctypes.c_void_p
    hc.hc_bin_of.argtypes = [ctypes.c_float] * 3
    hc.hc_bin_takes_face.argtypes = [ctypes.c_int, P, P, ctypes.c_int]
    n_bins = hc.hc_bin_count()
    rng = np.random.default_rng(1)
    sizes = []
    from stardist_b200 import rays3d as R3
    ray_sets = [(n, a, cases.rays_golden_spiral(n, a)) for n, a in ((96, (2, 1, 1)), (32, None), (64, (1, 1.5, 3)), (187, None), (16, None), (8, (4, 1, 1)))]
    ray_sets += [(0, "cartesian", R3.Rays_Cartesian(8, 5)), (0, "cartesian11", R3.Rays_Cartesian(11, 5)), (0, "octo", R3.Rays_Octo(3))]
    for n_rays, aniso, rays in ray_sets:
        v = np.ascontiguousarray(rays.vertices, np.float32); f = np.ascontiguousarray(rays.faces, np.int32)
        n_rays = len(v)
        takes = np.array([[hc.hc_bin_takes_face(b, v.ctypes.data, f.ctypes.data, j) for j in range(len(f))] for b in range(n_bins)], bool)
        sizes.append(takes.sum(1).max())
        u = rng.normal(size=(20000, 3))
        g = np.linspace(-1, 1, 9)                                     # cube-map cell borders (BIN_B = 4) and centres
        cube = np.array([np.roll([s, a, b], k) for s in (-1, 1) for a in g for b in g for k in range(3)], float)
        vd = v.astype(np.float64)
        mids = np.concatenate([vd[f[:, i]] + vd[f[:, (i + 1) % 3]] for i in range(3)])
        u = np.concatenate([u, cube, vd, -vd, mids, vd[f].sum(1), np.eye(3), -np.eye(3)]).astype(np.float32)
        u = u[np.abs(u).max(1) > 0]
        bins = np.array([hc.hc_bin_of(*map(float, w)) for w in u])
        assert bins.min() >= 0 and bins.max() < n_bins
        A, B, C = (vd[f[:, i]] for i in range(3))                     # [F,3]
        det = np.einsum("fi,fi->f", A, np.cross(B, C))
        ud = u.astype(np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            al = np.einsum("ni,fi->nf", ud, np.cross(B, C)) / det
            be = np.einsum("ni,fi->nf", ud, np.cross(C, A)) / det
            ga = np.einsum("ni,fi->nf", ud, np.cross(A, B)) / det
        s = np.abs(al) + np.abs(be) + np.abs(ga)
        un = vd / np.linalg.norm(vd, axis=1, keepdims=True)
        flat = np.abs(np.einsum("fi,fi->f", un[f[:, 0]], np.cross(un[f[:, 1]], un[f[:, 2]]))) < 1e-7      # degenerate face (Cartesian poles)
        # a degenerate face's tetrahedron "contains" a whole plane through the centre (all determinants vanish there and the
        # reference tests det >= 0): it must be in EVERY bin
        assert takes[:, flat].all()
        with np.errstate(divide="ignore", invalid="ignore"):
            in_cone = (np.minimum(np.minimum(al, be), ga) >= -1e-3 * s) & ~flat[None]
        listed = takes[bins]                                          # [n,F]
        missing = in_cone & ~listed
        assert not missing.any(), (n_rays, aniso, np.argwhere(missing)[:5])
        assert in_cone.any(1).mean() > 0.99                           # the triangulation covers the sphere: the check is not vacuous
    assert max(sizes) <= 64                                           # BIN_CAP: no list overflows for the ray sets in use


def test_halfspace_volume_is_exact_for_many_rays():
    """volume of hull_1 ∩ hull_2 (stage S4 of the 3-D NMS; geom3d.cuh face_cone_volume on the facets of convex_hull_planes)
    against scipy's Qhull (HalfspaceIntersection + ConvexHull) for 128 / 187 / 256 rays.  Clipping a facet against the other
    planes in index order lets the intermediate polygon pass the fixed vertex capacity (the facets come out of the gift
    wrapping as a growing patch); such a facet is clipped again in a scattered order.  Before that, 30 % of these volumes
    were 1e-5 ... 4e-3 too small (silently); now: no overflow, relative error < 1e-9."""
    from scipy.spatial import ConvexHull, HalfspaceIntersection
    so = os.path.join(ROOT, "tests", "hostcheck", "_build", "libhostcheck.so")
    if not os.path.exists(so):
        pytest.skip("hostcheck library not built")
    hc = ctypes.CDLL(so)
    if not hasattr(hc, "hc_planes_volume"):
        pytest.skip("hostcheck library predates the volume entry")
    P = ctypes.c_void_p
    hc.hc_convex_hull_planes.argtypes = [P, ctypes.c_int, P, ctypes.c_int]
    hc.hc_planes_volume.argtypes = [P, ctypes.c_int, P, ctypes.c_double, P, P]; hc.hc_planes_volume.restype = ctypes.c_double
    rng = np.random.default_rng(3)
    n_checked = 0
    for n_rays in (128, 187, 256):
        v = np.ascontiguousarray(cases.rays_golden_spiral(n_rays, None).vertices, np.float32)
        for _ in range(24):
            r = rng.uniform(4, 12); noise = rng.choice([0.0, 0.0, 0.05, 0.2])
            c1 = rng.integers(10, 40, 3).astype(np.float64); c2 = c1 + rng.integers(-6, 7, 3)
            planes = []
            for c, scale in ((c1, 1.0), (c2, rng.uniform(0.7, 1.3))):
                d = (r * scale * (1 + noise * rng.uniform(-1, 1, n_rays))).astype(np.float32)
                pts = np.ascontiguousarray((c[None].astype(np.float32) + d[:, None] * v).astype(np.float32), np.float64)
                out = np.zeros((512, 4))
                nf = hc.hc_convex_hull_planes(pts.ctypes.data, n_rays, out.ctypes.data, 512)
                assert nf == len(ConvexHull(pts).simplices)
                planes.append(out[:nf].copy()); ext = np.abs(pts).max()
            pl = np.ascontiguousarray(np.concatenate(planes))
            p = 0.5 * (c1 + c2)
            if (pl[:, :3] @ p + pl[:, 3]).max() >= -1e-6:
                continue                                              # the midpoint is not inside both hulls: S4 is not evaluated
            ovf = ctypes.c_int(0)
            vol = hc.hc_planes_volume(pl.ctypes.data, len(pl), p.ctypes.data, 4.0 * 64 + 1.0, None, ctypes.byref(ovf))
            want = ConvexHull(HalfspaceIntersection(pl, p).intersections).volume
            assert ovf.value == 0
            assert abs(vol - want) <= 1e-9 * want, (n_rays, vol, want)
            n_checked += 1
    assert n_checked >= 40


def overlap_pairs():
    """polyhedron pairs of test_volume_stages_equal_the_reference_qhull_functions: (n_rays, noise, ctypes arguments, arrays)"""
    P = ctypes.c_void_p
    rng = np.random.default_rng(1)
    for n_rays, aniso, noise, n_pairs in ((96, (2, 1, 1), 0.2, 60), (187, None, 0.0, 40), (256, None, 0.02, 30), (128, None, 0.05, 30)):
        rays = cases.rays_golden_spiral(n_rays, aniso)
        v = np.ascontiguousarray(rays.vertices, np.float32); f = np.ascontiguousarray(rays.faces, np.int32)
        for _ in range(n_pairs):
            c1 = rng.uniform(20, 60, 3).astype(np.float32); c2 = (c1 + rng.uniform(-8, 8, 3)).astype(np.float32)
            d1 = (10 * (1 + noise * rng.uniform(-1, 1, n_rays))).astype(np.float32)
            d2 = (10 * rng.uniform(0.8, 1.2) * (1 + noise * rng.uniform(-1, 1, n_rays))).astype(np.float32)
            pv1 = (c1[None] + d1[:, None] * v).astype(np.float32); pv2 = (c2[None] + d2[:, None] * v).astype(np.float32)
            a = (P(pv1.ctypes.data), P(c1.ctypes.data), P(pv2.ctypes.data), P(c2.ctypes.data), P(f.ctypes.data), n_rays, len(f))
            yield n_rays, noise, a, (pv1, c1, pv2, c2, f)


def test_volume_stages_equal_the_reference_qhull_functions(golden_dir):
    """S3 / S4 volumes of the Qhull-free routines (nms3d_pair.cuh, host build of the device headers) against the reference's own
    qhull_overlap_kernel / qhull_overlap_convex_hulls (stardist3d_impl.cpp:676-735,880-935, compiled unmodified into
    oracle/_ref/libsdref.so; their values: tests/golden/refshim.npz, make_refshim.py): the float the NMS compares is the same,
    incl. near-spherical polyhedra with 187 / 256 rays (every facet on the hull -- the case that overflowed the polygon buffer
    before the scattered re-clip)."""
    hc = _hostcheck()
    for f in (hc.hc_overlap_kernel, hc.hc_overlap_convex):
        f.restype = ctypes.c_float
    ref = np.load(os.path.join(golden_dir, "refshim.npz"))["overlap"]
    total = equal = 0
    for i, (n_rays, noise, a, _) in enumerate(overlap_pairs()):
        for want, got in ((ref[i, 0], hc.hc_overlap_kernel(*a)), (ref[i, 1], hc.hc_overlap_convex(*a[:4], n_rays))):
            assert (want >= 1e9) == (got >= 1e9) and (want == 0) == (got == 0), (n_rays, want, got)
            if want < 1e9:
                assert abs(want - got) <= 1e-6 * abs(want), (n_rays, noise, want, got)
            total += 1; equal += int(np.float32(want).view(np.int32) == np.float32(got).view(np.int32))
    assert total == 2 * len(ref) == 320 and equal >= 0.99 * total, (equal, total)


def test_ctypes_signatures_match_the_header():
    """include/stardist_b200.h is the boundary; stardist_b200/_lib.py is the binding a consumer would write.  extern "C" symbols
    carry no types, so a float / double or a missing-argument slip between the two would pass silently: compare, for every
    prototype, the parameter classes (pointer / i32 / i64 / f32 / f64) and the return class with the ctypes declaration.
    (The .cu files include the header, so the definitions themselves are checked by the compiler.)"""
    lib_path = os.path.join(ROOT, "stardist_b200", "libstardist_b200.so")
    if not os.path.exists(lib_path):
        pytest.skip("libstardist_b200.so not built")
    from stardist_b200 import _lib
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "stardist_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S); hdr = re.sub(r"//[^\n]*", "", hdr)
    protos = re.findall(r"([\w\s\*]+?)\b((?:sdb_|_LIB_)\w+)\s*\(([^)]*)\)\s*;", hdr, flags=re.S)

    def cls_c(p):
        p = " ".join(p.split())
        if p in ("void", ""): return None
        if "*" in p or "sdb_stream_t" in p: return "ptr"
        if re.search(r"\bdouble\b", p): return "f64"
        if re.search(r"\bfloat\b", p): return "f32"
        if re.search(r"long long|int64_t|size_t", p): return "i64"
        return "i32"

    def cls_py(t):
        if t in (ctypes.c_void_p, ctypes.c_char_p) or (isinstance(t, type) and issubclass(t, ctypes._Pointer)): return "ptr"
        return {ctypes.c_double: "f64", ctypes.c_float: "f32", ctypes.c_longlong: "i64", ctypes.c_ulonglong: "i64", ctypes.c_size_t: "i64",
                ctypes.c_int: "i32", ctypes.c_uint: "i32", ctypes.c_bool: "i32"}.get(t, str(t))

    checked, bad = 0, []
    for ret, name, params in protos:
        fn = getattr(lib, name)
        if fn.argtypes is None:
            continue                                   # bound lazily by the module that mirrors the reference extension
        want = [c for c in (cls_c(p) for p in params.split(",")) if c]
        got = [cls_py(t) for t in fn.argtypes]
        r = " ".join(ret.replace("extern", "").split())
        want_r = None if (r.endswith("void") and "*" not in r) else cls_c(r)
        got_r = None if fn.restype is None else cls_py(fn.restype)
        checked += 1
        if want != got or want_r != got_r:
            bad.append((name, want, got, want_r, got_r))
    assert checked >= 60 and not bad, bad


def test_frontier_peeling_model_equals_the_greedy_loop():
    """The device NMS (2-D: nms2d_rounds.cuh d_frontier2 / d_pairs / d_fast / d_clip; 3-D: nms3d.cu k_frontier / k_pretest /
    k_heavy) replaces the reference's serial greedy loop (stardist2d.cpp:520-600, stardist3d_impl.cpp:1120-1360) by rounds:
    an undecided candidate c is KEPT in round r unless some h < c (higher score) that reaches c is still undecided or was kept
    in this very round (whatever a racing read of state[h] returns among the values it can hold during the launch); the
    candidates kept in round r then test the undecided c > h they reach and suppress those that overlap.  This is a model of
    exactly that rule on random 'reach' / 'overlap' relations -- with the racy reads modelled by evaluating the candidates of a
    round in random order against a state array that changes under them -- against the greedy loop: same keep mask, always,
    and the lowest undecided index is never blocked (progress)."""
    rng = np.random.default_rng(0)
    for trial in range(200):
        n = int(rng.integers(1, 120))
        reach = np.triu(rng.random((n, n)) < rng.choice([0.02, 0.1, 0.4, 1.0]), 1)          # reach[h, c], h < c
        overlap = reach & (rng.random((n, n)) < rng.choice([0.1, 0.5, 0.9]))              # suppresses only what it reaches
        # reference: greedy in score order
        sup = np.zeros(n, bool)
        for i in range(n):
            if sup[i]: continue
            sup[i + 1:] |= overlap[i, i + 1:]
        want = ~sup
        UNDECIDED, SUPPRESSED = 0, 1
        state = np.zeros(n, int)
        rounds = 0
        while (state == UNDECIDED).any():
            kept_now = 2 + rounds
            und = np.flatnonzero(state == UNDECIDED)
            kept = []
            for c in rng.permutation(und):                         # racing warps: any order, state changes under them
                hs = np.flatnonzero(reach[:c, c])
                blocked = any(state[h] == UNDECIDED or state[h] == kept_now for h in hs)
                if not blocked:
                    state[c] = kept_now; kept.append(c)
            assert und.min() in kept                               # progress: the best undecided candidate is never blocked
            for h in kept:                                         # pair tests of this round (any order: they only suppress)
                cs = np.flatnonzero(overlap[h] & (state == UNDECIDED))
                state[cs] = SUPPRESSED
            rounds += 1
            assert rounds <= n
        assert np.array_equal(state >= 2, want), trial


def test_serial_nms3d_other_ray_classes_equal_reference():
    """the 3-D NMS arithmetic (host build of the device headers, hc_nms3d_serial) against the reference extension for the ray
    classes beyond Rays_GoldenSpiral: Rays_Cartesian (pole rings = groups of coincident directions, zero-area pole faces),
    Rays_Octo, Rays_Tetra -- same keep mask, incl. the constant-distance clouds where the coincident rays give DUPLICATE
    vertices (Qhull ignores them; the gift wrapping needs demote_duplicate_points, geom3d.cuh -- before that fix S4 never
    short-cut for such polyhedra and 50 of 600 decisions differed).  Subprocess with OMP_NUM_THREADS=1 (the reference's
    anisotropy sum races)."""
    code = r'''
import ctypes, json, os, sys, numpy as np
ROOT = sys.argv[1]
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from oracle import ref_ext
from stardist_b200 import rays3d as R3
hc = ctypes.CDLL(os.path.join(ROOT, "tests/hostcheck/_build/libhostcheck.so")); P = ctypes.c_void_p
hc.hc_nms3d_serial.argtypes = [P, P, P, P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_int, P, P]
out = []
for k, (name, rays) in enumerate([("cartesian", R3.Rays_Cartesian(8, 5)), ("octo", R3.Rays_Octo(2)), ("tetra", R3.Rays_Tetra(2)), ("octo3", R3.Rays_Octo(3))]):
    v = np.ascontiguousarray(rays.vertices, np.float32); f = np.ascontiguousarray(rays.faces, np.int32); R = len(v)
    for noise, nthr in ((0.2, 0.2), (0.5, 0.5), (0.0, 0.3)):
        rng = np.random.default_rng(100 * k + int(10 * noise)); n = 300
        p = np.ascontiguousarray(np.stack([rng.integers(2, s - 2, n) for s in (14, 18, 20)], 1), np.float32)
        s = np.ascontiguousarray(np.sort(rng.uniform(0.5, 1, n))[::-1], np.float32)
        d = np.ascontiguousarray(rng.uniform(2, 5, (n, 1)) * (1 + noise * rng.uniform(-1, 1, (n, R))), np.float32)
        want = ref_ext.stardist3d().c_non_max_suppression_inds(d, p, v, f, s, 1, 1, 0, np.float32(nthr))
        keep = np.zeros(n, np.uint8); sc = np.zeros(5, np.int32)
        hc.hc_nms3d_serial(d.ctypes.data, p.ctypes.data, v.ctypes.data, f.ctypes.data, n, R, len(f), ctypes.c_float(nthr), 1, 1, 0, keep.ctypes.data, sc.ctypes.data)
        out.append(dict(rays=name, noise=noise, kept=int(want.sum()), mismatches=int(np.count_nonzero(keep.astype(bool) != want)), s4=int(sc[3]), s5=int(sc[4])))
print("RESULT " + json.dumps(out))
'''
    so = os.path.join(ROOT, "tests", "hostcheck", "_build", "libhostcheck.so")
    if not (os.path.exists(so) and ref_ext.available()):
        pytest.skip("hostcheck / oracle/_ref not built")
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, "-c", code, ROOT], capture_output=True, text=True, env=env, timeout=900)
    lines = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert lines, r.stderr[-2000:]
    res = json.loads(lines[-1][7:])
    assert len(res) == 12
    for e in res:
        assert e["mismatches"] == 0, e
    cart0 = [e for e in res if e["rays"] == "cartesian" and e["noise"] == 0.0][0]
    assert cart0["s5"] < cart0["s4"], cart0          # duplicate vertices: S4 decides pairs again instead of passing all to S5


def test_rendering_rule_vs_reference_all_modes_and_ray_classes():
    """the DEFINING per-voxel rule of the device rendering (label3d.cu k_paint3d without its result-neutral short cuts; serial
    host build, hc_polyhedron_to_label) against the reference's c_polyhedron_to_label for render modes full / kernel / hull /
    bbox and the ray classes golden spiral, Octo, Tetra, Cartesian:
      * centres off the lattice: every mode, every ray class -- identical label volumes;
      * integer centres and half-integer radii (voxels exactly ON facets): kernel and bbox identical; full and hull differ on a
        handful of voxels (the hull-facet class of DESIGN.md §5: < 0.2 % of the labelled voxels);
      * Rays_Cartesian: its zero-area pole faces span degenerate tetrahedra that "contain" whole planes through the centre;
        without a hull test they were painted across the bounding box (5 268 of 12 120 voxels wrong on the lattice).  For ray
        sets with such faces the rule applies the reference's hull conjunct (gift-wrapping facets): same bounds as the others."""
    so = os.path.join(ROOT, "tests", "hostcheck", "_build", "libhostcheck.so")
    if not (os.path.exists(so) and ref_ext.available()):
        pytest.skip("hostcheck / oracle/_ref not built")
    hc = ctypes.CDLL(so)
    if not hasattr(hc, "hc_polyhedron_to_label"):
        pytest.skip("hostcheck library predates the rendering entry")
    from stardist_b200 import rays3d as R3
    P = ctypes.c_void_p
    hc.hc_polyhedron_to_label.argtypes = [P, P, P, P, ctypes.c_int, ctypes.c_int, ctypes.c_int, P] + [ctypes.c_int] * 4 + [P]
    ext = ref_ext.stardist3d()
    shape = (32, 40, 44)

    def diff(rays, noise, lattice, seed, n=16):
        v = np.ascontiguousarray(rays.vertices, np.float32); f = np.ascontiguousarray(rays.faces, np.int32); R = len(v)
        rng = np.random.default_rng(seed)
        if lattice:
            p = np.stack([rng.integers(6, s - 6, n) for s in shape], 1)
            d = np.round(rng.uniform(3, 7, (n, 1)) * 2) / 2 * (1 + noise * rng.uniform(-1, 1, (n, R)))
        else:
            p = np.stack([rng.uniform(6, s - 6, n) for s in shape], 1)
            d = rng.uniform(3, 7, (n, 1)) * (1 + noise * rng.uniform(-1, 1, (n, R)))
        d = np.ascontiguousarray(d, np.float32); p = np.ascontiguousarray(p, np.float32)
        labels = np.arange(1, n + 1, dtype=np.int32)
        out = []
        for mode in (0, 1, 2, 3):
            want = ext.c_polyhedron_to_label(d, p, v, f, labels, mode, 0, 0, 0, shape)
            got = np.zeros(shape, np.int32)
            hc.hc_polyhedron_to_label(d.ctypes.data, p.ctypes.data, v.ctypes.data, f.ctypes.data, n, R, len(f), labels.ctypes.data, *shape, mode, got.ctypes.data)
            out.append((int((want != got).sum()), int((want > 0).sum())))
        return out

    sets = [("golden", cases.rays_golden_spiral(96, (2, 1, 1))), ("golden32", cases.rays_golden_spiral(32, None)), ("octo", R3.Rays_Octo(3)),
            ("tetra", R3.Rays_Tetra(2)), ("cartesian", R3.Rays_Cartesian(8, 5))]
    for k, (name, rays) in enumerate(sets):
        for noise in (0.0, 0.3):
            r = diff(rays, noise, False, 10 * k + 1)
            assert all(nd == 0 for nd, _ in r), (name, noise, r)                       # off the lattice: identical, all modes
            r = diff(rays, noise, True, 10 * k + 2)
            (d_full, n_full), (d_ker, _), (d_hull, n_hull), (d_box, _) = r
            assert d_ker == 0 and d_box == 0, (name, noise, r)
            assert d_hull <= 0.002 * n_hull + 2, (name, noise, r)
            assert d_full <= 0.002 * n_full + 2, (name, noise, r)


def test_warp_gift_wrapping_model_with_demoted_duplicates():
    """lane-by-lane model of the device hull routine (nms3d.cu hull_planes_warp / warp_pivot: lane-strided scan, xor-shuffle
    tournament with a deterministic comparison, edge bookkeeping, guard) on point sets as the device sees them for
    Rays_Cartesian -- duplicate vertices moved to the centroid by demote_duplicate_points, several copies of that interior
    point included, or collinear pole points -- against scipy's hull of the distinct points: same volume, no give-up.
    (The serial routine of geom3d.cuh is compared with the reference directly; this covers the warp formulation, which exists
    only as device code.)"""
    from scipy.spatial import ConvexHull
    from stardist_b200 import rays3d as R3

    def orient(P,a,b,c,d):
        B=P[b]-P[a]; C=P[c]-P[a]; D=P[d]-P[a]
        return D[0]*(B[1]*C[2]-B[2]*C[1]) + D[1]*(B[2]*C[0]-B[0]*C[2]) + D[2]*(B[0]*C[1]-B[1]*C[0])
    def warp_pivot(P,n,a,b,skip):
        q=[-1]*32
        for lane in range(32):
            for r in range(lane,n,32):
                if r==a or r==b or r==skip: continue
                if q[lane]<0: q[lane]=r; continue
                if orient(P,a,b,q[lane],r)>0: q[lane]=r
        o=16
        while o>0:
            nq=list(q)
            for lane in range(32):
                other=q[lane^o]; best=q[lane]
                if q[lane]<0: best=other
                elif other>=0 and other!=q[lane]:
                    lo,hi=min(q[lane],other),max(q[lane],other)
                    best = hi if orient(P,a,b,lo,hi)>0 else lo
                nq[lane]=best
            q=nq; o>>=1
        assert len(set(q))==1
        return q[0]
    def demote(P):
        P=P.copy(); c=P.mean(0); n=len(P)   # (device sums sequentially; value differences irrelevant here)
        for i in range(n-1,0,-1):
            if any((P[j]==P[i]).all() for j in range(i)): P[i]=c
        return P
    def hull_warp(P):
        n=len(P)
        p0=0
        for i in range(1,n):
            if tuple(P[i])<tuple(P[p0]): p0=i
        p1=-1
        for i in range(n):
            if i==p0: continue
            if p1<0: p1=i; continue
            ax,ay=P[p1][0]-P[p0][0],P[p1][1]-P[p0][1]; bx,by=P[i][0]-P[p0][0],P[i][1]-P[p0][1]
            cr=ax*by-ay*bx
            if cr<0 or (cr==0 and bx*bx+by*by>ax*ax+ay*ay): p1=i
        p2=warp_pivot(P,n,p0,p1,-1)
        done=set(); facets=[]; stack=[]
        def emit(a,b,c):
            facets.append((a,b,c)); done.update([(a,b),(b,c),(c,a)])
        emit(p0,p1,p2); stack+= [(p1,p0,p2),(p2,p1,p0),(p0,p2,p1)]
        guard=0
        while stack:
            guard+=1
            if guard>16*n+64: return None
            a,b,opp=stack.pop()
            if (a,b) in done: continue
            q=warp_pivot(P,n,a,b,opp)
            if q<0: return None
            emit(a,b,q)
            if (q,b) not in done: stack.append((q,b,a))
            if (a,q) not in done: stack.append((a,q,b))
        return facets

    rng = np.random.default_rng(0)
    for rays in (R3.Rays_Cartesian(8, 5), R3.Rays_Cartesian(11, 5)):
        v = rays.vertices.astype(np.float32)
        for it in range(6):
            c = rng.integers(5, 40, 3).astype(np.float32)
            d = (rng.uniform(2, 6) * (1 + 0.3 * rng.uniform(-1, 1, len(v)))).astype(np.float32)
            if it % 3 == 0: d[:] = d[0]                      # equal everywhere: duplicates at both poles
            elif it % 3 == 2: d[:4] = d[0]                   # some duplicates, some collinear points
            P = (c[None] + d[:, None] * v).astype(np.float32).astype(np.float64)
            Pd = demote(P)
            F = hull_warp(Pd)
            assert F is not None, (len(v), it)
            want = ConvexHull(np.unique(P, axis=0)).volume
            vol = abs(sum(np.dot(Pd[a], np.cross(Pd[b], Pd[c_])) for a, b, c_ in F)) / 6
            assert abs(vol - want) <= 1e-9 * want, (len(v), it, vol, want)
