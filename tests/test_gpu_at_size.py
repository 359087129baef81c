"""Parity at the sizes BASELINE.json names (pytest -m gpu): the product path against the oracle on the benchmark's own
inputs -- integer results (survivor indices, polygons' integer centres, label maps) bit-equal.  The network maps are taken
from the product (cand_from=model) so that the integer post-processing is compared on identical floats; the maps themselves
are covered by the float-tolerance tests.  The oracle here is the reference's compiled C++ (oracle/_ref) + the numpy glue
pinned against the reference's Python modules."""
import hashlib, json, os, sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import cases
from oracle import ref_ext, nms_np, pipeline2d, pipeline3d

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sd():
    import stardist_b200
    from stardist_b200 import _lib
    _lib.require_cuda()
    return stardist_b200


def _same_partition(a, b):
    if not np.array_equal(a > 0, b > 0): return False
    pairs = np.unique(np.stack([a[a > 0], b[a > 0]], 1), axis=0)
    return len(pairs) == len(np.unique(a[a > 0])) == len(np.unique(b[b > 0]))


def _relabel_by(a, b):
    """b with its ids renamed to a's by majority vote"""
    pairs, counts = np.unique(np.stack([b[b > 0], a[b > 0]], 1), axis=0, return_counts=True)
    order = np.argsort(counts)
    lut = np.zeros(int(b.max()) + 1, a.dtype)
    lut[pairs[order, 0]] = pairs[order, 1]
    return lut[b]


def test_bench_image_1024_equals_oracle(sd):
    """configs[1]: the bench image (1024x1024, ~140 k candidates, ~190 k pair tests, ~1.1 k instances)"""
    if not ref_ext.available(): pytest.skip("oracle/_ref not present")
    import bench_data
    cfg = sd.Config2D(n_rays=32)
    model = sd.StarDist2D(cfg, name=None, basedir=None, weights=bench_data.bench_weights_2d(cfg))
    for seed in (0, 1):
        img, _ = bench_data.synthetic_image((1024, 1024), seed=seed)
        labels, res = model.predict_instances(img, prob_thresh=0.5, nms_thresh=0.4)
        ref_labels, ref = pipeline2d.predict_instances(cfg, model.weights, img, 0.5, 0.4, cand_from=model)
        assert len(ref['prob']) > 900
        assert np.array_equal(res['points'], ref['points']) and np.array_equal(res['prob'], ref['prob'])
        assert np.array_equal(res['coord'].view(np.int32), ref['coord'].view(np.int32))
        assert np.array_equal(labels, ref_labels)


def test_big_4096_equals_whole_image_and_oracle(sd):
    """predict_instances_big on 4096x4096 with 2048-blocks: the assembled result is the whole-image result up to the
    numbering of the ids (the reference's own criterion, tests/test_big.py:87-120), and the whole-image result is the oracle's"""
    if not ref_ext.available(): pytest.skip("oracle/_ref not present")
    import bench_data
    cfg = sd.Config2D(n_rays=32)
    model = sd.StarDist2D(cfg, name=None, basedir=None, weights=bench_data.bench_weights_2d(cfg))
    tile, _ = bench_data.synthetic_image((1024, 1024), seed=0)
    img = np.tile(tile, (4, 4))
    lb, pb = model.predict_instances_big(img, axes='YX', block_size=2048, min_overlap=128, context=96, show_progress=False)
    labels, res = model.predict_instances(img, prob_thresh=0.5, nms_thresh=0.4)
    ref_labels, ref = pipeline2d.predict_instances(cfg, model.weights, img, 0.5, 0.4, cand_from=model)
    assert np.array_equal(labels, ref_labels) and np.array_equal(res['points'], ref['points'])
    assert len(pb['prob']) == len(res['prob']) > 15000
    i, j = np.lexsort(tuple(res['points'].T)), np.lexsort(tuple(pb['points'].T))
    assert np.array_equal(res['points'][i], pb['points'][j]) and np.array_equal(res['prob'][i], pb['prob'][j])
    assert np.allclose(res['coord'][i], pb['coord'][j], atol=1e-2)      # block-local coordinates + origin vs global: float rounding (reference: atol 1e-2)
    # same objects; pixels shared by two overlapping polygons of different blocks go to the block written last
    # (big.py:319-326) instead of the higher score -- the reference's criterion (tests/test_big.py:104-105) is matching at 0.99
    # (a block renders its polygons in block-local float32 coordinates: a pixel centre within ~1e-4 of an edge can fall on the
    # other side than in global coordinates -- a few pixels in 10^7)
    assert np.mean((labels > 0) != (lb > 0)) < 1e-5
    from stardist_b200.matching import matching
    m = matching(labels, lb, thresh=0.99)
    assert m.accuracy == 1.0 and m.mean_true_score > 0.9999
    assert np.mean(_relabel_by(labels, lb) != labels) < 1e-4


def test_volume_3d_equals_oracle(sd):
    """configs[2] at 128x256x256 (~80 k candidates through the 3-D NMS cascade): survivors and the relabelled volume"""
    if not ref_ext.available(): pytest.skip("oracle/_ref not present")
    import bench_data
    from stardist_b200.rays3d import rays_from_json
    cfg = bench_data.bench_config_3d(96)
    model = sd.StarDist3D(cfg, name=None, basedir=None, weights=bench_data.bench_weights_3d(cfg))
    vol, _ = bench_data.synthetic_volume((128, 256, 256), seed=0, cell=(64, 256, 256))
    labels, res = model.predict_instances(vol, prob_thresh=0.7, nms_thresh=0.3)
    rays = rays_from_json(cfg.rays_json)
    # the reference's 32 MB label volume is too large to replay: tests/golden/at_size_3d.json holds the sha256 of its int32
    # bytes and its label count; where oracle/_ref is built the reference's volume is compared in full and against the digest
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "at_size_3d.json")))
    digest = lambda a: hashlib.sha256(np.ascontiguousarray(a, np.int32).tobytes()).hexdigest()
    if ref_ext.built():
        ref_labels, ref = pipeline3d.predict_instances(cfg, rays, vol, 0.7, 0.3, cand_from=model)
        assert digest(ref_labels) == golden["labels_sha256"] and ref_labels.max() == golden["n_labels"]
        assert np.array_equal(labels, ref_labels)
    else:
        prob, dist = model._last_maps()
        proba, dista, points = pipeline3d.candidates(cfg, prob, dist, vol.shape, 0.7)
        points, probi, disti, _ = nms_np.non_maximum_suppression_3d_sparse(dista, proba, points, rays, nms_thresh=0.3)
        ref = dict(points=points, prob=probi, dist=disti)
        assert labels.shape == tuple(golden["shape"]) and labels.max() == golden["n_labels"]
        assert digest(labels) == golden["labels_sha256"]
    assert len(ref['prob']) > 2000
    assert np.array_equal(res['points'], ref['points']) and np.array_equal(res['prob'], ref['prob']) and np.array_equal(res['dist'], ref['dist'])


CLOUDS = [  # shape, noise, n_rays, prob_thresh, nms_thresh, seed, anisotropy, use_bbox, use_kdtree  (tests/tools/nms3d_serial_fuzz.py)
    ((20, 26, 30), 0.2, 65, 0.93, 0.3, 1, None, 1, 1), ((20, 26, 30), 0.4, 100, 0.94, 0.2, 2, None, 1, 1),
    ((18, 24, 26), 0.3, 187, 0.96, 0.4, 3, None, 1, 1), ((24, 30, 33), 0.1, 32, 0.9, 0.1, 4, (2, 1, 1), 1, 1),
    ((24, 30, 33), 0.6, 48, 0.92, 0.5, 5, (1, 1.5, 3), 1, 1), ((22, 28, 31), 0.2, 24, 0.9, 0.3, 6, None, 0, 1),
    ((22, 28, 31), 0.2, 24, 0.9, 0.3, 7, None, 1, 0), ((22, 28, 31), 0.9, 40, 0.93, 0.05, 8, None, 1, 1),
    ((30, 34, 36), 0.0, 16, 0.9, 0.25, 9, None, 1, 1), ((16, 40, 44), 0.5, 70, 0.93, 0.6, 10, (4, 1, 1), 1, 1),
    ((20, 26, 30), 0.3, 65, 0.92, 0.45, 11, None, 1, 1), ((20, 26, 30), 0.5, 100, 0.93, 0.35, 12, (2, 1, 1), 1, 1),
]


@pytest.mark.parametrize("case", CLOUDS, ids=lambda c: "r%d_s%d" % (c[2], c[5]))
def test_device_nms3d_fuzz_vs_reference(sd, case):
    """the DEVICE 3-D NMS (block-wide summation order in S3 / S4, frontier peeling) against the reference extension on random
    candidate clouds beyond the goldens: 65 / 100 / 187 rays, anisotropic rays, flags -- 0 decisions may differ"""
    if not ref_ext.available(): pytest.skip("oracle/_ref not present")
    os.environ["OMP_NUM_THREADS"] = "1"          # the reference's anisotropy sum is racy
    from stardist_b200.lib.stardist3d import c_non_max_suppression_inds
    shape, noise, n_rays, pthr, nthr, seed, aniso, use_bbox, use_kd = case
    prob, dist = cases.create_random_data_3d(shape, noise, n_rays, seed)
    mask = prob > pthr
    m2 = np.zeros_like(mask); m2[2:-2, 2:-2, 2:-2] = True
    mask &= m2
    points = np.stack(np.where(mask), axis=1)
    d = dist[mask]; s = prob[mask]
    ind = np.argsort(s, kind='stable')[::-1]
    d = np.ascontiguousarray(d[ind], np.float32); p = np.ascontiguousarray(points[ind], np.float32); s = np.ascontiguousarray(s[ind], np.float32)
    rays = cases.rays_golden_spiral(n_rays, aniso)
    v = np.ascontiguousarray(rays.vertices, np.float32); f = np.ascontiguousarray(rays.faces, np.int32)
    want = ref_ext.stardist3d().c_non_max_suppression_inds(d, p, v, f, s, int(use_bbox), int(use_kd), 0, np.float32(nthr))
    got = c_non_max_suppression_inds(d, p, v, f, s, int(use_bbox), int(use_kd), 0, np.float32(nthr))
    assert len(d) > 200
    assert np.array_equal(got, want), "%d of %d decisions differ" % (int((got != want).sum()), len(d))
    # the S3 lower-bound short cut off: same decisions
    from stardist_b200 import _lib
    lib = _lib.load()
    try:
        lib.sdb_nms3d_set_s3_bound(0)
        got0 = c_non_max_suppression_inds(d, p, v, f, s, int(use_bbox), int(use_kd), 0, np.float32(nthr))
        lib.sdb_nms3d_set_s3_bound(2)          # bounds on the coarse fan only
        got2 = c_non_max_suppression_inds(d, p, v, f, s, int(use_bbox), int(use_kd), 0, np.float32(nthr))
        assert np.array_equal(got2, want)
        lib.sdb_nms3d_set_s3_bound(1)
        lib.sdb_nms3d_set_split(0)          # all heavy stages in one launch per round (hulls inside the CTA)
        got1 = c_non_max_suppression_inds(d, p, v, f, s, int(use_bbox), int(use_kd), 0, np.float32(nthr))
    finally:
        lib.sdb_nms3d_set_s3_bound(1); lib.sdb_nms3d_set_split(1)
    assert np.array_equal(got0, want) and np.array_equal(got1, want)
