"""Host-side formats either side of the path: ImageJ ROI export, TIFF in/out, the command line parser."""
import hashlib, json, os, zipfile
import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OBJ_KWARGS = (dict(), dict(single_mesh=False), dict(uv_map=True, scale=(2, 1, 0.5)), dict(scale=0.01))


def polyroi_cases():
    rng = np.random.default_rng(0)
    for _ in range(25):
        n = int(rng.integers(3, 40)); xs = rng.uniform(-5, 300, n); ys = rng.uniform(0, 200, n)
        for sub in (True, False):
            for pos in (None, 3):
                yield xs, ys, pos, sub


def obj_polys():
    import stardist_b200 as sd
    rays = sd.Rays_GoldenSpiral(12)
    rng = np.random.default_rng(0)
    return dict(dist=rng.uniform(2, 6, (4, 12)).astype(np.float32), points=rng.integers(5, 40, (4, 3)),
                rays_vertices=rays.vertices, rays_faces=rays.faces)


def test_polyroi_bytes_golden_and_reference():
    from stardist_b200.io import rois
    x = np.array([10.2, 30.7, 25.1, 8.4]); y = np.array([5.5, 7.25, 40.0, 33.3])
    b = bytes(rois.polyroi_bytearray(x, y, pos=2, subpixel=True))
    assert len(b) == 112 and b[:4] == b"Iout"
    assert hashlib.sha256(b).hexdigest() == "9e394be9b5d3ae592c63d1bd595a585848eff9eca31af44bf83dc8026b2b4719"
    # the reference's own function on the same inputs: tests/golden/io_ref.json (make_io_ref.py)
    want = json.load(open(os.path.join(GOLDEN, "io_ref.json")))["polyroi_bytearray"]
    assert [hashlib.sha256(bytes(rois.polyroi_bytearray(xs, ys, pos=pos, subpixel=sub))).hexdigest()
            for xs, ys, pos, sub in polyroi_cases()] == want


def test_export_imagej_rois_and_tiff_roundtrip(tmp_path):
    from stardist_b200.io import rois, tiff
    rng = np.random.default_rng(1)
    coord = rng.uniform(0, 100, (5, 2, 32))
    rois.export_imagej_rois(tmp_path / "set.zip", coord)
    with zipfile.ZipFile(tmp_path / "set.zip") as z:
        names = sorted(z.namelist())
        assert names == ["001_%03d.roi" % i for i in range(1, 6)]
        assert z.read(names[0])[:4] == b"Iout"
    a = rng.integers(0, 5000, (7, 33, 21)).astype(np.int32)
    tiff.imwrite(tmp_path / "a.tif", a)
    assert np.array_equal(tiff.imread(tmp_path / "a.tif"), a)
    b = rng.integers(0, 60000, (40, 50)).astype(np.uint16)
    tiff.imwrite(tmp_path / "b.tif", b)
    assert np.array_equal(tiff.imread(tmp_path / "b.tif"), b)
    with pytest.raises(ValueError):
        tiff.imwrite(tmp_path / "c.tif", np.zeros(3))


def test_cli_parser():
    from stardist_b200.scripts.predict import build_parser
    a = build_parser().parse_args(["-i", "x.tif", "y.tif", "-m", "model", "--n_tiles", "2", "3", "--pnorm", "2", "99", "--rois"])
    assert a.input == ["x.tif", "y.tif"] and a.n_tiles == [2, 3] and a.pnorm == [2.0, 99.0] and a.rois and a.outname == "{img}.stardist.tif"


def test_export_to_obj_file3D(tmp_path):
    """text identical to stardist/geometry/geom3d.py:277-347 (its output digests: tests/golden/io_ref.json)"""
    from stardist_b200.io import obj
    polys = obj_polys()
    text = obj.export_to_obj_file3D(polys, fname=str(tmp_path / "m.obj"))
    assert open(tmp_path / "m.obj").read() == text
    assert text.count("\nv ") + text.startswith("v ") == 4 * 12 and text.count("f ") == 4 * len(polys["rays_faces"]) and text.startswith("o poly_0\n")
    with pytest.raises(ValueError):
        obj.export_to_obj_file3D(dict(dist=polys["dist"]))
    want = json.load(open(os.path.join(GOLDEN, "io_ref.json")))["export_to_obj_file3D"]
    assert [hashlib.sha256(obj.export_to_obj_file3D(polys, **kw).encode()).hexdigest() for kw in OBJ_KWARGS] == want
