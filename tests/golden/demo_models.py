"""Rebuild the reference's shipped model folders models/examples/{2D_demo,3D_demo} (config.json, thresholds.json,
weights_best.h5) byte for byte from tests/golden/demo_models.npz and the weights in demo2d.npz / demo3d.npz
(see make_demo_models.py)."""
import hashlib, json, os
import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "demo_models.npz")


def rebuild(basedir):
    """writes <basedir>/2D_demo and <basedir>/3D_demo; the weight files are checked against the originals' sha256"""
    import demo2d, demo3d
    g = np.load(PATH)
    for name, mod in (("2D_demo", demo2d), ("3D_demo", demo3d)):
        w = np.load(mod.PATH)
        skel = g[name + "/skeleton"].tobytes()
        parts, p = [], 0
        for key, offset in json.loads(g[name + "/arrays"].tobytes()):
            raw = np.ascontiguousarray(w[key]).tobytes()
            n = offset - sum(len(x) for x in parts)        # skeleton bytes before this array
            parts.append(skel[p:p + n]); p += n
            parts.append(raw)
        parts.append(skel[p:])
        h5 = b"".join(parts)
        assert hashlib.sha256(h5).hexdigest() == g[name + "/sha256"].tobytes().decode(), name
        folder = os.path.join(basedir, name)
        os.makedirs(folder, exist_ok=True)
        open(os.path.join(folder, "weights_best.h5"), "wb").write(h5)
        for f in ("config", "thresholds"):
            open(os.path.join(folder, f + ".json"), "wb").write(g["%s/%s_json" % (name, f)].tobytes())
    return basedir
