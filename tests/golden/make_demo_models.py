"""tests/golden/demo_models.npz: what it takes, besides the weights in demo2d.npz / demo3d.npz, to rebuild the reference's
shipped model folders models/examples/{2D_demo,3D_demo} byte for byte (demo_models.py does the rebuild):
  <name>/skeleton     weights_best.h5 with the raw bytes of every kernel / bias array cut out (HDF5 structure only)
  <name>/arrays       json list of [weights key, offset in weights_best.h5] of the cut-out arrays, ascending offset
  <name>/sha256       sha256 of weights_best.h5
  <name>/config_json, <name>/thresholds_json   the two json files as they are
Usage: python tests/golden/make_demo_models.py <reference checkout>"""
import hashlib, json, os, sys
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import demo2d, demo3d, demo_models

if __name__ == "__main__":
    out = {}
    for name, mod in (("2D_demo", demo2d), ("3D_demo", demo3d)):
        folder = os.path.join(sys.argv[1], "models", "examples", name)
        h5 = open(os.path.join(folder, "weights_best.h5"), "rb").read()
        z = np.load(mod.PATH)
        keys = sorted((k for k in z.files if k.endswith(("/kernel", "/bias"))), key=lambda k: -z[k].nbytes)
        taken, arrays = [], []
        for k in keys:                    # largest first; an array whose bytes occur twice takes a free occurrence
            raw = np.ascontiguousarray(z[k]).tobytes(); i = h5.find(raw)
            while any(i < e and s < i + len(raw) for s, e in taken):
                i = h5.find(raw, i + 1)
            assert i >= 0, (name, k)
            taken.append((i, i + len(raw))); arrays.append([k, i])
        arrays.sort(key=lambda a: a[1]); taken.sort()
        skel, p = [], 0
        for s, e in taken:
            skel.append(h5[p:s]); p = e
        skel.append(h5[p:])
        out[name + "/skeleton"] = np.frombuffer(b"".join(skel), np.uint8)
        out[name + "/arrays"] = np.frombuffer(json.dumps(arrays).encode(), np.uint8)
        out[name + "/sha256"] = np.frombuffer(hashlib.sha256(h5).hexdigest().encode(), np.uint8)
        for f in ("config", "thresholds"):
            out["%s/%s_json" % (name, f)] = np.frombuffer(open(os.path.join(folder, f + ".json"), "rb").read(), np.uint8)
    np.savez_compressed(demo_models.PATH, **out)
    print(demo_models.PATH, os.path.getsize(demo_models.PATH), "bytes")
