"""tests/golden/refshim.npz: values of the reference's inner routines that tests/test_cpu_oracle.py compares the host build
of the device headers with, computed by oracle/_ref/libsdref.so (build it with `make -C oracle ref REF=<reference checkout>`):
  clip/<seed>/sha256  sha256 of the Clipper intersection areas (little-endian float32) of the fuzzed pairs of CLIP_CASES
  overlap      qhull_overlap_kernel / qhull_overlap_convex_hulls (float32, [pair, 2]) of the pairs of overlap_pairs()
Usage: python tests/golden/make_refshim.py"""
import ctypes, hashlib, os, sys
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))
import test_cpu_oracle as T
import clip_fuzz as cf

if __name__ == "__main__":
    out = {}
    for n_rays, radius, noise, seed in T.CLIP_CASES:
        a, b = cf.make_pairs(T.CLIP_PAIRS, n_rays, radius, noise, seed)
        r, _, _ = cf.run(a, b)
        out["clip/%d/sha256" % seed] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(r, "<f4").tobytes()).hexdigest().encode(), np.uint8)
    ref = cf.ref
    for f in (ref.sdref_overlap_kernel, ref.sdref_overlap_convex):
        f.restype = ctypes.c_float
    out["overlap"] = np.array([(ref.sdref_overlap_kernel(*a), ref.sdref_overlap_convex(*a)) for _, _, a, _ in T.overlap_pairs()], np.float32)
    path = os.path.join(HERE, "refshim.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")
