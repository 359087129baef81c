"""Fuzz the host build of clip2d.cuh against the reference Clipper (oracle/_ref/libsdref.so).
Usage: python tests/tools/clip_fuzz.py [n_pairs] [n_rays] [radius] [noise] [seed]"""
import ctypes, sys, numpy as np, os
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF_SO = os.path.join(ROOT, "oracle/_ref/libsdref.so")
ref = ctypes.CDLL(REF_SO) if os.path.exists(REF_SO) else None      # built only where the reference's sources are
hc = ctypes.CDLL(os.path.join(ROOT, "tests/hostcheck/_build/libhostcheck.so"))

def make_pairs(n_pairs, n_rays, radius, noise, seed, span=None):
    rng = np.random.default_rng(seed)
    phi = (np.float32(2*np.pi/n_rays) * np.arange(n_rays, dtype=np.float32)).astype(np.float32)
    def polys(c):
        d = (radius * (1 + noise * rng.uniform(-1, 1, (n_pairs, n_rays)))).astype(np.float32)
        y = (c[:, :1] + d * np.sin(phi)[None]).astype(np.float32)
        x = (c[:, 1:] + d * np.cos(phi)[None]).astype(np.float32)
        return np.stack([x.astype(np.int64), y.astype(np.int64)], -1)  # trunc toward zero
    ca = rng.integers(0, 1024, (n_pairs, 2)).astype(np.float32)
    sp = span if span is not None else 2.2 * radius
    cb = (ca + rng.integers(-int(sp), int(sp) + 1, (n_pairs, 2))).astype(np.float32)
    return polys(ca), polys(cb)

def host(a, b):
    n_pairs, n = a.shape[:2]
    a32 = np.ascontiguousarray(a, np.int32); b32 = np.ascontiguousarray(b, np.int32)
    h = np.zeros(n_pairs, np.float32); st = np.zeros(n_pairs, np.int32)
    P = ctypes.c_void_p
    hc.hc_clip_area_batch(P(a32.ctypes.data), P(b32.ctypes.data), n_pairs, n, P(h.ctypes.data), P(st.ctypes.data))
    return h, st

def run(a, b):
    n_pairs, n = a.shape[:2]
    a64 = np.ascontiguousarray(a, np.int64); b64 = np.ascontiguousarray(b, np.int64)
    r = np.zeros(n_pairs, np.float32)
    P = ctypes.c_void_p
    ref.sdref_clip_area_batch(P(a64.ctypes.data), P(b64.ctypes.data), n_pairs, n, P(r.ctypes.data))
    h, st = host(a, b)
    return r, h, st

def paths_ref(a, b):
    a64 = np.ascontiguousarray(a, np.int64); b64 = np.ascontiguousarray(b, np.int64)
    out = np.zeros((4096, 2), np.int64); cnt = np.zeros(64, np.int32)
    P = ctypes.c_void_p
    k = ref.sdref_clip_intersection(P(a64.ctypes.data), len(a), P(b64.ctypes.data), len(b), P(out.ctypes.data), P(cnt.ctypes.data), 64, 4096)
    res, o = [], 0
    for i in range(k): res.append(out[o:o+cnt[i]].copy()); o += cnt[i]
    return res
def paths_hc(a, b):
    a32 = np.ascontiguousarray(a, np.int32); b32 = np.ascontiguousarray(b, np.int32)
    out = np.zeros((4096, 2), np.int32); cnt = np.zeros(64, np.int32); st = ctypes.c_int(0)
    P = ctypes.c_void_p
    k = hc.hc_clip_paths(P(a32.ctypes.data), len(a), P(b32.ctypes.data), len(b), P(out.ctypes.data), P(cnt.ctypes.data), 64, 4096, ctypes.byref(st))
    res, o = [], 0
    for i in range(k): res.append(out[o:o+cnt[i]].copy()); o += cnt[i]
    return res, st.value

if __name__ == "__main__":
    n_pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 200000
    n_rays = int(sys.argv[2]) if len(sys.argv) > 2 else 32
    radius = float(sys.argv[3]) if len(sys.argv) > 3 else 10
    noise = float(sys.argv[4]) if len(sys.argv) > 4 else 0.1
    seed = int(sys.argv[5]) if len(sys.argv) > 5 else 0
    a, b = make_pairs(n_pairs, n_rays, radius, noise, seed)
    r, h, st = run(a, b)
    bad = np.nonzero(r.view(np.int32) != h.view(np.int32))[0]
    print(f"pairs={n_pairs} nonzero_ref={np.count_nonzero(r)} mismatches={len(bad)} status!=0: {np.count_nonzero(st)} (overflow {np.count_nonzero(st==2)})")
    for i in bad[:5]:
        print(" pair", i, "ref", r[i], "ours", h[i], "st", st[i])
        pr = paths_ref(a[i], b[i]); ph, s = paths_hc(a[i], b[i])
        print("  ref paths:", [p.tolist() for p in pr]); print("  our paths:", [p.tolist() for p in ph])
        print("  a:", a[i].tolist()); print("  b:", b[i].tolist())
