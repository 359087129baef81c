"""tests/golden/refcalls/*.npz.xz: the answers of the reference's compiled modules (oracle/_ref) that oracle/ref_ext.py replays
where oracle/_ref cannot be built.  Record them with oracle/_ref built, e.g.
    STARDIST_ORACLE_RECORD=/tmp/rec python -m pytest tests          (and smoke(), on a GPU machine for the GPU tests)
then merge one or more such directories:  python tests/golden/make_refcalls.py /tmp/rec [more dirs]
A key recorded twice with different answers is an error (the reference's 3-D NMS is only deterministic with one OpenMP thread).
Answers above MAX_ANSWER bytes are left out: a test that needs one stores a digest of it instead.  The one such answer, the
label volume of tests/test_gpu_at_size.py::test_volume_3d_equals_oracle, is pinned by at_size_3d.json (sha256 of
relabel_sequential of that answer as int32, its shape and label count), which that test checks against the reference
wherever oracle/_ref is built."""
import glob, io, lzma, os, sys
import numpy as np

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "refcalls")
LIMIT = 900 << 10        # compressed bytes per file
MAX_ANSWER = 16 << 20


def compress(entries):
    buf = io.BytesIO(); np.savez(buf, **entries)
    return lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME)


if __name__ == "__main__":
    merged = {}
    for d in sys.argv[1:]:
        for p in sorted(glob.glob(os.path.join(d, "*.npz"))):
            z = np.load(p)
            for k in z.files:
                a = z[k]
                if k in merged and not (merged[k].dtype == a.dtype and np.array_equal(merged[k], a)):
                    raise SystemExit("%s: %s recorded with two different answers" % (p, k))
                merged[k] = a
    for k in [k for k, a in merged.items() if a.nbytes > MAX_ANSWER]:
        print("left out", k, merged.pop(k).shape)
    chunks, cur = [], {}
    for k in sorted(merged):          # greedy split: a chunk is closed when adding to it would pass LIMIT
        cur[k] = merged[k]
        if len(cur) % 16 == 0 and len(compress(cur)) > LIMIT:
            last = cur.pop(k); chunks.append(cur); cur = {k: last}
    chunks.append(cur)
    for p in glob.glob(os.path.join(OUT, "*.npz.xz")): os.remove(p)
    os.makedirs(OUT, exist_ok=True)
    for i, c in enumerate(chunks):
        path = os.path.join(OUT, "refcalls_%02d.npz.xz" % i)
        open(path, "wb").write(compress(c))
        print(path, len(c), "answers", os.path.getsize(path), "bytes")
