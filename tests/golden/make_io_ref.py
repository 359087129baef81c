"""tests/golden/io_ref.json: sha256 digests of what the reference's polyroi_bytearray (stardist/utils.py) and
export_to_obj_file3D (stardist/geometry/geom3d.py) return on the inputs of tests/test_io_cpu.py.  The two functions are
compiled in isolation (their modules import csbdeep / skimage).  Usage: python tests/golden/make_io_ref.py <reference checkout>"""
import ast, hashlib, json, os, sys
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import test_io_cpu as T


def functions(path, names, ns):
    body = [n for n in ast.parse(open(path).read()).body if isinstance(n, ast.FunctionDef) and n.name in names]
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    return ns


if __name__ == "__main__":
    ref = sys.argv[1]
    u = functions(os.path.join(ref, "stardist", "utils.py"), ("polyroi_bytearray",), {"np": np})
    g = functions(os.path.join(ref, "stardist", "geometry", "geom3d.py"), ("dist_to_coord3D", "export_to_obj_file3D"),
                  {"np": np, "tqdm": (lambda x: x)})
    polys = T.obj_polys()
    out = {"polyroi_bytearray": [hashlib.sha256(bytes(u["polyroi_bytearray"](xs, ys, pos=pos, subpixel=sub))).hexdigest()
                                 for xs, ys, pos, sub in T.polyroi_cases()],
           "export_to_obj_file3D": [hashlib.sha256(g["export_to_obj_file3D"](dict(polys), **kw).encode()).hexdigest()
                                    for kw in T.OBJ_KWARGS]}
    json.dump(out, open(os.path.join(HERE, "io_ref.json"), "w"), indent=0)
    print(len(out["polyroi_bytearray"]), "+", len(out["export_to_obj_file3D"]), "digests")
