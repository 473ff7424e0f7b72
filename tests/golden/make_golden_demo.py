"""Generates the fixtures that stand in for the original GaussianAvatars checkout in tests/test_io.py and
tests/test_reference_compat.py, so that those comparisons run without it:

  demo_point_cloud_sample.ply   a seeded sample of the records of media/306/point_cloud.ply (the rows holding the
                                smallest and the largest binding are always in it), record bytes copied verbatim, file
                                order kept, under the original header with the vertex count set to the sample's
  demo_flame_param_sample.npz   media/306/flame_param.npz with every per-frame member cut to its first FRAMES frames
                                and every per-vertex member to its first VERTICES vertices; the other members are
                                copied byte for byte, stored (uncompressed) like the original
  reference_facts.json          what the tests assert about those files, computed from the originals with numpy
                                alone, and the parameter list of gaussian_renderer.render

    python tests/golden/make_golden_demo.py <path of the original GaussianAvatars checkout>
"""
import io
import json
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
SAMPLE_ROWS = 256           # x 252 B per record
FRAMES = 4
VERTICES = 512              # of the 5143 of the FLAME mesh
PER_FRAME = ("expr", "rotation", "neck_pose", "jaw_pose", "eyes_pose", "translation", "dynamic_offset")
PER_VERTEX = ("static_offset", "dynamic_offset")   # (frames, vertices, 3)


def ply_sample(src, dst):
    raw = open(src, "rb").read()
    end = raw.index(b"end_header\n") + len(b"end_header\n")
    header = raw[:end].decode("ascii")
    names = [ln.split()[-1] for ln in header.splitlines() if ln.startswith("property float ")]
    count = int(next(ln for ln in header.splitlines() if ln.startswith("element vertex ")).split()[-1])
    table = np.frombuffer(raw[end:], dtype="<f4").reshape(count, len(names))
    b = table[:, names.index("binding_0")]
    keep = set(np.random.default_rng(0).choice(count, SAMPLE_ROWS - 2, replace=False).tolist())
    keep |= {int(b.argmin()), int(b.argmax())}
    rows = np.array(sorted(keep)[:SAMPLE_ROWS])
    sample = table[rows]
    new_header = header.replace(f"element vertex {count}\n", f"element vertex {len(rows)}\n")
    with open(dst, "wb") as f:
        f.write(new_header.encode("ascii") + sample.tobytes())
    op = sample[:, names.index("opacity")].astype(np.float64)
    sb = sample[:, names.index("binding_0")]
    return {"source_vertices": count, "source_binding_min": int(b.min()), "source_binding_max": int(b.max()),
            "vertices": int(len(rows)), "binding_min": int(sb.min()), "binding_max": int(sb.max()),
            "opacity_sigmoid_mean": float((1.0 / (1.0 + np.exp(-op))).mean()), "properties": len(names)}


def flame_sample(src, dst):
    shapes = {}
    with zipfile.ZipFile(src) as zin, zipfile.ZipFile(dst, "w", zipfile.ZIP_STORED) as zout:
        for info in zin.infolist():
            key = info.filename[:-len(".npy")]
            data = zin.read(info)
            if key in PER_FRAME or key in PER_VERTEX:
                a = np.lib.format.read_array(io.BytesIO(data))
                a = a[:FRAMES] if key in PER_FRAME else a
                a = a[:, :VERTICES] if key in PER_VERTEX else a
                buf = io.BytesIO()
                np.lib.format.write_array(buf, np.ascontiguousarray(a), allow_pickle=False)
                data = buf.getvalue()
            zout.writestr(info.filename, data)
            shapes[key] = list(np.lib.format.read_array(io.BytesIO(data)).shape)
    return {"frames": FRAMES, "vertices": VERTICES, "shapes": shapes}


def render_signature(ref):
    sys.path.insert(0, ROOT)
    import inspect

    from tests import ref_import

    ref_import.REF = ref
    ref_import.prepare()
    import gaussian_renderer

    return [{"name": p.name, "has_default": p.default is not inspect.Parameter.empty,
             "default": None if p.default is inspect.Parameter.empty else p.default}
            for p in inspect.signature(gaussian_renderer.render).parameters.values()]


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    ref = os.path.abspath(sys.argv[1])
    demo = os.path.join(ref, "media", "306")
    facts = {"point_cloud": ply_sample(os.path.join(demo, "point_cloud.ply"),
                                       os.path.join(HERE, "demo_point_cloud_sample.ply")),
             "flame_param": flame_sample(os.path.join(demo, "flame_param.npz"),
                                         os.path.join(HERE, "demo_flame_param_sample.npz")),
             "render_signature": render_signature(ref)}
    with open(os.path.join(HERE, "reference_facts.json"), "w") as f:
        json.dump(facts, f, indent=1)
        f.write("\n")
    print(json.dumps(facts))


if __name__ == "__main__":
    main()
