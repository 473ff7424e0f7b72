"""CPU: the C-ABI library loads, exports every symbol include/gab200_rasterizer.h declares, the ctypes mirrors match
the C struct layouts, and the Python surface validates arguments like the reference -- no compute calls (no GPU)."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
HEADER = os.path.join(ROOT, "include", "gab200_rasterizer.h")


def _declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gab200_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from gaussianavatars_b200 import _native as N

    lib = N.lib()
    syms = _declared_symbols()
    assert len(syms) >= 12
    for s in syms:
        assert hasattr(lib, s), f"{s} is declared in include/gab200_rasterizer.h but not exported"
    assert set(N.EXPORTED_SYMBOLS) <= set(syms)
    assert lib.gab200_abi_version() == N.ABI_VERSION == 3
    assert b"invalid argument" in lib.gab200_status_string(-1)
    assert b"sm_100" in lib.gab200_status_string(-4)
    # loading the library and the calls above launch nothing; counted in a fresh process, since the GPU tests that
    # share this one have launched kernels
    code = ("from gaussianavatars_b200 import _native as N; lib = N.lib(); lib.gab200_abi_version(); "
            "lib.gab200_status_string(-1); lib.gab200_status_string(-4); print(lib.gab200_launch_count())")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.split()[-1:] == ["0"], (out.stdout, out.stderr)


def test_ctypes_structs_match_the_c_layout(tmp_path):
    """Compile a probe against the header with gcc and compare sizeof/offsetof with the ctypes mirrors."""
    from gaussianavatars_b200 import _native as N

    fields = {"gab200_forward_args": N.ForwardArgs, "gab200_frame_state": N.FrameState, "gab200_backward_args": N.BackwardArgs,
              "gab200_photometric_args": N.PhotometricArgs, "gab200_adam_segment": N.AdamSegment,
              "gab200_densify_args": N.DensifyArgs, "gab200_densify_out": N.DensifyOut,
              "gab200_regularize_args": N.RegularizeArgs}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(){"]
    for cname, ct in fields.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines.append("return 0;}")
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["/usr/bin/gcc", str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    got = dict(l.split() for l in out if l.strip())
    for cname, ct in fields.items():
        assert int(got[cname]) == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(ct, fname).offset, f"{cname}.{fname}"


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from gaussianavatars_b200 import _native as N

    monkeypatch.setattr(N, "_lib", None)
    monkeypatch.setattr(N, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(N.NativeLibraryError, match="no CPU / eager fallback"):
        N.lib()


def test_reference_surface_names_and_argument_validation():
    import gaussianavatars_b200 as g

    assert g.GaussianRasterizationSettings._fields == (
        "image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix", "projmatrix",
        "sh_degree", "campos", "prefiltered", "debug")
    z = torch.zeros
    rs = g.GaussianRasterizationSettings(8, 8, 1.0, 1.0, z(3), 1.0, torch.eye(4), torch.eye(4), 0, z(3), False, False)
    r = g.GaussianRasterizer(rs)
    assert isinstance(r, torch.nn.Module) and r.raster_settings is rs
    kw = dict(means3D=z(4, 3), means2D=z(4, 3), opacities=z(4, 1))
    with pytest.raises(Exception, match="Please provide excatly one of either SHs or precomputed colors!"):
        r(**kw, scales=z(4, 3), rotations=z(4, 4))
    with pytest.raises(Exception, match="Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!"):
        r(**kw, shs=z(4, 1, 3))
    with pytest.raises(Exception, match="scale/rotation pair"):
        r(**kw, shs=z(4, 1, 3), scales=z(4, 3))
    # the product never computes on the CPU
    with pytest.raises(RuntimeError, match="no CPU path"):
        r(**kw, shs=z(4, 1, 3), scales=z(4, 3), rotations=z(4, 4))
    with pytest.raises(RuntimeError, match="no CPU path"):
        g.rasterize_bound(rs, z(4, 3), z(4, 4), z(4, 3), z(4, 1), z(4, 1, 3), z(4, 0, 3))


def test_compat_shim_resolves_the_reference_import():
    code = ("import sys; sys.path.insert(0, %r); "
            "from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer; "
            "import gaussianavatars_b200 as g; "
            "assert GaussianRasterizer is g.GaussianRasterizer; print('ok')") % os.path.join(ROOT, "gaussianavatars_b200", "compat")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd="/tmp")
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under gaussianavatars_b200/ may import or load it."""
    pkg = os.path.join(ROOT, "gaussianavatars_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "libsplat_oracle" not in txt, f


def test_render_route_selection_and_camera_cache():
    from gaussianavatars_b200 import renderer as R
    from gaussianavatars_b200 import synthetic as syn

    class Raw:
        _xyz = _rotation = _scaling = _opacity = _features_dc = _features_rest = None

    class GettersOnly:
        pass

    assert R._has_raw(Raw()) and not R._has_raw(GettersOnly())
    cam = syn.orbit_camera(64, 48)
    blk = R._camera_block(cam, torch.device("cpu"))
    assert R._camera_block(cam, torch.device("cpu")) is blk  # uploaded once, cached on the camera object
    assert blk[0].shape == (4, 4) and blk[2].shape == (3,)


def test_face_csr_chunks_cover_every_splat_once():
    """The face-sorted chunk view handed to the backward's per-face reduction (gab200_backward_args.face_*)."""
    from gaussianavatars_b200 import rasterizer as R

    g = torch.Generator().manual_seed(0)
    F = 37
    binding = torch.randint(0, F, (1000,), generator=g).to(torch.int32)
    binding[:300] = 5  # a hot face (several chunks)
    b32, (perm, c_face, c_start, c_end) = R._face_csr(binding, F, chunk=16)
    assert b32 is binding  # already int32 + contiguous: no copy
    assert sorted(perm.tolist()) == list(range(1000))
    covered = torch.zeros(1000, dtype=torch.int32)
    for f, s, e in zip(c_face.tolist(), c_start.tolist(), c_end.tolist()):
        assert 0 < e - s <= 16
        ids = perm[s:e].long()
        assert (binding[ids] == f).all()
        covered[ids] += 1
    assert (covered == 1).all()
    assert R._face_csr(binding, F, chunk=16)[1][0] is perm  # cached per binding tensor + version
    # an int64 binding (the reference's FlameGaussianModel) is converted ONCE, and another tensor never hits its entry
    b64 = binding.long()
    c32, csr64 = R._face_csr(b64, F, chunk=16)
    assert c32.dtype == torch.int32 and R._face_csr(b64, F, chunk=16)[0] is c32
    other = torch.flip(b64, dims=(0,))
    assert not torch.equal(R._face_csr(other, F, chunk=16)[1][0], csr64[0])
    binding[0] = (int(binding[0]) + 1) % F   # in-place edit bumps the version -> rebuilt
    assert R._face_csr(binding, F, chunk=16)[1][0] is not perm


def test_symmetric_grad_buffer_is_inert_without_a_process_group():
    from gaussianavatars_b200 import dist as gdist

    class PC:
        def parameters(self):
            return [torch.zeros(4, 3)]

    buf = gdist.SymmetricGradBuffer(PC())
    assert buf.enabled is False
    assert gdist.allreduce_splat_grads(PC()) == 0


def test_adam_keeps_the_torch_optimizer_surface():
    """Host logic only (no launch): param_groups / names / lr scheduling / state_dict as the reference uses them
    (scene/gaussian_model.py:222-233, :89), and the configurations that are rejected."""
    import torch
    import gaussianavatars_b200 as g

    p = torch.nn.Parameter(torch.zeros(4, 3))
    q = torch.nn.Parameter(torch.zeros(4, 1))
    opt = g.Adam([{"params": [p], "lr": 1.6e-4, "name": "xyz"}, {"params": [q], "lr": 5e-2, "name": "opacity"}], lr=0.0, eps=1e-15)
    assert isinstance(opt, torch.optim.Optimizer)
    assert [gr["name"] for gr in opt.param_groups] == ["xyz", "opacity"]
    for gr in opt.param_groups:
        if gr["name"] == "xyz":
            gr["lr"] = 1e-5
    sd = opt.state_dict()
    assert sd["param_groups"][0]["lr"] == 1e-5 and sd["param_groups"][0]["eps"] == 1e-15
    opt.add_param_group({"params": [torch.nn.Parameter(torch.zeros(2))], "lr": 1e-3, "name": "pose"})
    opt.zero_grad(set_to_none=True)
    opt.step()                       # no gradients anywhere: nothing to launch, no error even without a GPU
    with pytest.raises(ValueError):
        g.Adam([p], amsgrad=True)
    p.grad = torch.ones_like(p)
    with pytest.raises(RuntimeError, match="no CPU or eager fallback"):
        opt.step()


def test_depth_hint_widening_stays_a_valid_key_range():
    """The hint handed to gab200_forward_args.depth_hint_* : ordered, inside (0, 0xFFFFFFFF), wider than the frame."""
    import struct
    from gaussianavatars_b200 import rasterizer as R

    def key(z):
        return struct.unpack("<I", struct.pack("<f", z))[0]

    for zmin, zmax in [(0.73, 1.31), (0.2000001, 0.2000002), (5.0, 5.0), (1e-3, 1e30), (3.0e38, 3.4e38)]:
        lo, hi = R._widen_depth_range(key(zmin), key(zmax))
        assert 0 < lo <= key(zmin) <= key(zmax) <= hi <= 0xFFFFFFFE
        assert hi > lo                                   # hi <= lo would mean "no hint" to the library
    lo, hi = R._widen_depth_range(key(0.73), key(1.31))
    span = key(1.31) - key(0.73)
    assert key(0.73) - lo == span // 8 and hi - key(1.31) == span // 8


def test_c_abi_example_compiles_and_links(tmp_path):
    """examples/abi_forward_backward.cu is the non-Python caller INTEGRATION.md describes: it must build against
    include/gab200_rasterizer.h from C++ and link against the shared library (running it needs a GPU)."""
    import shutil
    from gaussianavatars_b200 import _native as N

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    N.lib()  # the library must exist (build() ran)
    libdir = os.path.dirname(N.LIB_PATH)
    exe = tmp_path / "abi_example"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-ccbin", "/usr/bin/g++",
           "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "abi_forward_backward.cu"),
           "-L" + libdir, "-lgaussianavatars_b200", "-Xlinker", "-rpath=" + libdir, "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert exe.exists()
