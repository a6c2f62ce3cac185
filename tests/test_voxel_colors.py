"""CPU-side checks of the colour-carrying voxel filter (psulvsb_voxel_down_sample_colors*, csrc/k8_voxel_colors.cu),
PLY colours (psulvsb_ply_read_xyz_rgb) and multi-scale colored ICP: the restatements' own sanity, every refusal before
any device work, zero counts without a device, workspace sizes, the ctypes bindings against the header, the new
kernels' registers, and the pinned scene where the pyramid converges and the finest scale alone does not."""
import ctypes as C
import os
import re
import struct
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi, features, icp, io
from tests import multiscale_colored_icp_restatement as MR
from tests import voxel_colors_restatement as VCR
from tests import voxel_restatement as VR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")
BUF = np.zeros(4 * 33)


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def ccl(specs):
    arr = (capi.ColorCloud * max(len(specs), 1))()
    for c, spec in enumerate(specs):
        arr[c].points, arr[c].n, arr[c].colors = BUF.ctypes.data, 4, BUF.ctypes.data
        for k, v in spec.items():
            setattr(arr[c], k, v)
    return arr


# ---- the restatement ------------------------------------------------------------------------------------------------

def test_restatement_one_point_per_voxel_returns_the_input_colours():
    rng = np.random.default_rng(0)
    P = rng.uniform(-5.0, 5.0, (3, 300))
    Cl = rng.uniform(0.0, 1.0, (3, 300))
    v, c = VCR.voxel_down_sample_colors(P, Cl, 1e-6)
    assert same(v, P) and same(c, Cl)
    assert same(v, VR.voxel_down_sample(P, 1e-6))


def test_restatement_sums_in_input_order_with_one_division():
    P = np.zeros((3, 3))
    Cl = np.array([[0.1, 0.2, 0.3], [1.0, 1e-17, -1.0], [0.7, 0.7, 0.7]])
    v, c = VCR.voxel_down_sample_colors(P, Cl, 1.0)
    assert v.shape == (3, 1)
    want = [((0.1 + 0.2) + 0.3) / 3.0, ((1.0 + 1e-17) + -1.0) / 3.0, ((0.7 + 0.7) + 0.7) / 3.0]
    assert list(c[:, 0]) == want


def test_restatement_nan_colour_stays_in_its_voxel():
    P = np.array([[0.0, 0.1, 5.0, 5.1], [0.0] * 4, [0.0] * 4])
    Cl = np.full((3, 4), 0.5)
    Cl[1, 0] = np.nan
    v, c = VCR.voxel_down_sample_colors(P, Cl, 1.0)
    assert v.shape == (3, 2)
    assert np.isnan(c[1, 0]) and np.isfinite(c[[0, 2], 0]).all() and (c[:, 1] == 0.5).all()


def test_restatement_dropped_point_drops_its_colour():
    P = np.array([[0.0, np.nan, 0.2, 3.0], [0.0, 0.0, 0.0, 0.0], [0.0, 0.0, np.inf, 0.0]])
    Cl = np.array([[0.2, 9.0, 9.0, 0.4], [0.2, 9.0, 9.0, 0.4], [0.2, 9.0, 9.0, 0.4]])
    v, c = VCR.voxel_down_sample_colors(P, Cl, 1.0)
    assert same(v, VR.voxel_down_sample(P, 1.0)) and v.shape == (3, 2)
    assert same(c, np.array([[0.2, 0.4]] * 3))


# ---- refusals, zero counts, workspaces --------------------------------------------------------------------------------

def four(sel=(0, 1, 2, 3), v=0.1, n=4, arr=None, B=1, pts=True, cols=True, work=True, out=True, ocol=True, count=True):
    """Return codes of psulvsb_voxel_down_sample_colors, _host, _batch and _batch_host (the indices in `sel` only)."""
    L = capi.lib()
    p, c, w, o, oc, k = (BUF.ctypes.data if f else None for f in (pts, cols, work, out, ocol, count))
    arr = ccl([{}]) if arr is None else arr
    calls = (lambda: L.psulvsb_voxel_down_sample_colors(None, p, c, n, v, w, o, oc, k),
             lambda: L.psulvsb_voxel_down_sample_colors_host(p, c, n, v, o, oc, k),
             lambda: L.psulvsb_voxel_down_sample_colors_batch(None, arr, B, v, w, o, oc, k),
             lambda: L.psulvsb_voxel_down_sample_colors_batch_host(arr, B, v, o, oc, k))
    return tuple(calls[j]() for j in sel)


def test_refusals_come_before_any_device_work():
    inv = (capi.ERR_INVALID,) * 4
    for v in (0.0, -1.0, float("nan"), float("inf")):
        assert four(v=v) == inv, v
        assert four((2, 3), B=0, v=v) == inv[:2], v
    assert four((0, 1), cols=False) == inv[:2]                          # NULL colours of a non-empty cloud
    assert four((2, 3), arr=ccl([{}, {}, {"colors": None}]), B=3) == inv[:2]
    assert four(out=False) == inv and four(ocol=False) == inv and four(count=False) == inv
    assert four((0, 1), pts=False) == inv[:2]
    assert four((0, 2), work=False) == inv[:2]
    assert four((0, 1), n=-1) == inv[:2]
    assert four((2, 3), B=-1) == inv[:2]
    for spec in ({"n": -1}, {"points": None}):
        assert four((2, 3), arr=ccl([{}, {}, spec]), B=3) == inv[:2], spec
    big = 2 ** 30
    assert four((2, 3), arr=ccl([{"n": big}, {"n": big}]), B=2) == (capi.ERR_UNSUPPORTED,) * 2
    assert four((2, 3), B=0) == (capi.OK, capi.OK)
    with pytest.raises(ValueError):
        features.voxel_down_sample(np.zeros((3, 4)), 0.1, colors=np.zeros((3, 5)))
    with pytest.raises(ValueError):
        features.voxel_down_sample_batch([np.zeros((3, 4))], 0.1, colors=[])


def test_empty_clouds_give_zero_counts_without_a_device():
    L = capi.lib()
    m = np.full(3, 7, dtype=np.int32)
    assert L.psulvsb_voxel_down_sample_colors_host(None, None, 0, 0.1, None, None, m.ctypes.data) == capi.OK
    assert m[0] == 0
    m[:] = 7
    arr = ccl([{"n": 0, "points": None, "colors": None}] * 3)
    assert L.psulvsb_voxel_down_sample_colors_batch_host(arr, 3, 0.1, BUF.ctypes.data, BUF.ctypes.data,
                                                         m.ctypes.data) == capi.OK and list(m) == [0, 0, 0]
    v, c = features.voxel_down_sample(np.zeros((3, 0)), 0.1, colors=np.zeros((3, 0)))
    assert v.shape == (3, 0) and c.shape == (3, 0)
    vs, cs = features.voxel_down_sample_batch([np.zeros((3, 0))] * 2, 0.1, colors=[np.zeros((3, 0))] * 2)
    assert [a.shape for a in vs + cs] == [(3, 0)] * 4
    if L.psulvsb_device_count() == 0:
        assert four() == (capi.ERR_NO_DEVICE,) * 4
        with pytest.raises(capi.PsulvsbError):
            features.voxel_down_sample(np.zeros((3, 4)), 0.1, colors=np.zeros((3, 4)))


def test_workspace_sizes_depend_on_the_sizes_only():
    L = capi.lib()
    for n in (0, 1, 128, 129, 5000, 500000):
        w = L.psulvsb_voxel_down_sample_colors_workspace_bytes(n)
        assert w >= L.psulvsb_voxel_down_sample_workspace_bytes(n) + 8
        assert L.psulvsb_voxel_down_sample_colors_batch_workspace_bytes(ccl([{"n": n}]), 1) == w
    assert L.psulvsb_voxel_down_sample_colors_workspace_bytes(-1) == 0

    def vw(sizes, **kw):
        return L.psulvsb_voxel_down_sample_colors_batch_workspace_bytes(ccl([dict(n=n, **kw) for n in sizes]),
                                                                        len(sizes))

    base = [5000, 129, 0, 1]
    assert vw(base) == vw(base, points=None, colors=None, normals=BUF.ctypes.data) > 0
    assert vw([50000] + base[1:]) > vw(base) and vw([5000] * 592) > vw([5000] * 16)
    assert vw([]) == 0 and vw([-1, 5]) == 0
    assert L.psulvsb_voxel_down_sample_colors_batch_workspace_bytes(None, 3) == 0


# ---- bindings against the header ------------------------------------------------------------------------------------

def _prototypes(header, prefix):
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", header)).read(), flags=re.S)
    out = {}
    for m in re.finditer(r"(\w[\w\s\*]*?)\b(" + prefix + r"\w*)\s*\(([^)]*)\);", src):
        args = [a.strip() for a in m.group(3).split(",")]
        out[m.group(2)] = (m.group(1).strip(), args)
    return out


def _ctype_of(arg):
    if "*" in arg:
        if "psulvsb_color_cloud_t" in arg:
            return C.POINTER(capi.ColorCloud)
        return "ptr"
    return {"int": C.c_int, "double": C.c_double}[arg.rsplit(" ", 1)[0].replace("const ", "").strip()]


def test_ctypes_bindings_match_the_header(tmp_path):
    L = capi.lib()
    protos = _prototypes("psulvsb.h", "psulvsb_voxel_down_sample_colors")
    assert len(protos) == 6
    for name, (ret, args) in protos.items():
        f = getattr(L, name)
        assert name in capi.SYMBOLS
        assert len(f.argtypes) == len(args), name
        for got, arg in zip(f.argtypes, args):
            want = _ctype_of(arg)
            if want == "ptr":
                assert got in (C.c_void_p,) or issubclass(got, C._Pointer), (name, arg)
            else:
                assert got == want, (name, arg, got)
        if ret.startswith("unsigned long long"):
            assert f.restype == C.c_ulonglong, name
    rgb = _prototypes("psulvsb_io.h", "psulvsb_ply_read_xyz_rgb")["psulvsb_ply_read_xyz_rgb"]
    assert len(rgb[1]) == 5 and "psulvsb_ply_read_xyz_rgb" in io.IO_SYMBOLS
    io._lib()
    assert L.psulvsb_ply_read_xyz_rgb.argtypes[2] == C.POINTER(C.c_double)
    # the batch item is the colour-gradient batch's struct, whose layout a C compile pins
    src = tmp_path / "sizes.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "psulvsb.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(psulvsb_color_cloud_t), '
                   "offsetof(psulvsb_color_cloud_t, n), offsetof(psulvsb_color_cloud_t, colors), "
                   "offsetof(psulvsb_color_cloud_t, normals)); return 0; }\n")
    exe = str(tmp_path / "sizes")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    K = capi.ColorCloud
    assert list(map(int, subprocess.check_output([exe], text=True).split())) == [
        C.sizeof(K), K.n.offset, K.colors.offset, K.normals.offset]


# ---- registers ------------------------------------------------------------------------------------------------------

def test_voxel_colors_kernels_registers(tmp_path):
    """sm_100a, -Xptxas -v: k8_voxel_colors.cu holds ft_voxel.cuh's passes and the colour mean pass, each in its
    batch and batch-of-one instantiation, with no stack frame and no spills."""
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", os.path.join(CSRC, "k8_voxel_colors.cu"), "-o",
                        str(tmp_path / "k8vc.o")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = r.stderr.splitlines()
    seen = {}
    for i, line in enumerate(lines):
        m = re.search(r"Function properties for \S*?\d(k8_[a-z0-9_]+?)(?:ILb[01]E|E)", line)
        if not m:
            continue
        f = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 1])
        assert f and f.groups() == ("0", "0", "0"), lines[i:i + 3]
        seen[m.group(1)] = seen.get(m.group(1), 0) + 1
    assert seen == {"k8_voxel_bounds": 2, "k8_voxel_count": 2, "k8_cloud_scan": 2, "k8_grid_scatter": 1,
                    "k8_voxel_order": 2, "k8_voxel_first": 2, "k8_voxel_scan": 2, "k8_voxel_mean_colors": 2}, seen


# ---- PLY colours ----------------------------------------------------------------------------------------------------

def write_ply(path, pts, rgb, fmt, ctype, channels=("red", "green", "blue")):
    """x, y, z as float between an extra leading int property and a trailing float one, the colour channels of type
    ctype after them, then a face element with a list property."""
    n = pts.shape[1]
    hdr = ["ply", f"format {fmt} 1.0", f"element vertex {n}", "property int id", "property float x",
           "property float y", "property float z"]
    hdr += [f"property {ctype} {ch}" for ch in channels]
    hdr += ["property float confidence", "element face 2", "property list uchar int vertex_indices", "end_header"]
    code = {"uchar": "B", "uint8": "B", "float": "f", "double": "d", "ushort": "H"}[ctype]
    with open(path, "wb") as f:
        f.write(("\n".join(hdr) + "\n").encode())
        if fmt == "ascii":
            for i in range(n):
                row = [str(i)] + [repr(float(np.float32(v))) for v in pts[:, i]]
                row += [str(int(v)) if code in "BH" else repr(float(v)) for v in rgb[:len(channels), i]] + ["0.5"]
                f.write((" ".join(row) + "\n").encode())
            f.write(b"3 0 1 2\n3 1 2 3\n")
        else:
            e = "<" if fmt == "binary_little_endian" else ">"
            for i in range(n):
                f.write(struct.pack(e + "i", i) + struct.pack(e + "3f", *[float(v) for v in pts[:, i]]))
                vals = [int(v) if code in "BH" else float(v) for v in rgb[:len(channels), i]]
                f.write(struct.pack(e + code * len(channels), *vals) + struct.pack(e + "f", 0.5))
            f.write(struct.pack(e + "Biii", 3, 0, 1, 2) + struct.pack(e + "Biii", 3, 1, 2, 3))


@pytest.mark.parametrize("fmt", ["ascii", "binary_little_endian", "binary_big_endian"])
@pytest.mark.parametrize("ctype", ["uchar", "uint8", "float", "double"])
def test_ply_colours(tmp_path, fmt, ctype):
    rng = np.random.default_rng(2)
    pts = rng.uniform(-2.0, 2.0, (3, 97))
    if ctype in ("uchar", "uint8"):
        raw = rng.integers(0, 256, (3, 97)).astype(np.float64)
        want = raw / 255.0
    else:
        raw = rng.uniform(0.0, 1.0, (3, 97))
        if ctype == "float":                                               # values a float property can hold
            raw = raw.astype(np.float32).astype(np.float64)
        want = raw
    p = str(tmp_path / "c.ply")
    write_ply(p, pts, raw, fmt, ctype)
    xyz, rgb = io.read_ply_xyz_rgb(p)
    assert same(xyz, pts.astype(np.float32).astype(np.float64))
    assert same(rgb, want), np.abs(rgb - want).max()
    assert same(io.read_ply_xyz(p), xyz)                                  # the colour-blind reader is unchanged


def test_ply_colours_refused(tmp_path):
    pts = np.zeros((3, 4))
    p = str(tmp_path / "a.ply")
    write_ply(p, pts, np.zeros((3, 4)), "ascii", "uchar", channels=("red", "green"))
    with pytest.raises(capi.PsulvsbError) as e:
        io.read_ply_xyz_rgb(p)
    assert e.value.code == capi.ERR_INVALID and "blue" in str(e.value)
    assert io.read_ply_xyz(p).shape == (3, 4)
    write_ply(p, pts, np.zeros((3, 4)), "binary_little_endian", "ushort")
    with pytest.raises(capi.PsulvsbError) as e:
        io.read_ply_xyz_rgb(p)
    assert e.value.code == capi.ERR_INVALID and "unsupported type" in str(e.value)
    assert io.read_ply_xyz(p).shape == (3, 4)


# ---- the pyramid on the restatements --------------------------------------------------------------------------------

def test_pyramid_reaches_the_truth_where_the_finest_scale_alone_does_not():
    """The pinned scene: 3 scales (v, v/2, v/4) from a start 2.5 fine voxels off along z land within 0.01 degrees and
    0.01 fine spacings of the truth; colored ICP at v/4 alone from the same start finds no correspondence."""
    P, Q, Cs, Ct, Rt, tt, R0, t0 = MR.scene()
    fine = MR.SCENE_SCALES[-1]
    res = MR.multiscale_colored_icp(P, Q, Cs, Ct, R0, t0, MR.SCENE_SCALES)
    deg, dt = MR.pose_errors(res[-1]["R"], res[-1]["t"], Rt, tt)
    assert deg < MR.MAX_DEG and dt / fine < MR.MAX_FINE, (deg, dt / fine)
    assert res[-1]["fitness"] > 0.9
    alone = MR.multiscale_colored_icp(P, Q, Cs, Ct, R0, t0, (fine,))[0]
    deg1, dt1 = MR.pose_errors(alone["R"], alone["t"], Rt, tt)
    assert alone["n_corr"] == 0 and alone["iterations"] == 0 and alone["status"] == icp.NO_UPDATE
    assert dt1 / fine > 2.0 and deg1 > 1.0


def test_multiscale_arguments_are_checked():
    P = np.zeros((3, 4))
    with pytest.raises(ValueError):
        icp.multiscale_colored_icp(P, P, P, P, np.eye(3), np.zeros(3), ())
    with pytest.raises(ValueError):
        icp.multiscale_colored_icp(P, P, P, P, np.eye(3), np.zeros(3), (0.2, 0.1), max_iterations=(5,))
    with pytest.raises(ValueError):
        icp.multiscale_colored_icp(P, P, P, P, np.eye(3), np.zeros(3), (0.2,), max_correspondence_distances=(1, 2))
    with pytest.raises(ValueError):
        icp.multiscale_colored_icp_batch([P], [P, P], [P], [P], np.eye(3)[None], np.zeros((1, 3)), (0.2,))
