"""The C-ABI library builds for sm_100a, loads without a GPU, exports every symbol include/rtz.h
declares, and refuses to compute without a device (no CPU fallback)."""
import ctypes as C
import re
import subprocess
from pathlib import Path

import rtzlib as R

HEADER = R.ROOT / "include" / "rtz.h"


def _declared():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(rtz_[a-z0-9_]+)\s*\(", text)))


def test_exports_every_declared_symbol(pkg):
    names = _declared()
    assert len(names) >= 18 and "rtz_render" in names and "rtz_render_resident" in names
    lib = C.CDLL(str(pkg.binding.LIB_PATH))
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    # the ctypes binding covers the same set
    assert sorted(pkg.binding.SIGNATURES) == names
    assert pkg.lib().rtz_abi_version() == 2


def test_struct_layouts_match_header(pkg):
    """extern-struct compatible PODs: sizes as a C compiler lays them out."""
    src = r'''
    #include <stdio.h>
    #include "rtz.h"
    int main(void){ printf("%zu %zu %zu %zu %zu %zu\n", sizeof(rtz_sphere), sizeof(rtz_camera), sizeof(rtz_shard),
                           sizeof(rtz_stats), sizeof(rtz_hit), sizeof(rtz_scatter)); return 0; }
    '''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        (Path(d) / "s.c").write_text(src)
        subprocess.run(["gcc", "-std=c99", "-I", str(HEADER.parent), "-o", f"{d}/s", f"{d}/s.c"], check=True)
        sizes = [int(x) for x in subprocess.run([f"{d}/s"], capture_output=True, text=True, check=True).stdout.split()]
    B = pkg.binding
    assert sizes == [C.sizeof(B.rtz_sphere), C.sizeof(B.rtz_camera), C.sizeof(B.rtz_shard), C.sizeof(B.rtz_stats),
                     C.sizeof(B.rtz_hit), C.sizeof(B.rtz_scatter)]
    assert sizes == [C.sizeof(R.Sphere), C.sizeof(R.Camera), C.sizeof(R.Shard), C.sizeof(R.Stats), C.sizeof(R.Hit),
                     C.sizeof(R.Scatter)]


ZIG = R.ROOT / "raytracing-with-zig_b200" / "zig"


def _c_struct_fields(name):
    """[(field, ctype, array_len)] of a typedef struct in rtz.h, in declaration order."""
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, flags=re.S).group(1)
    out = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        ctype, names = decl.split(None, 1)
        for nm in names.split(","):
            m = re.match(r"\s*(\w+)(?:\[(\d+)\])?\s*$", nm)
            out.append((m.group(1), ctype, int(m.group(2) or 0)))
    return out


def test_zig_glue_matches_the_header_without_a_zig_compiler(pkg, tmp_path):
    """SURVEY 8f row 1: the Zig host layer cannot be compiled here (no zig in the image), so it is tied to
    include/rtz.h mechanically: (1) every extern struct in zig/rtz.zig lists the header's fields in the header's
    order with the matching Zig type; (2) the sizes and offsets in its `comptime` assertions are the ones a C
    compiler computes from rtz.h; (3) every `extern "rtz" fn` it declares is exported by librtz.so; (4) the three
    patches under zig/patch/ apply to the reference's build.zig, src/camera.zig and src/main.zig.  Those are kept
    as excerpts under golden/zig_reference/: the reference lines each hunk touches, with their context, hunks
    separated by a `// [...]` line."""
    zig = (ZIG / "rtz.zig").read_text()
    zig_type = {"double": "f64", "uint64_t": "u64", "int32_t": "i32", "uint32_t": "u32"}
    asserted = {}
    for kind, st, field, val in re.findall(r"std\.debug\.assert\(@(sizeOf|offsetOf)\((\w+)(?:, \"(\w+)\")?\) == (\d+)\);", zig):
        asserted[(st, field)] = int(val)
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "rtz.h"', "int main(void){"]
    expect_keys = []
    for st in ("rtz_sphere", "rtz_camera", "rtz_stats"):
        fields = _c_struct_fields(st)
        zbody = re.search(r"pub const %s = extern struct \{(.*?)\n\};" % st, zig, flags=re.S).group(1)
        zfields = re.findall(r"^\s*(\w+): (\[3\])?(\w+)", zbody, flags=re.M)
        assert [(f, zig_type[t], n) for f, t, n in fields] == [(f, t, 3 if arr else 0) for f, arr, t in zfields], st
        lines.append('printf("%%zu\\n", sizeof(%s));' % st)
        expect_keys.append((st, ""))
        for f, _, _ in fields:
            lines.append('printf("%%zu\\n", offsetof(%s, %s));' % (st, f))
            expect_keys.append((st, f))
    lines.append("return 0;}")
    (tmp_path / "o.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-I", str(HEADER.parent), "-o", str(tmp_path / "o"), str(tmp_path / "o.c")], check=True)
    vals = [int(x) for x in subprocess.run([str(tmp_path / "o")], capture_output=True, text=True, check=True).stdout.split()]
    assert dict(zip(expect_keys, vals)) == asserted          # every size / offset, nothing missing, nothing extra
    lib = C.CDLL(str(pkg.binding.LIB_PATH))
    externs = re.findall(r'pub extern "rtz" fn (\w+)\(', zig)
    assert "rtz_render" in externs and "rtz_render_multi" in externs
    assert all(hasattr(lib, fn) for fn in externs), [fn for fn in externs if not hasattr(lib, fn)]
    assert "RTZ_ABI_VERSION: i32 = %d" % pkg.lib().rtz_abi_version() in zig
    patches = sorted((ZIG / "patch").glob("*.patch"))
    assert [p.name for p in patches] == ["build.zig.patch", "camera.zig.patch", "main.zig.patch"]
    import shutil
    work = tmp_path / "ref"
    shutil.copytree(R.GOLDEN / "zig_reference", work)
    for p in patches:
        r = subprocess.run(["patch", "-p1", "-i", str(p)], cwd=work, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
    cam = (work / "src" / "camera.zig").read_text()
    assert 'rtz.render(self, "images/" ++ config.fileName, config.numGpus)' in cam and "self.rayColor(ray);\n                }\n                const avgColor" not in cam


def test_sm100a_code_with_tma_in_the_binary(pkg):
    """The shipped kernels are sm_100a SASS and the scene staging is a TMA bulk copy (UBLKCP)."""
    out = subprocess.run(["cuobjdump", "-sass", str(pkg.binding.LIB_PATH)], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "UBLKCP" in out and "trace_kernel" in out


def test_sweep_stays_on_the_uniform_datapath(pkg):
    """Codegen guard (no GPU needed): in the default kernel the sphere operands of the packed sweep must be
    uniform registers fed by LDCU, and no vote may be guarded by BRA.DIV.  ptxas only does that while it can
    prove the warp converged at the loop top; an innocent-looking edit of the regeneration code loses it
    silently and costs 45 % of the frame time (measured: 156 -> 230 ms on C3)."""
    out = subprocess.run(["cuobjdump", "-sass", str(pkg.binding.LIB_PATH)], capture_output=True, text=True).stdout
    body, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name:
            body.setdefault(name, []).append(line)
    default = [k for k in body if "trace_kernel_constILi128ELi6" in k]
    assert len(default) == 1, default
    sass = "\n".join(body[default[0]])
    assert len(re.findall(r"FFMA2 [^;]*UR\d+\.F32x2", sass)) >= 48, "sweep operands are no longer uniform registers"
    assert "BRA.DIV" not in sass and "LDCU.64" in sass
    # the same for the wavefront kernels that serve scenes of up to 32 / 256 spheres
    for name in ("trace_kernel_waveILi128ELi8", "trace_kernel_wave_nILi4ELi128ELi6"):
        wave = [k for k in body if name in k]
        assert len(wave) == 1, wave
        sass = "\n".join(body[wave[0]])
        assert len(re.findall(r"FFMA2 [^;]*UR\d+\.F32x2", sass)) >= 48, name + ": sweep operands are no longer uniform registers"
        assert "BRA.DIV" not in sass and "LDCU.64" in sass, name


def test_no_device_means_error_not_fallback(pkg):
    import torch
    if torch.cuda.is_available():
        return  # covered by the gpu tests on a GPU box
    l = pkg.lib()
    n = C.c_int32(-1)
    assert l.rtz_device_count(C.byref(n)) == 2 and n.value == 0  # RTZ_ERR_NO_DEVICE
    sp, cnt = R.chapter13_scene()
    cam = R.build_camera(8, 1.0, (0, 0, 0), (0, 0, -1), 90, spp=1, seed=1)
    out = (C.c_uint8 * (3 * 64))()
    bcam = pkg.rtz_camera.from_buffer_copy(bytes(cam))
    rc = l.rtz_render(C.byref(bcam), C.cast(sp, C.POINTER(pkg.rtz_sphere)), cnt, out, None)
    assert rc == 2 and b"no CUDA device" in l.rtz_strerror(rc)
    try:
        pkg.Renderer(0)
        raise AssertionError("Renderer must refuse to run without a GPU")
    except pkg.RtzError as e:
        assert e.status == 2
    # rtz_write_ppm is host-only I/O and works everywhere (PPM.saveBinary, src/ppm.zig:42-60)
    import tempfile, os
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "x.ppm").encode()
        assert l.rtz_write_ppm(p, 1, 1, (C.c_uint8 * 3)()) == 0
        assert open(p, "rb").read() == (R.GOLDEN / "test-binary.ppm").read_bytes()
        assert l.rtz_write_ppm(os.path.join(d, "nodir", "x.ppm").encode(), 1, 1, (C.c_uint8 * 3)()) == 4
