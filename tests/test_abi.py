"""The C-ABI library loads and exports every symbol include/dgvcc_b200.h declares (no GPU needed)."""
import os
import re

from dgvcc_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "dgvcc_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dgvcc_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported_and_bound():
    lib = _native.lib()
    names = declared_symbols()
    assert len(names) >= 10
    for name in names:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
        assert name in _native.SIGNATURES, f"{name} has no ctypes signature"
    assert set(_native.SIGNATURES) == set(names)
    assert lib.dgvcc_abi_version() >= 4


def test_workspace_layout_is_host_only_and_consistent():
    lay = _native.BLLayout()
    assert _native.lib().dgvcc_bl_workspace_layout(1000, 3, 2, 48, 64, lay) == 0
    offs = [lay.amax, lay.rz, lay.pbg, lay.ebg, lay.counts, lay.wsel, lay.residual, lay.loss_img, lay.ticket,
            lay.cpart, lay.zpart, lay.minpart]
    assert offs == sorted(offs) and all(o % 256 == 0 for o in offs) and lay.total > offs[-1]
    assert lay.rows_per_thread in (2, 4, 8) and lay.cols_per_thread in (1, 2) and lay.tiles > 0
    assert _native.lib().dgvcc_bl_workspace_layout(0, 1, 1, 8, 8, lay) == -1  # DGVCC_ERR_ARG


def test_meta_table_layout():
    import numpy as np
    from dgvcc_b200.losses.bl import build_meta
    counts = np.array([2500, 0, 3, 1024, 1025])
    rows = np.array([2501, 1, 4, 1025, 1026])
    meta, c, multi = build_meta(counts, rows, 1024)
    b = 5
    assert meta[:b + 1].tolist() == [0, 2500, 2500, 2503, 3527, 4552]
    assert meta[b + 1:2 * b + 2].tolist() == [0, 2501, 2502, 2506, 3531, 4557]
    assert meta[2 * b + 2:3 * b + 2].tolist() == [2250, 0, 3, 922, 923]   # ceil(0.9*(rows-1)), bl.py:76
    assert meta[3 * b + 2:4 * b + 3].tolist() == [0, 3, 4, 5, 6, 8]
    table = meta[4 * b + 3:].reshape(c, 4)
    assert c == 8 and multi == 1
    for i in range(b):  # chunks tile each image's points exactly
        mine = table[table[:, 0] == i]
        assert mine[:, 2].sum() == counts[i] and mine[0, 1] == 0
    assert sorted(table[:, 3].tolist()) == list(range(c))


def test_native_host_packing_matches_the_python_packing():
    """dgvcc_bl_pack_host (host-only C) writes byte for byte what build_meta + numpy concatenate write."""
    import numpy as np
    import torch
    from dgvcc_b200.losses import bl
    rng = np.random.default_rng(5)
    for counts, use_bg, chunk in (([2500, 0, 3, 1024, 1025], True, 1024), ([7], False, 4), ([0, 0], True, 1024),
                                  ([300, 12000, 5, 4097], True, 1024)):
        pts = [torch.from_numpy(rng.random((n, 2), dtype=np.float32)) for n in counts]
        tgt = [torch.from_numpy(rng.random(n, dtype=np.float32)) for n in counts]
        ref = bl.pack_batch(pts, tgt, use_background=use_bg, chunk=chunk)
        info, args = bl.pack_host_native(pts, tgt, use_bg, chunk, None, 0)
        assert (info.meta_bytes, info.off_points, info.off_targets, info.total_bytes) == \
            (ref.meta_bytes, ref.o_pts, ref.o_tgt, ref.total)
        assert (info.total_chunks, info.multi_chunk) == (ref.total_chunks, ref.multi_chunk)
        buf = torch.zeros((info.total_bytes,), dtype=torch.uint8)
        bl.pack_host_native(pts, tgt, use_bg, chunk, buf.data_ptr(), buf.numel(), args)
        assert torch.equal(buf, ref.buf), counts
    # the same on random batches: sizes around the chunk boundaries, chunk sizes 1 .. 4096, with and without background
    for _ in range(150):
        b = int(rng.integers(1, 10))
        counts = [int(rng.choice([0, 1, 2, 127, 128, 129, 511, 512, 513, 1023, 1024, 1025, 2049, int(rng.integers(0, 5000))]))
                  for _ in range(b)]
        chunk, use_bg = int(rng.choice([1, 3, 37, 128, 352, 512, 1024, 4096])), bool(rng.integers(0, 2))
        pts = [torch.from_numpy(rng.random((n, 2), dtype=np.float32)) for n in counts]
        tgt = [torch.from_numpy(rng.random(n, dtype=np.float32)) for n in counts]
        ref = bl.pack_batch(pts, tgt, use_background=use_bg, chunk=chunk)
        info, args = bl.pack_host_native(pts, tgt, use_bg, chunk, None, 0)
        assert (info.total_bytes, info.total_chunks, info.multi_chunk) == (ref.total, ref.total_chunks, ref.multi_chunk)
        buf = torch.zeros((info.total_bytes,), dtype=torch.uint8)
        bl.pack_host_native(pts, tgt, use_bg, chunk, buf.data_ptr(), buf.numel(), args)
        assert torch.equal(buf, ref.buf), (counts, chunk, use_bg)


def test_checked_variant_builds_beside_the_product_library():
    """`DGVCC_BOUNDS_CHECK=1` selects libdgvcc_b200_chk.so: same exports, device-side index checks compiled in
    (csrc/common.cuh); the product library reports 0 and carries no assert call."""
    import ctypes
    import subprocess
    from dgvcc_b200 import build
    product = _native.lib()
    assert product.dgvcc_bounds_checked() == 0
    path = build.build(checked=True)          # a no-op when __graft_entry__.build() has been run
    assert path.endswith("libdgvcc_b200_chk.so") and path != product._name
    chk = ctypes.CDLL(path)
    for name in declared_symbols():
        assert hasattr(chk, name), f"{name} missing from the checked variant"
    assert chk.dgvcc_bounds_checked() == 1 and chk.dgvcc_abi_version() == product.dgvcc_abi_version()

    def assert_calls(lib):
        out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-elf", lib], capture_output=True, text=True).stdout
        return out.count("__assertfail")
    if os.path.exists("/usr/local/cuda/bin/cuobjdump"):
        assert assert_calls(path) > 0 and assert_calls(product._name) == 0


def test_device_code_is_the_build_the_gpu_suite_ran_on():
    """profiles/r2d_sass_digest.txt records the SASS digests of the build the full GPU suite last ran on
    (profiles/r2d_gputest_head.log).  Comments, compiled-out checks, host code and Python may change freely; a change of
    the DEVICE code must come with a new GPU run and a regenerated digest file (scripts/sass_digest.py)."""
    import subprocess
    import sys
    obj_dir = os.path.join(ROOT, "dgvcc_b200", "lib", "obj")
    if not (os.path.exists("/usr/local/cuda/bin/cuobjdump") and os.path.isdir(obj_dir)):
        import pytest
        pytest.skip("needs cuobjdump and the object files of an in-tree build")
    _native.lib()   # builds when stale
    recorded = [l.split() for l in open(os.path.join(ROOT, "profiles", "r2d_sass_digest.txt")) if not l.startswith("#")]
    now = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "sass_digest.py")], capture_output=True, text=True)
    assert now.returncode == 0, now.stderr
    assert [l.split() for l in now.stdout.splitlines()] == recorded


def test_no_entry_point_crashes_on_null_or_degenerate_arguments():
    """Error behaviour of the ABI: integer codes, never a crash.  Every exported function is called (i) with null
    pointers and zeros, (ii) with valid host pointers and sizes 0 / -1 and (iii) 1500 times with random small, boundary
    and absurd (2^31 - 1) sizes, in ONE child process (a crash then names the call it died in).  The child sees no
    device, even where there is one: every launcher first hands its stream to the CUDA runtime (the device guard in
    csrc/common.cuh) and only then checks its arguments, and the host pointers the child passes also stand in for stream
    handles.  A runtime without a device rejects such a call with a code; one with a device would dereference them.
    (Found dgvcc_isw_workspace_bytes(0, 0, 0), dgvcc_lw_loss_forward(hw = 0) and overflowing shapes dividing by zero in
    the split-K plans; the ISW-family launchers now check isw_shape_ok first.)"""
    import subprocess
    import sys
    child = r'''
import ctypes, sys
sys.path.insert(0, %r)
from dgvcc_b200 import _native
lib = _native.lib()
buf = ctypes.create_string_buffer(1 << 22)
addr = ctypes.addressof(buf)
for mode in ("null", 0, -1):
    for name in sorted(_native.SIGNATURES):
        if mode != "null" and name in ("dgvcc_peer_free", "dgvcc_peer_close"):   # would hand a host pointer to cudaFree
            continue
        res, args = _native.SIGNATURES[name]
        vals = []
        for a in args:
            is_ptr = a is ctypes.c_void_p or (hasattr(a, "_type_") and not isinstance(a._type_, str))
            if is_ptr:
                vals.append(None if mode == "null" else (ctypes.c_void_p(addr) if a is ctypes.c_void_p else ctypes.cast(addr, a)))
            elif a in (ctypes.c_float, ctypes.c_double):
                vals.append(0.0)
            elif a is ctypes.c_size_t:
                vals.append(0 if mode == "null" else 1 << 22)
            else:
                vals.append(0 if mode == "null" else mode)
        print("calling", name, mode, flush=True)
        getattr(lib, name)(*vals)
# (iii) random small / boundary / absurd sizes with valid host pointers (the host-only writers get small sizes only)
import random
rng = random.Random(20261019)
writers = {"dgvcc_bl_pack_host", "dgvcc_dmap_batch_plan"}
skip = {"dgvcc_peer_free", "dgvcc_peer_close", "dgvcc_peer_export", "dgvcc_peer_open", "dgvcc_peer_alloc"}
pool = sorted(set(_native.SIGNATURES) - skip)
for it in range(1500):
    name = rng.choice(pool)
    res, args = _native.SIGNATURES[name]
    big = name not in writers and rng.random() < 0.3
    vals = []
    for a in args:
        if a is ctypes.c_void_p:
            vals.append(ctypes.c_void_p(addr))
        elif hasattr(a, "_type_") and not isinstance(a._type_, str):
            vals.append(ctypes.cast(addr, a))
        elif a in (ctypes.c_float, ctypes.c_double):
            vals.append(rng.choice([0.0, 1.0, 8.0, -1.0, 1e30, float("nan")]))
        elif a is ctypes.c_size_t:
            vals.append(rng.choice([0, 16, 1 << 22]))
        else:
            vals.append(rng.choice([0, 1, 2, 3, 5, 31, 32, 33, 64, 100, -1] + ([2 ** 31 - 1, 2 ** 30, 65536] if big else [])))
    print("calling", name, [v for v in vals if isinstance(v, (int, float))], flush=True)
    getattr(lib, name)(*vals)
print("survived", flush=True)
''' % ROOT
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "-c", child], capture_output=True, text=True, timeout=300, env=env)
    last = (p.stdout.strip().splitlines() or ["<nothing>"])[-1]
    assert p.returncode == 0 and last == "survived", f"child rc={p.returncode}, last line: {last}\n{p.stderr[-600:]}"


def test_ctypes_signatures_match_the_header_prototypes():
    """Argument by argument: every prototype of include/dgvcc_b200.h against dgvcc_b200._native.SIGNATURES (pointer /
    int / int64_t / size_t / float / double, and the return type) -- a wrong ctypes width is silent garbage on the GPU."""
    import ctypes
    text = open(os.path.join(ROOT, "include", "dgvcc_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = re.findall(r"\b(int|size_t)\s+(dgvcc_\w+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S)
    assert {p[1] for p in protos} == set(_native.SIGNATURES)

    def c_kind(arg):
        arg = " ".join(arg.split())
        if arg in ("void", ""):
            return None
        if "*" in arg:
            return "ptr"
        for token, kind in (("int64_t", "i64"), ("size_t", "size"), ("double", "f64"), ("float", "f32"), ("int", "i32")):
            if re.search(rf"\b{token}\b", arg):
                return kind
        raise AssertionError(f"unclassified C argument: {arg}")

    def py_kind(a):
        if a is ctypes.c_void_p or (hasattr(a, "_type_") and not isinstance(a._type_, str)):
            return "ptr"
        return {ctypes.c_int64: "i64", ctypes.c_size_t: "size", ctypes.c_double: "f64", ctypes.c_float: "f32",
                ctypes.c_int: "i32"}[a]

    for ret, name, args in protos:
        res, py_args = _native.SIGNATURES[name]
        assert res is {"int": ctypes.c_int, "size_t": ctypes.c_size_t}[ret], name
        assert [k for k in map(c_kind, args.split(",")) if k] == [py_kind(a) for a in py_args], name


def test_header_is_plain_c_and_links_from_a_c_program(tmp_path):
    """The boundary is a C ABI: include/dgvcc_b200.h compiles as strict C99 (and as C++), and a C program linked against
    the library calls an entry point -- no torch, no Python, no C++ runtime needed by the caller."""
    import shutil
    import subprocess
    if not shutil.which("gcc"):
        import pytest
        pytest.skip("no gcc")
    lib = _native.lib()
    inc, libdir = os.path.join(ROOT, "include"), os.path.dirname(lib._name)
    src = tmp_path / "caller.c"
    src.write_text('#include <stdio.h>\n#include "dgvcc_b200.h"\n'
                   'int main(void) {\n'
                   '    dgvcc_bl_layout lay;\n'
                   '    int rc = dgvcc_bl_workspace_layout(1000, 3, 2, 48, 64, &lay);\n'
                   '    printf("%d %d %d\\n", dgvcc_abi_version(), rc, dgvcc_bl_workspace_layout(0, 1, 1, 8, 8, &lay));\n'
                   '    return 0;\n}\n')
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", inc, str(src)], check=True)
    if shutil.which("g++"):
        cpp = tmp_path / "caller.cpp"
        cpp.write_text('#include "dgvcc_b200.h"\nint main() { return dgvcc_abi_version() > 0 ? 0 : 1; }\n')
        subprocess.run(["g++", "-std=c++11", "-Wall", "-Werror", "-fsyntax-only", "-I", inc, str(cpp)], check=True)
    exe = tmp_path / "caller"
    subprocess.run(["gcc", "-std=c99", "-I", inc, str(src), "-o", str(exe), "-L", libdir, "-ldgvcc_b200",
                    f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert int(out[0]) == lib.dgvcc_abi_version() and out[1:] == ["0", "-1"]


def test_ctypes_structures_mirror_the_header_structs(tmp_path):
    """Field by field: name, offset and size of every struct dgvcc_b200._native mirrors, measured by a C program
    compiled against the header (a field the header does not have fails to compile)."""
    import ctypes
    import shutil
    import subprocess
    if not shutil.which("gcc"):
        import pytest
        pytest.skip("no gcc")
    mirrors = {"dgvcc_bl_layout": _native.BLLayout, "dgvcc_bl_packed": _native.BLPacked,
               "dgvcc_bl_shard": _native.BLShard, "dgvcc_dmap_plan": _native.DmapPlan}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dgvcc_b200.h"', 'int main(void) {']
    for cname, cls in mirrors.items():
        lines.append(f'    printf("{cname} %zu\\n", sizeof({cname}));')
        for field, _ in cls._fields_:
            lines.append(f'    printf("{cname}.{field} %zu %zu\\n", offsetof({cname}, {field}), sizeof((({cname}*)0)->{field}));')
    lines += ['    return 0;', '}']
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines) + "\n")
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict((l.split()[0], [int(v) for v in l.split()[1:]]) for l in
               subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in mirrors.items():
        assert got[cname] == [ctypes.sizeof(cls)], cname
        for field, ftype in cls._fields_:
            assert got[f"{cname}.{field}"] == [getattr(cls, field).offset, ctypes.sizeof(ftype)], f"{cname}.{field}"
    assert _native.BL_PHASES == 8 and _native.DMAP_META_COLS == 12   # DGVCC_BL_PHASES, DGVCC_DMAP_META_COLS
