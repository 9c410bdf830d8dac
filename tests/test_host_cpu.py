"""CPU tests of the host side: C-ABI library loads and exports every symbol the headers declare (no compute calls
without a GPU), SDPA reader / model preparation, option handling and clean errors."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import jump_examples as je

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(lrn_[A-Za-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol(pkg):
    from loraine_jl_b200 import _lib
    L = C.CDLL(_lib.LIB_PATH)
    names = _declared("loraine_b200.h") + _declared("loraine_b200_debug.h") + _declared("loraine_b200_dd.h")
    assert len(names) >= 60
    for n in names:
        assert hasattr(L, n), n
    assert set(_lib.DECLARED_SYMBOLS) <= set(names)
    assert set(_lib.DD_SYMBOLS) == set(_declared("loraine_b200_dd.h"))


def test_timer_names_follow_the_reference_sections(pkg):
    """TimerOutputs section names of the reference (src/makeBBBB.jl:2,30, src/prepare_W.jl:37, src/Solvers.jl:676)."""
    from loraine_jl_b200 import _lib
    L = _lib.lib()
    names = [L.lrn_timer_name(i, 0).decode() for i in range(len(_lib.T_NAMES))]
    assert names[2] == "BBBBs" and L.lrn_timer_name(2, 1) == b"BBBB_rank1"
    assert names[10] == "prep W SVD" and names[7] == "prec"
    assert L.lrn_timer_name(99, 0) is None


def test_create_without_gpu_fails_loudly(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    n, bs, c, body = pkg.problems.theta_torus(4, 6)
    opt = pkg.Optimizer()
    opt.set_attribute("verb", 0)
    opt.copy_to(pkg.raw_from_sdpa_arrays(n, bs, c, body))
    with pytest.raises(Exception) as ei:
        opt.optimize()
    assert "no CPU fallback" in str(ei.value) or "no usable" in str(ei.value)


def test_non_float64_is_rejected(pkg):
    """north_star: Optimizer{Float64xN} errors cleanly instead of falling back (examples/k.jl:8 uses Float64x2)."""
    with pytest.raises(TypeError):
        pkg.Optimizer(T=np.float32)
    with pytest.raises(TypeError):
        pkg.Optimizer(T="Float64x3")
    # Float64x2 exists for models WITHOUT PSD blocks only (double-double LP path); a semidefinite model is rejected
    opt = pkg.Optimizer(T="Float64x2")
    with pytest.raises(TypeError):
        opt.copy_to(pkg.RawProblem(**je.fields(je.ex_corr("Max"))))
    md = pkg.prepare_model(pkg.RawProblem(**je.fields(je.ex_k_lp())))
    with pytest.raises(TypeError):
        pkg.load(md, dict(verb=0), T=np.longdouble)


def test_options_surface(pkg):
    """RawOptimizerAttribute keys = DEFAULT_OPTIONS (src/Solvers.jl:169-185, src/MOI_wrapper.jl:86-103)."""
    want = {"kit": 0, "tol_cg": 1e-2, "tol_cg_up": 0.5, "tol_cg_min": 1e-7, "eDIMACS": 1e-7, "preconditioner": 1, "erank": 1,
            "aamat": 1, "fig_ev": 0, "verb": 1, "datarank": 0, "initpoint": 0, "timing": 1, "maxit": 100, "datasparsity": 8}
    assert pkg.DEFAULT_OPTIONS == want
    opt = pkg.Optimizer()
    with pytest.raises(KeyError):
        opt.set_attribute("no_such_option", 1)
    opt.set_attribute("kit", 1)
    assert opt.get_attribute("kit") == 1


def test_load_parameter_checks(pkg, capsys):
    """src/Solvers.jl:263-291"""
    md = pkg.prepare_model(pkg.RawProblem(**je.fields(je.ex_corr("Max"))))
    s, _ = pkg.load(md, dict(verb=0, kit=7, erank=-2, datarank=-5, initpoint=3))
    assert (s.kit, s.erank, s.datarank, s.initpoint) == (0, 1, 0, 1)
    s, _ = pkg.load(md, dict(verb=0, kit=1, tol_cg=1e-9, tol_cg_min=1e-3, eDIMACS=1e-5, preconditioner=9))
    assert s.tol_cg == 1e-3 and s.tol_cg_min == 1e-5 and s.preconditioner == 1


def test_sdpa_roundtrip_and_model(pkg, tmp_path, golden_dir):
    z = np.load(os.path.join(golden_dir, "vib3.npz"))
    n, bs, c, body = int(z["n"]), [int(b) for b in z["bs"]], z["c"], z["body"]
    f = tmp_path / "p.dat-s"
    pkg.model.write_sdpa(str(f), n, bs, c, body)
    n2, bs2, c2, body2 = pkg.read_sdpa(str(f))
    assert n2 == n and bs2 == bs
    np.testing.assert_array_equal(c2, c)
    np.testing.assert_array_equal(body2, body)
    raw = pkg.raw_from_sdpa_arrays(n, bs, c, body)
    md = pkg.prepare_model(raw)
    assert md.nlmi == sum(1 for b in bs if b > 0) and md.nlin == -sum(b for b in bs if b < 0)
    for i, m in enumerate(md.msizes):
        assert md.AA[i].shape == (n, m * m)
        # both triangles stored: AA row k reshaped is symmetric
        k = int(np.argmax(md.nzA[:, i]))
        M = md.AA[i][k].toarray().reshape(m, m, order="F")
        np.testing.assert_array_equal(M, M.T)
    assert (np.diff(md.nzA[md.sigmaA[:, 0], 0]) <= 0).all()       # nnz-descending order


def test_rank_one_factors(pkg):
    n, bs, c, body = pkg.problems.theta_torus(3, 4)
    md = pkg.prepare_model(pkg.raw_from_sdpa_arrays(n, bs, c, body), datarank=-1)
    m = md.msizes[0]
    for k in (0, m - 1, m, n - 1):
        bk = md.B[0][k].toarray().ravel()
        Ak = -md.AA[0][k].toarray().reshape(m, m, order="F")
        np.testing.assert_allclose(np.outer(bk, bk), Ak, atol=1e-12)
    n, bs, c, body = pkg.problems.large_schur(12, 30, 1)
    with pytest.raises(ValueError):
        pkg.prepare_model(pkg.raw_from_sdpa_arrays(n, bs, c, body), datarank=-1)


def test_generators_shapes(pkg):
    n, bs, c, body = pkg.problems.maxcut_torus(6, 8, 1)
    assert n == 48 and bs == [48] and (body[body[:, 0] > 0][:, 2] == body[body[:, 0] > 0][:, 3]).all()
    n, bs, c, body = pkg.problems.multiblock_lp(3, 10, 7, 5)
    assert n == 30 and bs == [10, 10, 10, -7]
    n, bs, c, body = pkg.problems.large_schur(20, 60, 3)
    cnt = np.bincount(body[body[:, 0] > 0][:, 0].astype(int))[1:]
    assert n == 60 and (cnt >= 1).all() and cnt.max() <= 15


def test_full_size_checker_matches_oracle_assembly(pkg):
    """The sampled-entry checker of the full-size GPU test (tests/test_gpu_solver.py::schur_entry_ref, the defining formula
    tr(A_j W A_k W) of src/makeBBBB.jl:39-64) agrees with the oracle's Schur assembly on a small instance of the same family."""
    import importlib.util
    from oracle import loraine_oracle as lo, sdpa_io
    spec = importlib.util.spec_from_file_location("tgs", os.path.join(os.path.dirname(__file__), "test_gpu_solver.py"))
    tgs = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tgs)
    arrays = pkg.problems.large_schur(m=30, n=200, seed=3)
    md = lo.prepare_model(sdpa_io.raw_from_sdpa_arrays(*arrays), datarank=0, kappa=8)
    rng = np.random.default_rng(1)
    Q = rng.standard_normal((30, 30))
    W = Q @ Q.T / 30 + np.eye(30)
    H = lo.makeBBBBs(md, [W])
    AA = md.AA[0].tocsr()
    err = max(abs(tgs.schur_entry_ref(AA, W, j, k) - H[max(j, k), min(j, k)]) for j in range(0, 200, 7) for k in range(0, 200, 11))
    assert err <= 1e-12 * np.abs(H).max()


@pytest.mark.parametrize("name,datarank", [("theta1", 0), ("control1", 0), ("tru3", 0), ("vib3", 0), ("maxcut", -1), ("c4mini", 0)])
def test_native_model_preparation_matches_the_python_host(pkg, golden_dir, name, datarank):
    """lrn_create_from_triplets' host side (csrc/model.cu: prep_AA!, C = -A[i,1], prep_B, C_lin / d_lin / b conventions of
    src/model.jl:120-229 and src/MOI_wrapper.jl:186-217) against model.py on the same SDPA triplets -- no device needed."""
    import scipy.sparse as sp
    from loraine_jl_b200 import _lib
    L = _lib.lib()
    if name == "maxcut":
        n, bs, c, body = pkg.problems.maxcut_torus(6, 8, 3)
    elif name == "c4mini":
        n, bs, c, body = pkg.problems.multiblock_lp(5, 20, 40, 50)
    else:
        z = np.load(os.path.join(golden_dir, name + ".npz"))
        n, bs, c, body = int(z["n"]), [int(b) for b in z["bs"]], z["c"], z["body"]
    md = pkg.prepare_model(pkg.raw_from_sdpa_arrays(n, bs, c, body), datarank=datarank, kappa=8)
    body = np.asarray(body, float).reshape(-1, 5)
    tk, tb, ti, tj = (np.ascontiguousarray(body[:, k], dtype=np.int64) for k in range(4))
    tv = np.ascontiguousarray(body[:, 4])
    bsa = np.array(bs, dtype=np.int64)
    cc = np.ascontiguousarray(c, dtype=np.float64)
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))

    def fetch(iblk, which, shape, veclen):
        cap = 4 * body.shape[0] + 16
        colptr = np.zeros(shape[1] + 1, dtype=np.int64)
        rowval = np.zeros(cap, dtype=np.int64)
        nzval = np.zeros(cap)
        vec = np.zeros(max(1, veclen))
        nnz = L.lrn_dbg_model_block(n, len(bs), ip(bsa), tv.shape[0], ip(tk), ip(tb), ip(ti), ip(tj), dp(tv), dp(cc), datarank,
                                    iblk, which, cap, ip(colptr), ip(rowval), dp(nzval), dp(vec) if veclen else None)
        assert nnz >= 0, nnz
        return sp.csc_matrix((nzval[:nnz], rowval[:nnz], colptr), shape=shape), vec[:veclen]

    def same(A, B):
        D = (sp.csc_matrix(A) - sp.csc_matrix(B))
        return (abs(D).max() if D.nnz else 0.0) <= 1e-9 * max(1.0, abs(sp.csc_matrix(B)).max() if sp.csc_matrix(B).nnz else 1.0)

    for i, m in enumerate(md.msizes):
        AA, b = fetch(i, 0, (n, m * m), n)
        assert same(AA, md.AA[i]) and AA.nnz == sp.csc_matrix(md.AA[i]).nnz
        assert np.array_equal(b, md.b)
        Ci, _ = fetch(i, 1, (m, m), 0)
        assert same(Ci, md.C[i])
        if datarank == -1:
            Bi, _ = fetch(i, 2, (n, m), 0)
            Bd, Br = Bi.toarray(), md.B[i].toarray()
            sgn = np.sign(np.sum(Bd * Br, axis=1)); sgn[sgn == 0] = 1          # b_k is defined up to its sign
            assert np.abs(Bd - sgn[:, None] * Br).max() <= 1e-9
    if md.nlin:
        Cl, d = fetch(0, 3, (n, md.nlin), md.nlin)
        assert same(Cl, md.C_lin) and np.allclose(d, md.d_lin, rtol=0, atol=1e-12)


def _build_c_host(tmp_path):
    import subprocess
    from loraine_jl_b200 import _lib
    exe = str(tmp_path / "c_abi_host")
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = ["/usr/bin/gcc", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c_abi_host.c"),
           "-L", libdir, "-lloraine_b200", f"-Wl,-rpath,{libdir}", "-lm", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_plain_c_host_compiles_against_the_header_only(pkg, tmp_path):
    """tests/c_abi_host.c drives a whole solve through include/loraine_b200.h (no torch types, no Python): it must compile as
    C (not C++) with -Wall -Werror and link against the shared library alone; without a GPU it must fail loudly."""
    import subprocess
    import torch
    exe = _build_c_host(tmp_path)
    if not torch.cuda.is_available():
        from loraine_jl_b200 import model as M
        z = np.load(os.path.join(ROOT, "tests", "golden", "theta1.npz"))
        path = str(tmp_path / "theta1.dat-s")
        M.write_sdpa(path, int(z["n"]), [int(b) for b in z["bs"]], z["c"], z["body"])
        r = subprocess.run([exe, path], capture_output=True, text=True)
        assert r.returncode == 2 and "no CPU fallback" in r.stderr


def _c_prototypes():
    """{entry point: number of parameters} from the three headers."""
    protos = {}
    for header in ("loraine_b200.h", "loraine_b200_debug.h", "loraine_b200_dd.h"):
        txt = open(os.path.join(ROOT, "include", header)).read()
        txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
        for m in re.finditer(r"\b(lrn_[A-Za-z0-9_]+)\s*\(([^;{]*?)\)\s*;", txt, flags=re.S):
            args = m.group(2).strip()
            protos[m.group(1)] = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
    return protos


def _c_param_types():
    """{entry point: [Julia ccall types each C parameter may be bound to]}"""
    def julia_types(decl):
        d = " ".join(decl.replace("const", " ").split())
        is_array = "[" in d
        d = re.sub(r"\[[0-9]*\]", "", d)
        stars = d.count("*")
        base = re.sub(r"\b[A-Za-z_][A-Za-z0-9_]*$", "", d.replace("*", " ")).strip() or d.replace("*", " ").strip()
        base = base.split()[0]
        if is_array:
            stars += 1
        prim = {"int32_t": "Int32", "int64_t": "Int64", "double": "Float64"}
        if base in ("lrn_handle_t", "lrn_dd_handle_t"):
            return ["Ptr{Cvoid}"] if stars == 0 else ["Ref{Ptr{Cvoid}}", "Ptr{Ptr{Cvoid}}"]
        if base == "lrn_options_t":
            return ["Ref{Options}", "Ptr{Options}"]
        if base == "char":
            return ["Cstring", "Ptr{UInt8}"]
        if base == "void":
            return ["Ptr{Cvoid}", "Ptr{UInt8}"]
        j = prim[base]
        if stars == 0:
            return [j]
        if stars == 1:
            return [f"Ptr{{{j}}}", f"Ref{{{j}}}"]
        return [f"Ptr{{Ptr{{{j}}}}}"]
    out = {}
    for header in ("loraine_b200.h", "loraine_b200_debug.h", "loraine_b200_dd.h"):
        txt = open(os.path.join(ROOT, "include", header)).read()
        txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
        for m in re.finditer(r"\b(lrn_[A-Za-z0-9_]+)\s*\(([^;{]*?)\)\s*;", txt, flags=re.S):
            args = m.group(2).strip()
            out[m.group(1)] = [] if args in ("", "void") else [julia_types(a.strip()) for a in args.split(",")]
    return out


def _julia_ccalls(path):
    """[(entry point, number of argument types, number of arguments)] of every ccall in a Julia source file."""
    src = open(path).read()
    out = []
    for m in re.finditer(r"ccall\(\(:(lrn_[A-Za-z0-9_]+),\s*LIB\[\]\),", src):
        i = m.end()
        depth, j, parts, cur = 1, i, [], ""
        while depth > 0:                      # split the rest of the ccall(...) at top-level commas
            ch = src[j]
            if ch in "([{":
                depth += 1
            elif ch in ")]}":
                depth -= 1
                if depth == 0:
                    break
            if ch == "," and depth == 1:
                parts.append(cur.strip())
                cur = ""
            else:
                cur += ch
            j += 1
        parts.append(cur.strip())
        ret, types, args = parts[0], parts[1], parts[2:]
        assert types.startswith("(") and types.endswith(")"), (m.group(1), types)
        inner = types[1:-1].strip()
        # split the type tuple at its top-level commas (Ref{Ptr{Cvoid}} contains braces, not commas, but be safe)
        tparts, d, cur = [], 0, ""
        for ch in inner:
            if ch in "({[":
                d += 1
            elif ch in ")}]":
                d -= 1
            if ch == "," and d == 0:
                tparts.append(cur.strip())
                cur = ""
            else:
                cur += ch
        if cur.strip():
            tparts.append(cur.strip())
        nargs = len([a for a in args if a != ""])
        if any(a.endswith("...") for a in args):           # csc(A)... splats three arrays
            nargs += 2 * sum(1 for a in args if a.endswith("..."))
        out.append((m.group(1), ret, len(tparts), nargs, tparts))
    return out


@pytest.mark.parametrize("fname", ["LoraineB200.jl", "LoraineB200DD.jl"])
def test_julia_ccalls_match_the_headers(fname):
    """The Julia shims cannot be executed here (no Julia): at least every ccall must name an exported entry point with the
    header's number of parameters, pass as many arguments as it declares types, and use the header's return type."""
    protos = _c_prototypes()
    calls = _julia_ccalls(os.path.join(ROOT, "julia", fname))
    assert len(calls) >= 15
    ctypes_ = _c_param_types()
    for name, ret, ntypes, nargs, jtypes in calls:
        assert name in protos, name
        assert ntypes == protos[name], (name, ntypes, protos[name])
        assert nargs == ntypes, (name, nargs, ntypes)
        for k, (jt, allowed) in enumerate(zip(jtypes, ctypes_[name])):          # Int32 vs Int64, Float64 vs pointer, ...
            assert jt in allowed, (name, k, jt, allowed)
        want = "Cstring" if name.endswith("last_error") else ("Int64" if name == "lrn_kernel_launches" else "Int32")
        assert ret == want, (name, ret)


def test_options_struct_layout_is_the_same_in_c_python_and_julia(pkg):
    """lrn_options_t (include/loraine_b200.h) = _lib.lrn_options_t (ctypes) = struct Options (julia/LoraineB200.jl): same
    fields, order and widths -- the struct crosses the boundary by pointer."""
    import ctypes as C
    from loraine_jl_b200 import _lib
    txt = open(os.path.join(ROOT, "include", "loraine_b200.h")).read()
    body = re.search(r"typedef struct lrn_options \{(.*?)\} lrn_options_t;", txt, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    c_fields = [(m.group(2), m.group(1)) for m in re.finditer(r"\b(int32_t|double)\s+(\w+)\s*;", body)]
    py_fields = [(n, {C.c_int32: "int32_t", C.c_double: "double"}[t]) for n, t in _lib.lrn_options_t._fields_]
    assert c_fields == py_fields
    jl = open(os.path.join(ROOT, "julia", "LoraineB200.jl")).read()
    jbody = re.search(r"struct Options[^\n]*\n(.*?)\nend", jl, flags=re.S).group(1)
    j_fields = [(m.group(1), {"Int32": "int32_t", "Float64": "double"}[m.group(2)]) for m in re.finditer(r"(\w+)::(Int32|Float64)", jbody)]
    assert j_fields == c_fields
    assert C.sizeof(_lib.lrn_options_t) == 8 * 4 + 2 * 8 + 2 * 4


def _reference_src():
    """src/ of a Loraine.jl v0.2.5 checkout named by LORAINE_JL_DIR; the repository does not carry the Julia sources"""
    d = os.environ.get("LORAINE_JL_DIR")
    if not d or not os.path.isdir(os.path.join(d, "src")):
        pytest.skip("reference sources not present (set LORAINE_JL_DIR to a Loraine.jl checkout)")
    return os.path.join(d, "src")


@pytest.mark.parametrize("fname", ["LoraineB200.jl", "LoraineB200DD.jl"])
def test_julia_shim_overrides_existing_reference_methods(fname):
    """Every `function S.name(...)` of the shims must be a method of a function the reference defines in module Solvers with the
    same number of positional arguments, and every `invoke(S.name, Tuple{...}, ...)` must name as many types.  Reads the
    reference sources: skipped unless LORAINE_JL_DIR names a checkout of Loraine.jl."""
    ref = _reference_src()
    defs = {}
    for f in ("Solvers.jl", "predictor_corrector.jl", "prepare_W.jl", "initial_point.jl"):
        for m in re.finditer(r"^function\s+(\w+)\(([^)]*)\)", open(os.path.join(ref, f)).read(), flags=re.M):
            args = [a for a in m.group(2).split(";")[0].split(",") if a.strip()]
            defs.setdefault(m.group(1), set()).add(len(args))
    src = open(os.path.join(ROOT, "julia", fname)).read()
    overrides = re.findall(r"^function S\.(\w+)\(([^)]*)\)", src, flags=re.M)
    assert len(overrides) >= 10
    for name, args in overrides:
        n = len([a for a in args.split(",") if a.strip()])
        assert name in defs, name
        assert n in defs[name], (name, n, defs[name])
    for m in re.finditer(r"invoke\(S\.(\w+),\s*Tuple\{([^}]*(?:\{[^}]*\})?[^}]*)\}", src):
        name = m.group(1)
        ntypes = len([t for t in re.sub(r"\{[^}]*\}", "", m.group(2)).split(",") if t.strip()])
        assert name in defs and ntypes in defs[name], (name, ntypes, defs.get(name))


@pytest.mark.parametrize("fname", ["LoraineB200.jl", "LoraineB200DD.jl"])
def test_julia_shim_uses_existing_solver_and_model_fields(fname):
    """Every `solver.field` / `md.field` the shims touch must be a field of the reference's MySolver / MyModel structs
    (src/Solvers.jl:18-107, src/model.jl:34-60).  Skipped unless LORAINE_JL_DIR names a checkout of Loraine.jl."""
    ref = _reference_src()

    def struct_fields(path, name):
        txt = open(path).read()
        body = re.search(r"mutable struct " + name + r"[^\n]*\n(.*?)\n\s*function ", txt, flags=re.S).group(1)
        return {m.group(1) for m in re.finditer(r"^\s*(\w+)(?:::[^\n]*)?\s*(?:#.*)?$", body, flags=re.M) if m.group(1) not in ("end",)}

    solver_fields = struct_fields(os.path.join(ref, "Solvers.jl"), "MySolver")
    model_fields = struct_fields(os.path.join(ref, "model.jl"), "MyModel")
    assert {"X", "S", "y", "cholBBBB", "regcount", "alpha_lin", "mu", "sigma", "itertime"} <= solver_fields
    assert {"AA", "C", "b", "C_lin", "d_lin", "nlmi", "nlin", "msizes", "n"} <= model_fields
    src = open(os.path.join(ROOT, "julia", fname)).read()
    src = re.sub(r"#[^\n]*", "", src)
    used_s = set(re.findall(r"\bsolver\.(\w+)", src))
    used_m = set(re.findall(r"\bmd\.(\w+)", src))
    assert used_s and used_s <= solver_fields, sorted(used_s - solver_fields)
    assert used_m <= model_fields, sorted(used_m - model_fields)


def _julia_block_balance(src):
    """(number of block openers, number of `end`s, final bracket depth) of a Julia source, ignoring strings, comments, and
    the `for` / `if` of comprehensions and the `end` of indexing (both live inside brackets)."""
    src = re.sub(r'"""(?:.|\n)*?"""', '""', src)
    src = re.sub(r'"(?:\\.|[^"\\\n])*"', '""', src)
    src = re.sub(r"#[^\n]*", "", src)
    src = re.sub(r"'(?:\\.|[^'\\\n])'", "' '", src)
    tokens = re.findall(r"[A-Za-z_]\w*|[()\[\]{}]|\S", src)
    openers = {"function", "if", "for", "while", "begin", "struct", "module", "try", "let", "do", "quote", "macro"}
    depth = opened = closed = 0
    prev = ""
    for t in tokens:
        if t in "([{":
            depth += 1
        elif t in ")]}":
            depth -= 1
        elif depth == 0 and t in openers and prev != ":" and prev != ".":      # not the symbol :if / a field .begin
            opened += 1
        elif depth == 0 and t == "end" and prev != ":":
            closed += 1
        prev = t
    return opened, closed, depth


@pytest.mark.parametrize("fname", ["LoraineB200.jl", "LoraineB200DD.jl"])
def test_julia_shim_blocks_are_balanced(fname):
    """No Julia parser here: at least brackets close and every block opener has its `end`."""
    opened, closed, depth = _julia_block_balance(open(os.path.join(ROOT, "julia", fname)).read())
    assert depth == 0
    assert opened == closed and opened > 20, (opened, closed)
