"""Check every foreign-function binding of the repo against the C prototypes of include/abo.h:
  * every `ccall((:name, LIB), Ret, (ArgTypes...), ...)` of julia/AboCuda.jl (Julia cannot be executed in the build image,
    so the signatures are verified statically: argument count, integer widths, pointer-ness, pointee types);
  * the ctypes `argtypes` table of abstractbayesopt.jl_b200/_lib.py (argument count, scalar widths, pointer-ness).
Exit code 0 and a one-line summary when everything matches; a list of mismatches otherwise.  Used by
tests/test_ffi_signatures.py."""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def c_prototypes(path=os.path.join(ROOT, "include", "abo.h")):
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(int32_t|const char\s*\*)\s+(abo_\w+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S):
        ret, name, args = m.group(1), m.group(2), " ".join(m.group(3).split())
        params = [] if args in ("", "void") else [a.strip() for a in args.split(",")]
        protos[name] = ("cstring" if "char" in ret else "int32", [classify_c(a) for a in params])
    return protos


def classify_c(a):
    """C parameter -> canonical class: int32 | int64 | uint64 | double | ptr:<pointee> | pptr"""
    a = re.sub(r"\bconst\b", "", a).strip()
    arr = re.search(r"\[\s*\d*\s*\]\s*$", a)
    if arr:                                                           # `double ms[3]` decays to a pointer
        a = a[:arr.start()].strip() + "*"
    stars = a.count("*")
    base = a.replace("*", " ").split()
    typ = base[0] if base else ""
    if stars == 0:
        return {"int32_t": "int32", "int64_t": "int64", "uint64_t": "uint64", "double": "double"}.get(typ, "?" + typ)
    if stars >= 2:
        return "pptr"
    return "ptr:" + {"double": "double", "int64_t": "int64", "int32_t": "int32", "uint8_t": "uint8", "void": "void",
                     "abo_ctx": "void", "abo_gp": "void", "char": "char"}.get(typ, "?" + typ)


JL = {"Int32": "int32", "Int64": "int64", "UInt64": "uint64", "Float64": "double", "Cstring": "cstring", "Ptr{Cvoid}": "ptr:void",
      "Ref{Ptr{Cvoid}}": "pptr", "Ptr{Float64}": "ptr:double", "Ref{Float64}": "ptr:double", "Ptr{Int64}": "ptr:int64",
      "Ref{Int64}": "ptr:int64", "Ptr{Int32}": "ptr:int32", "Ref{Int32}": "ptr:int32", "Ptr{UInt8}": "ptr:uint8"}


def split_top(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch in "({[":
            depth += 1
        if ch in ")}]":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur.strip()); cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur.strip())
    return out


def julia_ccalls(path=os.path.join(ROOT, "julia", "AboCuda.jl")):
    src = open(path).read()
    calls = []
    for m in re.finditer(r"ccall\(\(:(\w+),\s*LIB\),\s*(\w+(?:\{[^}]*\})?),\s*\(", src):
        i = m.end()
        depth, j = 1, i
        while depth:
            depth += {"(": 1, ")": -1}.get(src[j], 0); j += 1
        types = split_top(src[i:j - 1])
        rest = src[j:]
        # count the actual arguments up to the closing parenthesis of the ccall
        depth, k, cur = 1, 0, ""
        while depth:
            ch = rest[k]
            depth += {"(": 1, ")": -1, "[": 1, "]": -1, "{": 1, "}": -1}.get(ch, 0)
            if depth:
                cur += ch
            k += 1
        nargs = len([a for a in split_top(cur.lstrip(", \n")) if a])
        line = src.count("\n", 0, m.start()) + 1
        calls.append((m.group(1), m.group(2), types, nargs, line))
    return calls


def check_julia(protos):
    errs, n = [], 0
    for name, ret, types, nargs, line in julia_ccalls():
        n += 1
        where = f"julia/AboCuda.jl:{line} ccall :{name}"
        if name not in protos:
            errs.append(f"{where}: not declared in include/abo.h"); continue
        cret, cargs = protos[name]
        if JL.get(ret) != cret:
            errs.append(f"{where}: return type {ret} vs {cret}")
        if len(types) != len(cargs):
            errs.append(f"{where}: {len(types)} argument types, the header has {len(cargs)}"); continue
        if nargs != len(types):
            errs.append(f"{where}: {nargs} arguments passed for {len(types)} declared types")
        for q, (jt, ct) in enumerate(zip(types, cargs)):
            cj = JL.get(jt)
            ok = cj == ct or (ct.startswith("ptr:") and cj == "ptr:void" and ct == "ptr:void")
            if not ok:
                errs.append(f"{where}: argument {q + 1} is {jt} ({cj}), the header says {ct}")
    return n, errs


def check_ctypes(protos):
    sys.path.insert(0, ROOT)
    src = open(os.path.join(ROOT, "abstractbayesopt.jl_b200", "_lib.py")).read()
    table = re.search(r"sigs = \{(.*?)\n        \}", src, flags=re.S).group(1)
    errs, n = [], 0
    for m in re.finditer(r'"(abo_\w+)":\s*\[(.*?)\],?\n', table):
        name, args = m.group(1), split_top(m.group(2))
        n += 1
        if name not in protos:
            errs.append(f"_lib.py {name}: not declared in include/abo.h"); continue
        cargs = protos[name][1]
        if len(args) != len(cargs):
            errs.append(f"_lib.py {name}: {len(args)} argtypes, the header has {len(cargs)}"); continue
        for q, (a, ct) in enumerate(zip(args, cargs)):
            cls = {"i32": "int32", "i64": "int64", "u64": "uint64", "dbl": "double"}.get(a, "ptr")
            if (cls == "ptr") != (ct.startswith("ptr") or ct == "pptr") or (cls != "ptr" and cls != ct):
                errs.append(f"_lib.py {name}: argument {q + 1} is {a}, the header says {ct}")
    declared = set(re.findall(r'"(abo_\w+)"', re.search(r"SYMBOLS = \[(.*?)\]", src, flags=re.S).group(1)))
    for name in protos:
        if name not in declared:
            errs.append(f"_lib.py SYMBOLS: {name} of include/abo.h is missing")
    return n, errs


if __name__ == "__main__":
    protos = c_prototypes()
    nj, ej = check_julia(protos)
    nc, ec = check_ctypes(protos)
    for e in ej + ec:
        print(e)
    print(f"{len(protos)} prototypes in include/abo.h; {nj} ccall sites in julia/AboCuda.jl, {nc} ctypes signatures: "
          f"{len(ej) + len(ec)} mismatches")
    sys.exit(1 if ej or ec else 0)
