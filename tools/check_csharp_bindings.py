"""Static check of integration/B200Native.cs against include/cnhe.h and the reference's interfaces (no .NET toolchain in the image).

1. every prototype of include/cnhe.h has exactly one [DllImport] with the same name, the same number of parameters and, per
   parameter, a C# type the C type may marshal as (pointers -> IntPtr / arrays / out scalars, size_t -> UIntPtr, ...);
2. every member of the reference's IVector / IMatrix / IFactory / IComputationEnvironment interfaces is implemented by the B200
   classes (the lists below, which must equal the member names recorded from the reference's interface files in
   tests/golden/reference_interfaces.json).

Run directly (exit code 1 on a mismatch) or through tests/test_abi_exports.py."""
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ALLOWED = {
    "cnhe_ctx *": {"IntPtr"}, "const cnhe_ctx *": {"IntPtr"}, "cnhe_vec *": {"IntPtr"}, "const cnhe_vec *": {"IntPtr"},
    "cnhe_ctx **": {"out IntPtr"}, "cnhe_vec **": {"out IntPtr", "IntPtr[]"},
    "const cnhe_vec *const *": {"IntPtr[]"}, "cnhe_vec *const *": {"IntPtr[]"},
    "const uint64_t *": {"ulong[]", "IntPtr"}, "uint64_t *": {"ulong[]", "IntPtr", "out ulong"},
    "const double *": {"double[]"}, "double *": {"double[]", "out double"},
    "int *": {"out int", "int[]"}, "const int *": {"int[]"}, "const int32_t *": {"int[]"}, "int32_t *": {"int[]"},
    "uint32_t *": {"out uint"}, "float *": {"out float"}, "size_t *": {"out UIntPtr"}, "size_t": {"UIntPtr"},
    "const char *": {"string", "byte[]"}, "char *": {"byte[]"}, "uint8_t *": {"byte[]"}, "const uint8_t *": {"byte[]"},
    "int": {"int"}, "uint32_t": {"uint"}, "uint64_t": {"ulong"}, "int64_t": {"long"}, "double": {"double"},
}
RETURNS = {"int": "int", "const char *": "IntPtr", "uint64_t": "ulong"}

# interface members of the reference (HE Wrapper/IVector.cs:20-136, IMatrix.cs:18-122, IFactory.cs:20-130, IComputationEnvironment.cs)
IVECTOR = ["Decrypt", "DecryptFullPrecision", "Write", "Data", "Subtract", "Add", "DotProduct", "PointwiseMultiply", "SumAllSlots", "Duplicate",
           "Rotate", "Permute", "Dim", "Scale", "RegisterScale", "IsEncrypted", "IsSigned", "BlockSize", "Format", "Dispose"]
IMATRIX = ["Decrypt", "Write", "Mul", "Add", "ElementWiseMultiply", "RowCount", "ColumnCount", "Data", "Scale", "RegisterScale", "Format", "GetColumn",
           "GetRow", "SetColumn", "IsEncrypted", "BlockSize", "DataDisposedExternaly", "ConvertToColumnVector", "Interleave", "Dispose"]
IFACTORY = ["GetPlainVector", "GetEncryptedVector", "GetValueFromString", "GetStringFromValue", "CopyVector", "LoadVector", "GetPlainMatrix",
            "GetEncryptedMatrix", "GetMatrix", "LoadMatrix", "AllocateComputationEnv", "FreeComputationEnv", "Save"]
IENV = ["ParentFactory", "Primes"]


def c_prototypes():
    h = open(os.path.join(ROOT, "include", "cnhe.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    out = {}
    for ret, name, args in re.findall(r"^\s*((?:const\s+)?[A-Za-z_0-9]+\s*\**)\s*(cnhe_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", h, flags=re.M):
        args = re.sub(r"\s+", " ", args.strip())
        params = [] if args == "void" else [a.strip() for a in args.split(",")]
        types = []
        for a in params:
            m = re.match(r"^(.*?[\s\*])([A-Za-z_][A-Za-z_0-9]*)$", a)
            t = m.group(1) if m and m.group(2) not in ("int", "char", "double", "uint64_t", "uint32_t", "size_t") else a
            types.append(re.sub(r"\s+", " ", t.strip()))
        out[name] = (re.sub(r"\s+", " ", ret.strip()), types)
    return out


def cs_imports(src):
    out = {}
    for ret, name, args in re.findall(r"\[DllImport\([^\]]*\)\]\s*public static extern (\w+) (cnhe_\w+)\(([^)]*)\);", src):
        params = [a.strip() for a in args.split(",")] if args.strip() else []
        out.setdefault(name, []).append((ret, [" ".join(p.split()[:-1]) for p in params]))
    return out


def interface_members(path, fallback):
    try:
        src = open(path, encoding="utf-8-sig").read()
    except OSError:
        return fallback
    body = src[src.index("interface"):]
    names = set(re.findall(r"\b([A-Z][A-Za-z]+)\s*(?:\(|\{\s*get)", body))
    return sorted(names | {"Dispose"} if "IDisposable" in body.split("{")[0] else names)


def class_body(src, name):
    i = src.index("class " + name)
    depth, j = 0, src.index("{", i)
    for k in range(j, len(src)):
        depth += src[k] == "{"
        depth -= src[k] == "}"
        if depth == 0:
            return src[j:k]
    raise ValueError(name)


def check():
    errors = []
    src = open(os.path.join(ROOT, "integration", "B200Native.cs")).read()
    protos, imports = c_prototypes(), cs_imports(src)
    for name, (ret, types) in protos.items():
        if name not in imports:
            errors.append("no [DllImport] for %s" % name)
            continue
        if len(imports[name]) != 1:
            errors.append("%s is imported %d times" % (name, len(imports[name])))
        cret, ctypes_ = imports[name][0]
        if RETURNS.get(ret) != cret:
            errors.append("%s: return type %s does not marshal %s" % (name, cret, ret))
        if len(ctypes_) != len(types):
            errors.append("%s: %d parameters in C#, %d in cnhe.h" % (name, len(ctypes_), len(types)))
            continue
        for i, (ct, cs) in enumerate(zip(types, ctypes_)):
            if cs not in ALLOWED.get(ct, set()):
                errors.append("%s: parameter %d is `%s` in cnhe.h but `%s` in C#" % (name, i, ct, cs))
    for name in imports:
        if name not in protos:
            errors.append("[DllImport] %s is not declared in include/cnhe.h" % name)
    with open(os.path.join(ROOT, "tests", "golden", "reference_interfaces.json")) as f:
        reference = json.load(f)
    for cls, iface, members in (("B200BfvVector", "IVector", IVECTOR), ("B200BfvMatrix", "IMatrix", IMATRIX), ("B200BfvFactory", "IFactory", IFACTORY),
                                ("B200BfvEnvironment", "IComputationEnvironment", IENV)):
        found = set(reference[iface])
        if set(members) != found:
            errors.append("%s: member list in this script differs from the reference: %s" % (iface, sorted(found ^ set(members))))
        body = class_body(src, cls)
        for m in members:
            if not re.search(r"\bpublic\b[^;{=]*\b%s\b\s*(\(|\{|=>|;)" % m, body) and not re.search(r"\bpublic\b[^;{(]*\b%s\b" % m, body):
                errors.append("%s does not implement %s.%s" % (cls, iface, m))
    return errors, len(protos)


if __name__ == "__main__":
    errs, n = check()
    for e in errs:
        print("MISMATCH:", e)
    print("%d C prototypes checked against integration/B200Native.cs: %s" % (n, "OK" if not errs else "%d problems" % len(errs)))
    sys.exit(1 if errs else 0)
