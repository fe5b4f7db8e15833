"""CPU-only: the ctypes table _lib.SIGNATURES against the prototypes of include/b200seg.h, entry by entry and argument by argument.
A row that disagrees with the header (a missing argument, an int where the header has a float) would corrupt arguments silently
at call time, so it is caught here from the two files alone, without building or loading the library."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_SCALARS = {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "long long": ctypes.c_longlong, "float": ctypes.c_float,
            "double": ctypes.c_double}


def header_prototypes():
    """name -> (return type, [parameter types]) of every b200seg_* prototype, types with names and whitespace normalised"""
    text = open(os.path.join(ROOT, "include", "b200seg.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    text = re.sub(r"^\s*#[^\n]*", " ", text, flags=re.M)
    protos = {}
    for ret, name, params in re.findall(r"B200SEG_API\s+([^;()]*?)\s*\b(b200seg_\w+)\s*\(([^()]*)\)\s*;", text):
        types = []
        for p in params.split(","):
            p = " ".join(p.replace("*", " * ").split())
            if p in ("", "void"):
                continue
            words = p.split()
            if len(words) > 1 and words[-1] != "*":
                words = words[:-1]                        # drop the parameter name
            types.append(" ".join(words))
        protos[name] = (" ".join(ret.replace("*", " * ").split()), types)
    assert len(protos) == len(set(re.findall(r"\b(b200seg_\w+)\s*\(", text))), "a prototype the parser did not read"
    return protos


def _is_int64(t):
    return t is not None and getattr(t, "_type_", None) in ("q", "l") and ctypes.sizeof(t) == 8


def _mismatch(c_type, ct):
    """why ctypes type `ct` cannot carry the C type `c_type`, or None when it can"""
    base = " ".join(w for w in c_type.split() if w not in ("const", "*"))
    if "*" in c_type:
        if ct is ctypes.c_void_p:
            return None
        pointee = ctypes.c_void_p if c_type.count("*") > 1 else _SCALARS.get(base)
        target = getattr(ct, "_type_", None)
        if isinstance(target, type) and pointee is not None and ctypes.sizeof(target) == ctypes.sizeof(pointee):
            return None
        return f"header {c_type!r} wants c_void_p or a POINTER of the same width, ctypes has {ct}"
    if base in ("int64_t", "long long"):
        return None if _is_int64(ct) else f"header {c_type!r} wants a 64-bit integer, ctypes has {ct}"
    if base not in _SCALARS:
        return f"header type {c_type!r} has no ctypes mapping in this test"
    return None if ct is _SCALARS[base] else f"header {c_type!r} wants {_SCALARS[base]}, ctypes has {ct}"


def test_signatures_match_header():
    from rnd_semantic_segmentation_b200._lib import SIGNATURES
    protos = header_prototypes()
    assert len(protos) >= 90
    errors = [f"{name}: declared in include/b200seg.h, no SIGNATURES row" for name in sorted(set(protos) - set(SIGNATURES))]
    errors += [f"{name}: SIGNATURES row, not declared in include/b200seg.h" for name in sorted(set(SIGNATURES) - set(protos))]
    for name in sorted(set(protos) & set(SIGNATURES)):
        ret, params = protos[name]
        restype, argtypes = SIGNATURES[name]
        if ret == "void":
            if restype is not None:
                errors.append(f"{name}: returns void, restype is {restype}")
        elif ret == "const char *":
            if restype is not ctypes.c_char_p:
                errors.append(f"{name}: returns const char*, restype is {restype}")
        elif why := _mismatch(ret, restype):
            errors.append(f"{name}: return value: {why}")
        if len(argtypes) != len(params):
            errors.append(f"{name}: {len(params)} arguments in the header, {len(argtypes)} in SIGNATURES")
            continue
        for i, (c_type, ct) in enumerate(zip(params, argtypes)):
            if why := _mismatch(c_type, ct):
                errors.append(f"{name}: argument {i}: {why}")
    assert not errors, "\n".join(errors)
