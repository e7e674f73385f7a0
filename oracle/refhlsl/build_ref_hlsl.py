#!/usr/bin/env python
"""Builds oracle/_ref/libref_hlsl.so: the REFERENCE'S OWN shader source, compiled for the CPU.

  python oracle/refhlsl/build_ref_hlsl.py <checkout of aras-p/UnityGaussianSplatting> [--keep]

Recipe (TEST INFRASTRUCTURE; nothing here is product code, nothing of the reference is copied into the repo):
  1. read package/Shaders/{GaussianSplatting.hlsl, SphericalHarmonics.hlsl, SplatUtilities.compute,
     RenderGaussianSplats.shader} of the reference checkout named on the command line;
  2. apply the purely syntactic rewrites below (HLSL-only syntax -> C++ spelling; no expression is touched):
       - drop #pragma / #include lines, [numthreads(..)] attributes and `: SEMANTIC` annotations,
       - `out T x` / `inout T x` parameters -> `T& x`,
       - unsuffixed floating literals get an `f` (HLSL literals are float, C++ ones would be double),
       - `(Struct)0` -> `Struct()`, `discard;` -> flag + return,
       - of SplatUtilities.compute only the hot-path / export functions are kept (the edit kernels use atomics and
         writable textures the shim does not model);
  3. write the result to oracle/_ref/ref_cs.inc and ref_ps.inc (intermediates, deleted after a successful build unless
     --keep is given) and compile
     ref_hlsl_harness.cpp, which includes them together with hlsl_shim.hpp, into oracle/_ref/libref_hlsl.so.
The tests do not load the library: tests/golden/make_ref_hlsl_golden.py runs it once and stores what it computed
(tests/golden/ref_hlsl.npz), so the comparison with the reference needs neither its checkout nor this build."""
from __future__ import annotations

import re
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
OUT = HERE.parent / "_ref"

SEMANTIC = re.compile(r"\s*:\s*(SV_\w+|TEXCOORD\d*|COLOR\d*|POSITION\d*)\b")
FLOAT_LIT = re.compile(r"(?<![\w.])((?:\d+\.\d*|\.\d+)(?:[eE][+-]?\d+)?|\d+[eE][+-]?\d+)(?![\w.])")
OUT_PARAM = re.compile(r"\b(?:in)?out\s+(\w+)\s+(\w+)(\s*\[)?")
ZERO_CAST = re.compile(r"\(([A-Za-z_]\w*)\)\s*0\s*;")

KEEP_FUNCS = {"FloatToSortableUint", "CSSetIndices", "CSCalcDistances", "DecomposeCovariance", "IsSplatCut", "CSCalcViewData",
              "ColorToSH0", "InvSigmoid", "RotateSH", "CalcSHRotMatrix", "CSExportData"}
KNOWN_TYPES = {"float", "float2", "float3", "float4", "float3x3", "float4x4", "uint", "int", "half", "half3", "half4", "bool",
               "StructuredBuffer", "RWStructuredBuffer", "ByteAddressBuffer", "RWByteAddressBuffer", "Texture2D", "static"}


def rewrite(text: str) -> str:
    lines = []
    for line in text.splitlines():
        s = line.strip()
        if s.startswith("#pragma") or s.startswith("#include"):
            continue
        lines.append(line)
    text = "\n".join(lines)
    text = re.sub(r"\[numthreads\([^\]]*\)\]", "", text)
    text = SEMANTIC.sub("", text)
    text = OUT_PARAM.sub(lambda m: "%s %s%s" % (m.group(1), m.group(2), m.group(3)) if m.group(3) else "%s& %s" % (m.group(1), m.group(2)), text)
    # literals: not inside preprocessor lines (`#if 0`), not hex
    out = []
    for line in text.splitlines():
        if line.lstrip().startswith("#"):
            out.append(line)
        else:
            out.append(FLOAT_LIT.sub(lambda m: m.group(1) + "f", line))
    text = "\n".join(out)
    text = ZERO_CAST.sub(lambda m: "%s();" % m.group(1), text)
    text = re.sub(r"\bdiscard\s*;", "{ g_discarded = true; return half4(0.0f); }", text)
    return text


def top_level_items(text: str):
    """Split into top-level items: preprocessor lines, declarations (`...;`) and definitions (`... { ... }` [;])."""
    items, i, n = [], 0, len(text)
    while i < n:
        while i < n and text[i] in " \t\r\n":
            i += 1
        if i >= n:
            break
        if text.startswith("//", i):
            j = text.find("\n", i)
            i = n if j < 0 else j + 1
            continue
        if text.startswith("/*", i):
            i = text.find("*/", i) + 2
            continue
        if text[i] == "#":
            j = text.find("\n", i)
            j = n if j < 0 else j
            items.append(text[i:j])
            i = j + 1
            continue
        depth, j = 0, i
        while j < n:
            c = text[j]
            if text.startswith("//", j):
                j = text.find("\n", j)
                j = n if j < 0 else j
                continue
            if c == "{":
                depth += 1
            elif c == "}":
                depth -= 1
                if depth == 0:
                    k = j + 1
                    while k < n and text[k] in " \t\r\n":
                        k += 1
                    j = k + 1 if k < n and text[k] == ";" else j + 1
                    break
            elif c == ";" and depth == 0:
                j += 1
                break
            j += 1
        items.append(text[i:j])
        i = j
    return items


def slice_compute(text: str, sh_text: str) -> str:
    """Keep preprocessor lines, struct definitions, globals of modelled types and the whitelisted functions."""
    text = text.replace('#include "SphericalHarmonics.hlsl"', "@@SH@@")
    kept = []
    for it in top_level_items(rewrite(text.replace("@@SH@@", "\n__SH_MARKER__;\n"))):
        head = it.split("{", 1)[0]
        if it.startswith("#"):
            kept.append(it)
        elif it.strip() == "__SH_MARKER__;":
            kept.append(rewrite(sh_text))
        elif head.lstrip().startswith("struct"):
            kept.append(it)
        elif "{" in it and "(" in head:            # function definition
            name = re.search(r"(\w+)\s*\(", head).group(1)
            if name in KEEP_FUNCS:
                kept.append(it)
        else:                                      # global declaration
            first = re.match(r"\s*(\w+)", it).group(1)
            if first in KNOWN_TYPES and "RWTexture2D" not in it:
                kept.append(it)
    return "\n\n".join(kept) + "\n"


def main() -> int:
    args = [a for a in sys.argv[1:] if a != "--keep"]
    if len(args) != 1:
        sys.stderr.write("usage: build_ref_hlsl.py <reference checkout> [--keep]\n")
        return 2
    REF = Path(args[0]) / "package" / "Shaders"
    if not REF.is_dir():
        sys.stderr.write("build_ref_hlsl: %s is not a directory\n" % REF)
        return 1
    OUT.mkdir(exist_ok=True)
    gs = (REF / "GaussianSplatting.hlsl").read_text()
    sh = (REF / "SphericalHarmonics.hlsl").read_text()
    cs = (REF / "SplatUtilities.compute").read_text()
    shader = (REF / "RenderGaussianSplats.shader").read_text()
    ps = shader[shader.index("CGPROGRAM") + len("CGPROGRAM"):shader.index("ENDCG")]
    (OUT / "ref_cs.inc").write_text("// GENERATED from the reference's GaussianSplatting.hlsl + SplatUtilities.compute + SphericalHarmonics.hlsl\n"
                                    "#define SHADER_STAGE_COMPUTE 1\n" + rewrite(gs) + "\n" + slice_compute(cs, sh))
    (OUT / "ref_ps.inc").write_text("// GENERATED from the reference's GaussianSplatting.hlsl + RenderGaussianSplats.shader\n"
                                    "#undef SHADER_STAGE_COMPUTE\n#undef GAUSSIAN_SPLATTING_HLSL\n" + rewrite(gs) + "\n" + rewrite(ps))
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-math-errno", "-fopenmp", "-fPIC", "-shared", "-w",
           "-I", str(HERE), "-I", str(OUT), "-o", str(OUT / "libref_hlsl.so"), str(HERE / "ref_hlsl_harness.cpp")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode == 0 and "--keep" not in sys.argv:
        # the rewritten reference text is a build intermediate: only the compiled library stays on disk
        (OUT / "ref_cs.inc").unlink()
        (OUT / "ref_ps.inc").unlink()
    if r.returncode != 0:
        sys.stderr.write(r.stdout[-6000:])
        return 1
    print("built", OUT / "libref_hlsl.so")
    return 0


if __name__ == "__main__":
    sys.exit(main())
