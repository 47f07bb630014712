#!/usr/bin/env python3
"""Normalised SASS comparison of the kernels of two builds of libh263cu.so.

    python tools/sass_compare.py OLD.so NEW.so [-v]

Dumps both with `cuobjdump -sass`, keeps each kernel's instruction text (addresses and encodings dropped) and
compares the kernels by demangled name, parameter lists ignored.  Kernel templates that gained an output-mode
parameter are matched to the old names: recon_tile_kernel<..., false / true> (the former device-RGBA flag) is
recon_tile_kernel<..., 0 / 1>, and recon_mb_kernel, deblock_rgba_kernel and deblock_rgba_tile_kernel are their
<false> (RGBA) instantiations, and resample_rgb_kernel<dtype> is resample_rgb_kernel<dtype, false> (the stretch form).
Prints SAME / DIFF per kernel of the old build and exits non-zero on any difference.
"""
import difflib
import re
import subprocess
import sys

INS = re.compile(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;")


def kernels(path):
    txt = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    out = {}
    for part in re.split(r"\n\s*Function : ", txt)[1:]:
        name, body = part.split("\n", 1)
        out[name.strip()] = [re.sub(r"\s+", " ", m.group(1)) for m in map(INS.match, body.splitlines()) if m]
    return out


def demangle(names):
    r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return dict(zip(names, r))


def key(demangled, old):
    k = demangled.split("(")[0].replace("void ", "")
    if old and not k.startswith("h263dev::resample_rgb_kernel<"):  # its bool (the fit flag) stays a bool
        k = re.sub(r", false>$", ", 0>", k)
        k = re.sub(r", true>$", ", 1>", k)
    if old:
        if k in ("h263dev::recon_mb_kernel", "h263dev::deblock_rgba_kernel", "h263dev::deblock_rgba_tile_kernel"):
            k += "<false>"
        k = re.sub(r"^(h263dev::resample_rgb_kernel<\d+u)>$", r"\1, false>", k)
    return k


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    dold, dnew = demangle(list(old)), demangle(list(new))
    ok = {key(dold[k], True): v for k, v in old.items()}
    nk = {key(dnew[k], False): v for k, v in new.items()}
    bad = 0
    for k in sorted(ok):
        if k not in nk:
            print("MISSING", k)
            bad += 1
            continue
        same = ok[k] == nk[k]
        bad += not same
        print("SAME" if same else "DIFF", len(ok[k]), len(nk[k]), k)
        if not same and "-v" in sys.argv:
            print("\n".join(list(difflib.unified_diff(ok[k], nk[k], lineterm=""))[:60]))
    print("only in the new build:", sorted(k for k in nk if k not in ok))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
