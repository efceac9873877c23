"""Compare the SASS of the tc_fused_kernel and factor_finish_kernel instantiations that two builds of the library share.

    python tools/sass_diff.py OLD.so NEW.so

A template parameter added with a default changes the mangled name but not the code: an instantiation of NEW whose trailing
arguments are those defaults (tc_fused_kernel <..., AMODE = 0, KRAO = false>, factor_finish_kernel <..., KPLANES = true>) is
compared with the OLD instantiation that has the same leading arguments.  Prints, per kernel of OLD, whether the instruction
text is identical, and how many are identical once the numbers of the uniform registers are erased (ptxas numbers them in an
order that can change with the rest of the translation unit)."""
import re
import subprocess
import sys

CUDA = "/usr/local/cuda/bin"
KERNELS = ("tc_fused_kernel", "factor_finish_kernel")


def functions(lib):
    out = subprocess.run([f"{CUDA}/cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            name = m.group(1)
            res[name] = []
        elif name and re.search(r"/\*[0-9a-f]{4}\*/", line):
            res[name].append(re.sub(r"/\*[0-9a-f]{4}\*/|/\* 0x[0-9a-f]+ \*/", "", line).strip())
    names = list(res)
    demangled = subprocess.run([f"{CUDA}/cu++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return {d: res[n] for n, d in zip(names, demangled.splitlines()) if any(k in d for k in KERNELS)}


def main():
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    renamed = {}
    for d, body in new.items():
        d = re.sub(r"(tc_fused_kernel<[^>]*), \(int\)0, \(bool\)0>", r"\1>", d)
        d = re.sub(r"(factor_finish_kernel<[^>]*), \(bool\)1>", r"\1>", d)
        renamed.setdefault(d, body)
    erase = lambda body: [re.sub(r"\bUR\d+\b", "UR", l) for l in body]  # noqa: E731
    same = same_erased = 0
    for d, body in sorted(old.items()):
        nb = renamed.get(d)
        tag = "missing" if nb is None else "identical" if nb == body else "uniform registers only" if erase(nb) == erase(body) else "DIFFERENT"
        same += tag == "identical"
        same_erased += tag in ("identical", "uniform registers only")
        print(f"{tag:24s} {d.split('(CUtensorMap')[0].split('(const float')[0]}")
    print(f"{len(old)} kernels: {same} identical, {same_erased} identical up to the numbering of uniform registers")
    return 0 if same_erased == len(old) else 1


if __name__ == "__main__":
    sys.exit(main())
