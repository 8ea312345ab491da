"""Compare the device code of two builds of libkissmcmc_cuda.so kernel by kernel.

    python kissmcmc.jl_b200/build.py a.so; (change the sources); python kissmcmc.jl_b200/build.py b.so
    python profiles/sass_diff.py a.so b.so

Each kernel is keyed by its mangled name with the per-build anonymous-namespace hash removed; its SASS is compared as
instruction text (addresses and encodings dropped), and its `cuobjdump -res-usage` line (registers, shared memory, stack)
as is.  Prints one summary line and the names of the kernels that differ; exits 1 if any does.
"""
import re
import subprocess
import sys

ANON = re.compile(r"_GLOBAL__N__[0-9a-f_]+")


def _run(*args):
    return subprocess.run(["cuobjdump", *args], check=True, capture_output=True, text=True).stdout


def sass(lib):
    out, name = {}, None
    for line in _run("-sass", lib).splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = ANON.sub("_GLOBAL__N__", m.group(1))
            out[name] = []
        elif name and "/*" in line:
            text = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)
            text = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", text).strip()
            if text:
                out[name].append(text)
    return out


def res_usage(lib):
    out, name = {}, None
    for line in _run("-res-usage", lib).splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = ANON.sub("_GLOBAL__N__", m.group(1))
        elif name and "REG:" in line:
            out[name] = line.strip()
            name = None
    return out


def main(a, b):
    sa, sb, ra, rb = sass(a), sass(b), res_usage(a), res_usage(b)
    names = sorted(set(sa) | set(sb))
    diff = [n for n in names if sa.get(n) != sb.get(n) or ra.get(n) != rb.get(n)]
    print(f"{len(names)} kernels ({len(sa)} / {len(sb)}), {len(names) - len(diff)} identical SASS and resource usage, "
          f"{len(diff)} differ")
    for n in diff:
        print("  differs:", n)
    return 1 if diff else 0


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:3]))
