"""Compare two builds of libdrt_cuda.so kernel by kernel (no GPU needed):
    python tools/compare_builds.py OLD.so NEW.so [OLD_PTXAS.log NEW_PTXAS.log]
SASS: `cuobjdump -sass` of each library, split at every `Function :` header and compared by name instruction for instruction
(addresses and encodings dropped; the order of the functions does not matter).  With the two logs of a build made with
`make EXTRA="-Xptxas -v"`: the registers, stack, spill and shared-memory lines of every function.  Exits 1 on any difference."""
import re, subprocess, sys


def sass(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for ln in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            name = m.group(1)
            funcs.setdefault(name, [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", ln)
        if m and name:
            funcs[name].append(m.group(1))
    return funcs


def ptxas(path):
    props, name = {}, None
    for ln in open(path):
        m = re.search(r"Function properties for (\S+)", ln) or re.search(r"Compiling entry function '(\S+)'", ln)
        if m:
            name = re.sub(r"_INTERNAL_[0-9a-f]{8}_", "_INTERNAL_", m.group(1))   # a per-build hash of the translation unit
            continue
        if name and ("stack frame" in ln or "Used " in ln):
            props.setdefault(name, []).append(ln.split("ptxas info    :")[-1].strip())
    return props


def compare(what, old, new):
    same = sum(1 for k in old if k in new and old[k] == new[k])
    print(f"{what}: {len(old)} functions in the old build, {len(new)} in the new one, {same} identical")
    diff = sorted(k for k in set(old) | set(new) if old.get(k) != new.get(k))
    for k in diff:
        print(f"  differs: {k}" + ("" if k in old and k in new else "  (only in the " + ("new" if k in new else "old") + " build)"))
    return not diff


def main():
    a, b = sass(sys.argv[1]), sass(sys.argv[2])
    ok = compare("SASS", a, b)
    print(f"  of them {sum('13render_kernelI' in k for k in b)} render_kernel, {sum('22render_kernel_adaptiveI' in k for k in b)} render_kernel_adaptive")
    print("  instructions:", sum(len(v) for v in a.values()), "old,", sum(len(v) for v in b.values()), "new")
    if len(sys.argv) > 4:
        ok = compare("ptxas -v", ptxas(sys.argv[3]), ptxas(sys.argv[4])) and ok
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
