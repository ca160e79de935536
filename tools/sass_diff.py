"""Per-kernel SASS comparison of two builds of libb200whisper.so: which kernels were added or removed, and which of the
kernels both contain differ in their instructions.  Two things differ between builds of the SAME source and are
normalised away: the anonymous-namespace hash in every kernel's mangled name, and register numbers -- ptxas does not
number registers deterministically (two compiles of an unchanged gemm_tc.cu swap UR6 / UR8 in the gemm_tc kernels), so
kernels are compared as instruction sequences (opcodes, modifiers, operand kinds, immediates) without register numbers.

Usage: python tools/sass_diff.py BEFORE.so AFTER.so > profiles/<name>.txt"""
import re
import subprocess
import sys


REG = re.compile(r"\b(U?R|U?P|B)\d+\b")


def canonical(lines):
    return [REG.sub(lambda m: m.group(1), x) for x in lines]


def kernels(lib):
    """normalised mangled name -> (original mangled name, instructions without register numbers or encodings)"""
    out, cur = {}, None
    for line in subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]+(_\d+)?", "ANON", m.group(1))
            out[cur] = (m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(.*?)\s*;", line)
        if cur and m:
            out[cur][1].append(m.group(1))
    return {k: (orig, canonical(lines)) for k, (orig, lines) in out.items()}


def main():
    before, after = kernels(sys.argv[1]), kernels(sys.argv[2])
    names = sorted(set(before) | set(after))
    orig = [(after.get(n) or before.get(n))[0] for n in names]
    dm = subprocess.run(["c++filt"], input="\n".join(orig), capture_output=True, text=True).stdout.splitlines()
    short = {n: re.sub(r"\(.*", "", d.replace("(anonymous namespace)::", "").replace("bw::", "").replace("void ", ""))
             for n, d in zip(names, dm)}
    rows = {"added": [], "removed": [], "changed": [], "identical": []}
    for n in sorted(names, key=lambda n: short[n]):
        if n not in before:
            rows["added"].append(f"{short[n]}  ({len(after[n][1])} instructions)")
        elif n not in after:
            rows["removed"].append(f"{short[n]}  ({len(before[n][1])} instructions)")
        elif before[n][1] != after[n][1]:
            b, a = before[n][1], after[n][1]
            diff = sum(x != y for x, y in zip(b, a)) + abs(len(b) - len(a))
            rows["changed"].append(f"{short[n]}  ({len(b)} -> {len(a)} instructions, {diff} differ)")
        else:
            rows["identical"].append(f"{short[n]}  ({len(after[n][1])} instructions)")
    print(f"# cuobjdump -sass {sys.argv[1]} -> {sys.argv[2]}: {len(names)} kernels (a kernel whose signature changed is listed as"
          " removed + added)")
    for k, v in rows.items():
        print(f"\n## {k}: {len(v)}")
        for r in v:
            print("  " + r)


if __name__ == "__main__":
    main()
