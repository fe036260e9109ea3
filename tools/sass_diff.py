"""Per-kernel SASS comparison of two builds of the library, from `cuobjdump -sass` -- works without a GPU.
Prints the kernels only in A (-), only in B (+), kernels only in B whose instructions equal those of a kernel only in A
(= A -> B: the kernel renamed, e.g. by a changed template parameter) and common kernels whose instructions differ (!);
exit code 1 when a kernel is new or changed, 0 when every difference is a rename or a removal.  A kernel in an
anonymous namespace carries its translation unit's file name and a hash in its mangled name; that prefix is normalised,
so a kernel moved to another .cu file compares as the same kernel.
usage: python tools/sass_diff.py A.so B.so"""
import re
import subprocess
import sys

ANON = re.compile(r"\d+_GLOBAL__N__[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]{8}")


def kernels(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    d, name = {}, None
    for line in ANON.sub("ANON", out).splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            d[name] = []
        # instruction lines (/*addr*/ ... ; /* encoding */) and the encoding's second word (scheduling control bits)
        elif name and re.match(r"\s*/\*([0-9a-f]{4,}| 0x[0-9a-f]{16} )\*/", line):
            d[name].append(re.sub(r"\s+", " ", line.strip()))
    return {k: "\n".join(v) for k, v in d.items()}


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    only_a, only_b = sorted(set(a) - set(b)), sorted(set(b) - set(a))
    by_code = {}
    for k in only_a:
        by_code.setdefault(a[k], []).append(k)
    renamed = [(by_code[b[k]].pop(0), k) for k in only_b if by_code.get(b[k])]
    for k in sorted(set(only_a) - {old for old, _ in renamed}):
        print("-", k)
    for k in sorted(set(only_b) - {new for _, new in renamed}):
        print("+", k)
    for old, new in renamed:
        print("=", old, "->", new)
    diff = [k for k in sorted(set(a) & set(b)) if a[k] != b[k]]
    for k in diff:
        print("!", k)
    print(f"{len(a)} kernels in A, {len(b)} in B, {len(set(a) & set(b)) - len(diff)} identical, {len(renamed)} renamed, "
          f"{len(diff)} differ")
    sys.exit(1 if diff or len(only_b) > len(renamed) else 0)


if __name__ == "__main__":
    main()
