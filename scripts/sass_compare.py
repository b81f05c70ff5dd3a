"""Per-kernel SASS comparison of two builds of the same object: python scripts/sass_compare.py OLD.o NEW.o

Prints, for every kernel, whether its SASS (cuobjdump -sass, instruction addresses stripped) is the same in both objects,
differs, or exists in one only.  The hash that nvcc puts in the names of anonymous-namespace kernels depends on the
source path, so it is normalised away before names are matched.
"""
import re
import subprocess
import sys


def kernels(obj):
    out = subprocess.run(["cuobjdump", "-sass", obj], check=True, capture_output=True, text=True).stdout
    d, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1))
            d[cur] = []
        elif cur:
            d[cur].append(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip())
    return d


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    for k in sorted(set(old) | set(new)):
        status = "new only" if k not in old else "old only" if k not in new else "same" if old[k] == new[k] else "DIFFERENT"
        print(f"{status:10s} {k}")


if __name__ == "__main__":
    main()
