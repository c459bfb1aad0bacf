"""Per-kernel SASS comparison of two objects / shared libraries (cuobjdump, no GPU needed).

    python tools/sass_diff.py old.o new.o

Prints which kernels are instruction-identical, which differ and which exist on one side only.  Used to prove that
a source change leaves kernels byte-for-byte unchanged, so they need no re-validation on the GPU."""
import collections
import re
import subprocess
import sys


def kernels(path):
    out = subprocess.run(['cuobjdump', '-sass', path], capture_output=True, text=True, check=True).stdout
    d, name = collections.OrderedDict(), None
    for line in out.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            name = m.group(1)
            d[name] = []
        elif name is not None:
            d[name].append(re.sub(r'/\*[0-9a-f]{4}\*/', '', line).strip())     # drop instruction offsets
    return d


def norm(name):
    # a defaulted trailing template argument <.., 0> / <.., false>
    return name.replace('ELi0EEEvNS', 'EEEvNS').replace('ELb0EEEvNS', 'EEEvNS')


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    bn = {norm(k): v for k, v in b.items()}
    an = {norm(k) for k in a}
    same, diff = [], []
    for k, v in a.items():
        if norm(k) in bn:
            (same if v == bn[norm(k)] else diff).append(k)
    print(f'identical: {len(same)}   different: {len(diff)}')
    for k in diff:
        print('  DIFFERENT', k)
    for k in a:
        if norm(k) not in bn:
            print('  only in', sys.argv[1], k)
    for k in bn:
        if k not in an:
            print('  only in', sys.argv[2], k)
    return 1 if diff else 0


if __name__ == '__main__':
    sys.exit(main())
