#!/usr/bin/env python
"""Compare the SASS of the kernels two builds of libcrowdsim_b200.so have in common.

  python scripts/sass_compare.py OLD.so NEW.so

Kernels are matched by their demangled names after dropping the policy template argument of the newer build (`LIN = 0` of
step_kernel / step_flat_kernel, `HLIN = false` of lookahead_kernel / lookahead_humans_kernel), so that the ORCA-human
instantiations of a build with the linear policy are compared with the kernels of a build without it. For each matched
kernel the instruction lines of `cuobjdump -sass` (addresses removed, encodings kept) must be identical. Prints one line per
kernel and exits non-zero on any difference or on a kernel of OLD that NEW lacks. Needs only cuobjdump and c++filt (no GPU).
"""
import re
import subprocess
import sys


def demangle(name):
    return subprocess.run(['c++filt', name], capture_output=True, text=True, check=True).stdout.strip()


def key(name):
    d = demangle(name)
    d = re.sub(r', 0>', '>', d) if re.search(r'step(_flat)?_kernel<', d) else d
    d = re.sub(r'(lookahead(_humans)?_kernel)<false>', r'\1', d)
    return re.sub(r'^void ', '', d)


def functions(so):
    out = subprocess.run(['cuobjdump', '-sass', so], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            cur = funcs.setdefault(key(m.group(1)), [])
            continue
        m = re.match(r'\s*/\*[0-9a-f]{4,}\*/\s*(.*)$', line)
        if cur is not None and m:
            cur.append(m.group(1).strip())
        elif cur is not None and re.match(r'\s*/\* 0x[0-9a-f]+ \*/\s*$', line):
            cur.append(line.strip())              # second half of an instruction's encoding
    return funcs


def main(old, new):
    a, b = functions(old), functions(new)
    bad = 0
    for name in sorted(a):
        if name not in b:
            print('MISSING  ', name); bad += 1
        elif a[name] != b[name]:
            n = sum(1 for x, y in zip(a[name], b[name]) if x != y) + abs(len(a[name]) - len(b[name]))
            print('DIFFERS  ', name, '(%d of %d lines)' % (n, len(a[name]))); bad += 1
        else:
            print('identical', name, '(%d lines)' % len(a[name]))
    print('%d kernels compared, %d differ or are missing; %d kernels only in %s' % (len(a), bad, len(set(b) - set(a)), new))
    return 1 if bad else 0


if __name__ == '__main__':
    sys.exit(main(*sys.argv[1:3]))
