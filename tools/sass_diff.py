"""Compares the SASS of two builds of libphoenix_b200.so function by function.

    python tools/sass_diff.py <lib_a.so> <lib_b.so>

Prints every function that exists in only one library and every function whose instructions or encodings differ,
and exits non-zero if it printed anything.  A refactor of host code or of shared device helpers should print
nothing.

Before the comparison it normalises what changes without the code changing: the anonymous-namespace component of
mangled names (a length-prefixed _GLOBAL__N_ identifier whose hash and suffix depend on the translation unit) and
the /*addr*/ comments.
"""
import re
import subprocess
import sys

ANON = re.compile(r'(\d+)_GLOBAL__N_')
ADDR = re.compile(r'/\*[0-9a-f]{4,}\*/')


def normalise(text):
    out, pos = [], 0
    for m in ANON.finditer(text):
        if m.start() < pos:
            continue
        out.append(text[pos:m.start()])
        out.append('<anon>')
        pos = m.end(1) + int(m.group(1))          # the identifier after the length is group(1) characters long
    out.append(text[pos:])
    return ADDR.sub('', ''.join(out))


def functions(lib):
    """{name: instruction lines}; a name that occurs in several units gets '#k' appended from its second occurrence."""
    sass = subprocess.run(['cuobjdump', '-sass', lib], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in normalise(sass).splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            name, k = m.group(1), 1
            while name in funcs:
                name, k = f'{m.group(1)}#{k}', k + 1
            funcs[name] = []
        elif name is not None and '/* 0x' in line:          # an instruction, or the second half of its encoding
            funcs[name].append(' '.join(line.split()))
    return funcs


def main(argv):
    if len(argv) != 3:
        sys.exit(__doc__)
    a, b = functions(argv[1]), functions(argv[2])
    lines = [f'only in {argv[1]}: {n}' for n in sorted(a.keys() - b.keys())]
    lines += [f'only in {argv[2]}: {n}' for n in sorted(b.keys() - a.keys())]
    lines += [f'differs: {n}' for n in sorted(a.keys() & b.keys()) if a[n] != b[n]]
    for line in lines:
        print(line)
    return 1 if lines else 0


if __name__ == '__main__':
    sys.exit(main(sys.argv))
