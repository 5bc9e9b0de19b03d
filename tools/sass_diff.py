"""Kernel-by-kernel SASS comparison of two builds of libb200tts.so (no GPU needed).

    python tools/sass_diff.py OLD.so NEW.so [--map 'REGEX=>REPLACEMENT' ...]

`cuobjdump -sass` of both libraries is split per function; instruction addresses and encodings are stripped, so two
functions compare equal when they are the same instruction stream.  --map rewrites NEW's mangled names before they are
matched against OLD's (e.g. a kernel that gained a template parameter).  Prints one line per kernel of OLD: `same`,
`DIFFERENT (n of m lines)` or `missing`, then the kernels only NEW has; exits 1 when a kernel of OLD is missing or differs,
unless it is listed with --allow.
"""
from __future__ import annotations

import argparse
import re
import subprocess
import sys

FUNC = re.compile(r'^\s*Function : (\S+)')
ADDR = re.compile(r'/\*[0-9a-f]{4,}\*/')
ENC = re.compile(r'/\* 0x[0-9a-f]+ \*/')


def sass_by_function(lib: str) -> dict:
    out = subprocess.run(['cuobjdump', '-sass', lib], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = FUNC.match(line)
        if m:
            name = m.group(1)
            funcs[name] = []
            continue
        if name is None:
            continue
        s = ENC.sub('', ADDR.sub('', line)).strip()
        if s and not s.startswith('.'):
            funcs[name].append(re.sub(r'\s+', ' ', s))
    return funcs


def main(argv=None) -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument('old')
    ap.add_argument('new')
    ap.add_argument('--map', action='append', default=[], help="REGEX=>REPLACEMENT applied to NEW's function names")
    ap.add_argument('--allow', action='append', default=[], help='substring of an OLD function allowed to differ')
    a = ap.parse_args(argv)
    old, new_raw = sass_by_function(a.old), sass_by_function(a.new)
    new = {}
    for n, body in new_raw.items():
        for rule in a.map:
            pat, rep = rule.split('=>', 1)
            n = re.sub(pat, rep, n)
        new[n] = body
    bad = 0
    for n in sorted(old):
        if n not in new:
            status = 'missing'
        elif old[n] == new[n]:
            status = 'same'
        else:
            diff = sum(1 for x, y in zip(old[n], new[n]) if x != y) + abs(len(old[n]) - len(new[n]))
            status = f'DIFFERENT ({diff} of {len(old[n])} lines)'
        allowed = any(s in n for s in a.allow)
        if status != 'same' and not allowed:
            bad += 1
        print(f'{status:<28} {n}' + ('   (allowed)' if allowed and status != 'same' else ''))
    for n in sorted(set(new) - set(old)):
        print(f'{"new":<28} {n}')
    print(f'{len(old)} kernels compared, {bad} unexpected difference(s)')
    return 1 if bad else 0


if __name__ == '__main__':
    sys.exit(main())
