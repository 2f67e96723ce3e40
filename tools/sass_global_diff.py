"""Compare the SASS of two builds of one object file kernel by kernel: instruction counts, whether the opcode sequence
is identical, and whether the global-memory instructions (loads, stores, reductions, TMA, L2 prefetch) form the same
sequence once register numbers and immediates are ignored -- the evidence that a kernel change cannot have changed its
DRAM traffic.  Usage: cuobjdump -sass old.o > old.sass; cuobjdump -sass new.o > new.sass;
python tools/sass_global_diff.py old.sass new.sass"""
import collections
import re
import subprocess
import sys

GLOBAL = re.compile(r'^(LDG|STG|REDG|ATOMG|LD|ST|UTMALDG|UTMASTG|UTMAREDG|UTMAPF|UBLKPF|UBLKCP|CCTL|UTMACCTL)(\.|$)')


def parse(path):
    funcs, cur = {}, None
    for line in open(path):
        m = re.match(r'\s+Function : (\S+)', line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = re.match(r'\s+/\*[0-9a-f]{4,}\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)\s*(.*?);', line)
        if m and cur:
            funcs[cur].append((m.group(2), m.group(3)))
    return funcs


def norm(operands):
    return re.sub(r'\bU?R\d+\b|\bU?P\d+\b|0x[0-9a-f]+', '#', operands)


def demangle(name):
    return subprocess.run(['c++filt', name], stdout=subprocess.PIPE, text=True).stdout.strip()


def main(old_path, new_path):
    old, new = parse(old_path), parse(new_path)
    for f in sorted(set(old) | set(new), key=demangle):
        a, b = old.get(f, []), new.get(f, [])
        ga = [(o, norm(x)) for o, x in a if GLOBAL.match(o)]
        gb = [(o, norm(x)) for o, x in b if GLOBAL.match(o)]
        same = [o for o, _ in a] == [o for o, _ in b]
        print(f"{demangle(f)}: {len(a)} -> {len(b)} instructions; opcode sequence {'identical' if same else 'differs'}; "
              f"global-memory instructions {len(ga)} -> {len(gb)}, "
              + ("the same sequence (registers and immediates aside)" if ga == gb else "DIFFERENT"))
        if not same:
            ca, cb = collections.Counter(o for o, _ in a), collections.Counter(o for o, _ in b)
            d = {o: cb[o] - ca[o] for o in set(ca) | set(cb) if cb[o] != ca[o]}
            print("    opcode count changes:", ", ".join(f"{o} {v:+d}" for o, v in sorted(d.items())))


if __name__ == "__main__":
    main(*sys.argv[1:3])
