"""Opcode mix of the loops of one kernel, read from `cuobjdump -sass`.

    python tools/sass_loop_mix.py OBJ_OR_CUBIN KERNEL_SUBSTRING [--min-len N] [--per K] [--json]

Every backward branch (a BRA whose target lies at or before it) closes a loop; its body is the instruction range
[target, branch].  For each loop the script prints the instruction count, the FP64 instructions (DFMA, DMUL, DADD, ...)
and the rest by opcode.  --per K divides the counts by K (e.g. the nodes covered by one trip of the node loop).
A fully unrolled loop has no backward branch: --range START END (hex addresses) counts that span instead, and --vote
counts the code a warp vote (VOTE.ALL) branches around, i.e. the straight-line path taken when the vote passes (the tile
kernel's clamp-free node loop).
Nested loops are listed separately; an outer loop's count includes its inner loops' bodies once.
The kernel is the first function whose (mangled) name contains KERNEL_SUBSTRING.
"""
import argparse
import collections
import json
import os
import re
import subprocess
import sys

FP64 = {'DFMA', 'DMUL', 'DADD', 'DSETP', 'DMNMX', 'DSET'}
CUOBJDUMP = os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'bin', 'cuobjdump')

_FUNC = re.compile(r'^\s*Function\s*:\s*(\S+)')
_INSN = re.compile(r'^\s*/\*([0-9a-f]{4,})\*/\s*(@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_]*)((?:\.[A-Z0-9_]+)*)\s*([^;]*);')
_TARGET = re.compile(r'0x([0-9a-f]+)')


def kernels(path):
    exe = CUOBJDUMP if os.path.exists(CUOBJDUMP) else 'cuobjdump'
    text = subprocess.run([exe, '-sass', path], capture_output=True, text=True, check=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        mf = _FUNC.match(line)
        if mf:
            name = mf.group(1)
            out[name] = []
            continue
        mi = _INSN.match(line)
        if mi and name is not None:
            out[name].append((int(mi.group(1), 16), mi.group(3), mi.group(4), mi.group(5)))
    return out


def loops(insns):
    res = []
    for k, (addr, op, _mods, args) in enumerate(insns):
        if op != 'BRA':
            continue
        mt = _TARGET.search(args)
        if not mt:
            continue
        tgt = int(mt.group(1), 16)
        if tgt > addr:
            continue
        body = [x for x in insns if tgt <= x[0] <= addr]
        res.append((tgt, addr, body))
    return res


def mix(body):
    ops = collections.Counter(op + ('.64' if op in ('LDCU', 'LDC', 'LDS', 'LDG') and '.64' in mods else '')
                              for _a, op, mods, _args in body)
    fp64 = sum(n for op, n in ops.items() if op in FP64)
    return {'instructions': len(body), 'fp64': fp64, 'other': len(body) - fp64, 'opcodes': dict(ops.most_common())}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('obj')
    ap.add_argument('kernel')
    ap.add_argument('--min-len', type=int, default=20, help='skip loops with fewer instructions')
    ap.add_argument('--per', type=float, default=1.0, help='divide the FP64 / other counts by this')
    ap.add_argument('--range', nargs=2, metavar=('START', 'END'), help='count this address span (hex) instead')
    ap.add_argument('--vote', action='store_true', help='count the span each VOTE.ALL branches around instead')
    ap.add_argument('--json', action='store_true')
    args = ap.parse_args()
    ks = kernels(args.obj)
    names = [n for n in ks if args.kernel in n]
    if not names:
        sys.exit('no kernel matching %r in %s' % (args.kernel, args.obj))
    name = names[0]
    rows = []
    spans = loops(ks[name])
    if args.vote:
        spans = []
        insns = ks[name]
        for k, (addr, op, _mods, _args) in enumerate(insns):
            if op != 'VOTE' or k + 1 >= len(insns) or insns[k + 1][1] != 'BRA':
                continue
            mt = _TARGET.search(insns[k + 1][3])
            lo, hi = insns[k + 1][0] + 16, int(mt.group(1), 16)
            spans.append((lo, hi, [x for x in insns if lo <= x[0] < hi]))
    if args.range:
        lo, hi = (int(v, 16) for v in args.range)
        spans = [(lo, hi, [x for x in ks[name] if lo <= x[0] < hi])]
    for tgt, end, body in spans:
        if len(body) < args.min_len:
            continue
        m = mix(body)
        m.update({'start': '0x%04x' % tgt, 'end': '0x%04x' % end,
                  'fp64_per': round(m['fp64'] / args.per, 2), 'other_per': round(m['other'] / args.per, 2)})
        rows.append(m)
    if args.json:
        print(json.dumps({'kernel': name, 'per': args.per, 'loops': rows}))
        return
    print(name)
    for m in rows:
        print('loop %s-%s: %d instructions, %d FP64, %d other  (per %g: %.2f FP64, %.2f other)' % (
            m['start'], m['end'], m['instructions'], m['fp64'], m['other'], args.per, m['fp64_per'], m['other_per']))
        print('    ' + ' '.join('%s:%d' % kv for kv in m['opcodes'].items()))


if __name__ == '__main__':
    main()
