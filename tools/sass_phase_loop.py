"""Static instruction counts of the chunk loop of every k_dm_phase_tc instantiation, from the SASS of the built library.

    python tools/sass_phase_loop.py [libaogym.so] [--md]

The chunk loop is the innermost backward branch around the kernel's tcgen05.ld (LDTM): its body handles one
16-pixel chunk per epilogue warp.  For each instantiation <STREHL, NOBS, MODE, NP> (NP = 240 for every mode and detector
size; 128, 256 and 512 for the fused modes 1 and 2 with NOBS 2 and 5) this prints the loop's instruction
count, its XU (conversion / transcendental pipe) instructions, MUFU, F2I and F2F separately, its packed FP32x2
instructions (FFMA2, FADD2, FMUL2: one issue slot for two FP32 operations, counted under fma too), its bulk and tensor
copy issues (UBLKCP, UTMALDG), the instructions of the fill path (the innermost BSSY .. BSYNC region that holds those
copies: the prefetch issue, which a warp runs on every chunk in a per-warp ring and on every fourth chunk in a ring
shared by four warps), and the mix over the pipes below.  Counts are static (both sides of a branch count), CPU only: cuobjdump -sass of the sm_100a cubin."""
import argparse
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PIPES = [   # (pipe, opcode prefixes); first match wins
    ('xu', ('MUFU', 'F2I', 'I2F', 'F2F', 'FRND', 'POPC', 'FLO', 'BREV')),
    ('fp64', ('DADD', 'DFMA', 'DMUL', 'DSETP')),
    ('fma', ('FFMA', 'FADD', 'FMUL', 'IMAD', 'HFMA2', 'HADD2', 'HMUL2', 'FSWZADD')),
    ('tmem', ('LDTM', 'STTM', 'UTC')),
    ('lsu', ('LDS', 'STS', 'LDG', 'STG', 'LDL', 'STL', 'LD.', 'ST.', 'SHFL', 'ATOM', 'RED', 'LDSM')),
    ('uniform', ('U', 'R2UR', 'S2UR', 'LDCU')),   # UBLKCP (bulk copy) counts here, as a uniform-datapath instruction
    ('sync/branch', ('SYNCS', 'BAR', 'WARPSYNC', 'BRA', 'BSSY', 'BSYNC', 'EXIT', 'NOP', 'YIELD', 'NANOSLEEP', 'ELECT',
                     'VOTE', 'FENCE', 'MEMBAR', 'CCTL', 'CALL', 'RET', 'BPT', 'ACQBULK', 'WARPGROUP')),
    ('alu', ('LOP3', 'IADD3', 'IADD', 'VIADD', 'SHF', 'SHL', 'SHR', 'ISETP', 'FSETP', 'PRMT', 'SEL', 'FSEL', 'MOV',
             'IABS', 'IMNMX', 'VIMNMX', 'FMNMX', 'LEA', 'PLOP3', 'P2R', 'R2P', 'CS2R', 'S2R', 'LDC', 'IMNMX', 'FCHK')),
]
LINE = re.compile(r'/\*([0-9a-f]{4,})\*/\s+(@!?U?P[T0-9]+\s+)?([A-Z0-9_.]+)([^;]*);')
FUNC = re.compile(r'Function : (\S+)')
INST = re.compile(r'k_dm_phase_tcILb(\d)ELi(\d+)ELi(\d)ELi(\d+)E')


def pipe_of(op):
    for pipe, prefixes in PIPES:
        if op.startswith(prefixes):
            return pipe
    return 'other'


def functions(sass):
    name, body = None, []
    for line in sass.splitlines():
        m = FUNC.search(line)
        if m:
            if name:
                yield name, body
            name, body = m.group(1), []
            continue
        m = LINE.search(line)
        if m and name:
            body.append((int(m.group(1), 16), m.group(3), m.group(4)))
    if name:
        yield name, body


def chunk_loop(body):
    """instructions of the innermost backward branch whose range holds an LDTM"""
    ldtm = [a for a, op, _ in body if op.startswith('LDTM')]
    best = None
    for a, op, args in body:
        if not op.startswith('BRA'):
            continue
        m = re.search(r'(0x[0-9a-f]+)', args)
        if not m:
            continue
        tgt = int(m.group(1), 16)
        if tgt < a and any(tgt <= x < a for x in ldtm) and (best is None or a - tgt < best[1] - best[0]):
            best = (tgt, a)
    if best is None:
        return []
    return [(a, op) for a, op, _ in body if best[0] <= a <= best[1]]


COPIES = ('UBLKCP', 'UTMALDG')
PACKED = ('FFMA2', 'FADD2', 'FMUL2')


def fill_path(body, loop):
    """instructions of the innermost BSSY .. BSYNC region of the loop that holds all of its copy issues"""
    copies = [a for a, op in loop if op.startswith(COPIES)]
    if not copies:
        return 0
    lo, hi = loop[0][0], loop[-1][0]
    best = None
    for a, op, args in body:
        if not (lo <= a <= hi and op.startswith('BSSY')):
            continue
        m = re.search(r'(0x[0-9a-f]+)', args)
        end = int(m.group(1), 16) if m else -1
        if a < min(copies) and max(copies) < end and (best is None or end - a < best[1] - best[0]):
            best = (a, end)
    return sum(1 for a, _ in loop if best[0] <= a < best[1]) if best else 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('lib', nargs='?', default=os.path.join(ROOT, 'adaptive_optics_gym_b200', 'libaogym.so'))
    ap.add_argument('--md', action='store_true', help='markdown table')
    args = ap.parse_args()
    cuobjdump = os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'bin', 'cuobjdump')
    sass = subprocess.run([cuobjdump, '-sass', args.lib], check=True, capture_output=True, text=True).stdout
    rows = []
    for name, body in functions(sass):
        m = INST.search(name)
        if not m:
            continue
        loop = chunk_loop(body)
        ops = collections.Counter(op.split('.')[0] for _, op in loop)
        pipes = collections.Counter(pipe_of(op) for _, op in loop)
        key = tuple(int(g) for g in m.groups())
        copies = sum(1 for _, op in loop if op.startswith(COPIES))
        packed = sum(ops[o] for o in PACKED)
        rows.append((key, len(loop), pipes['xu'], ops['MUFU'], ops['F2I'], ops['F2F'], packed, copies, fill_path(body, loop), pipes))
    rows.sort()
    cols = ['fma', 'alu', 'xu', 'fp64', 'lsu', 'tmem', 'uniform', 'sync/branch', 'other']
    if args.md:
        print('| instantiation | loop instr | XU | MUFU | F2I | F2F | packed | copies | fill path | ' + ' | '.join(cols) + ' |')
        print('|---' * (9 + len(cols)) + '|')
    else:
        print('%-16s %6s %4s %4s %4s %4s %6s %6s %4s  ' % ('<S,NOBS,MODE,NP>', 'instr', 'XU', 'MUFU', 'F2I', 'F2F', 'packed', 'copies',
                                                             'fill') +
              ' '.join('%7s' % c[:7] for c in cols))
    for key, n, xu, mufu, f2i, f2f, packed, copies, fill, pipes in rows:
        k = '<%d,%d,%d,%d>' % key
        if args.md:
            print('| `%s` | %d | %d | %d | %d | %d | %d | %d | %d | ' % (k, n, xu, mufu, f2i, f2f, packed, copies, fill) +
                  ' | '.join(str(pipes[c]) for c in cols) + ' |')
        else:
            print('%-16s %6d %4d %4d %4d %4d %6d %6d %4d  ' % (k, n, xu, mufu, f2i, f2f, packed, copies, fill) +
                  ' '.join('%7d' % pipes[c] for c in cols))
    return 0 if rows else 1


if __name__ == '__main__':
    sys.exit(main())
