"""Static instruction count and opcode mix of the symbol loop of one kernel.

usage: python tools/sass_loop_count.py LIB_OR_CUBIN KERNEL [--all] [--alu]

KERNEL is matched against the demangled names printed by cu++filt, e.g. 'k_demod<false, 1, 1>'; it must
match exactly one kernel.  A loop is a backward branch whose range holds no EXIT or RET (a branch back from
an out-of-line block placed after the kernel's exits is not a loop).  The reported loop is the largest one,
for k_demod the loop over OFDM symbols; --all lists every loop.  --alu adds the loop's count of alu-pipe instructions
(ALU_OPS).  Needs cuobjdump and cu++filt from the CUDA toolkit.
"""
import collections
import re
import subprocess
import sys

# Opcodes that issue to the integer alu pipe, for the opcodes k_viterbi's loops contain.  Calibrated against ncu's
# smsp__inst_executed_pipe_alu on a B200 (profiles/r02_viterbi_pipe_counts.json, r02_ncu_full_viterbi_quad.json):
# with this set, round 2's k_viterbi chunk loop has 508 alu instructions, 508 x 1539 chunks / 32 frames per warp =
# 24432 per frame against the measured 24430.5 -- a fit to that one number, which several opcode sets reach.  Among
# them this is the one that also matches a second kernel: of k_viterbi_quad's loop (unchanged since round 2) 330 of
# 572 instructions are in the set, 57.7 %, or 59.2 % of the 557 that are not uniform-datapath (U*, S2UR), against
# ncu's 59.2 % (alu at
# 56.36 % of its half rate, 1.904 warp-instructions per SM cycle).  A static count ignores the loops' branches, so
# the match is a cross-check, not a measurement.  VIADD, VIMNMX and IMAD are not alu here.
ALU_OPS = {"VIADDMNMX", "PRMT", "LOP3", "ISETP", "SHF", "IADD3", "SEL", "BREV", "VIMNMX3"}

INS = re.compile(r'^\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;')


def functions(path):
    out = subprocess.run(["cuobjdump", "-sass", path], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            name = m.group(1)
            funcs[name] = []
            continue
        m = INS.match(line)
        if m and name:
            body = re.sub(r'^@!?U?P[T0-9]\s+', '', m.group(2).strip())
            funcs[name].append((int(m.group(1), 16), body.split()[0], body))
    return funcs


def demangle(names):
    out = subprocess.run(["cu++filt"], input="\n".join(names), check=True, capture_output=True, text=True).stdout
    return dict(zip(names, out.splitlines()))


def loops(ins):
    found = []
    for addr, op, body in ins:
        if not op.startswith('BRA'):
            continue
        m = re.search(r'0x([0-9a-f]+)', body)
        if not m or int(m.group(1), 16) >= addr:
            continue
        lo = int(m.group(1), 16)
        rng = [x for x in ins if lo <= x[0] <= addr]
        if any(x[1].startswith(('EXIT', 'RET')) for x in rng):
            continue
        found.append((lo, addr, rng))
    return found


def main():
    if len(sys.argv) < 3:
        sys.exit(__doc__)
    path, want = sys.argv[1], sys.argv[2]
    funcs = functions(path)
    names = demangle(list(funcs))
    # cu++filt prints template arguments as (bool)0, (int)1
    norm = lambda s: re.sub(r'\s', '', s).replace('false', '0').replace('true', '1')
    bare = lambda v: re.sub(r'^void\s+', '', re.sub(r'\((bool|int)\)', '', v).split('(')[0])
    hit = [k for k, v in names.items() if k == want or norm(bare(v)) == norm(want)]
    if len(hit) != 1:
        sys.exit("%d kernels match %r: %s" % (len(hit), want, [names[k] for k in hit]))
    found = loops(funcs[hit[0]])
    if not found:
        sys.exit("no loop in " + names[hit[0]])
    print("kernel %s: %d instructions" % (names[hit[0]], len(funcs[hit[0]])))
    pick = max(found, key=lambda l: len(l[2]))
    for lo, hi, rng in (found if "--all" in sys.argv else [pick]):
        mix = collections.Counter(x[1].split('.')[0] for x in rng)
        print("loop 0x%x..0x%x: %d instructions%s" % (lo, hi, len(rng), "  (symbol loop)" if rng is pick[2] else ""))
        print("  " + "  ".join("%s %d" % kv for kv in mix.most_common()))
        if "--alu" in sys.argv:
            print("  alu %d" % sum(n for op, n in mix.items() if op in ALU_OPS))


if __name__ == "__main__":
    main()
