#!/usr/bin/env python
"""Per-region, per-pipe instruction counts of the env-step kernel's grid-stride loop (no GPU needed).

The step kernel is bound by the integer ALU pipe (LOP3 / SHF / IADD3 / ISETP ... at 16 lanes per clock per scheduler),
not by HBM, so the count of ALU-pipe instructions per board is the number to drive down; IMAD runs on the FMA pipe,
which the step body leaves mostly idle.  The loop is split into:
  main   instructions before the loop's first global store, outside the reset block
  reset  the largest BSSY..BSYNC block between the loop head and its first global store (the auto-reset branch;
         a divergent block: a warp pays all of it when any lane takes it)
  tail   from the first global store to the loop's back edge (stores + the Philox block of the next board)

usage: python profiles/sass_pipes.py [libb2048.so | .cubin] [kernel ...]
       (default: the library next to this repo and step_fast_kernel<RANDOM_LEGAL, track, plain>)
       -v  also print the mnemonics of each region"""
import collections, os, re, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_LIB = os.path.join(ROOT, "rl-2048-with-reinforce-and-actor-critic_b200", "libb2048.so")
DEFAULT_KERNELS = ["_ZN2b216step_fast_kernelILi3ELb1ELb1EEEvNS_8StepArgsE"]

ALU = {"LOP3", "LOP", "SHF", "SHL", "SHR", "SEL", "FSEL", "ISETP", "FSETP", "IADD3", "IADD", "VIADD", "VIADDMNMX", "LEA",
       "PRMT", "POPC", "FLO", "BREV", "IMNMX", "VIMNMX", "IABS", "BMSK", "SGXT", "PLOP3", "P2R", "R2P", "MOV", "ICMP",
       "ISCADD", "CS2R"}
FMA = {"IMAD", "FFMA", "FMUL", "FADD", "HFMA2", "HADD2", "HMUL2", "IDP", "IMUL"}
FP64 = {"DADD", "DMUL", "DFMA", "DSETP", "F2F", "F2I", "I2F", "I2FP", "F2FP"}
MEM = {"LDS", "LDG", "STG", "STS", "LD", "ST", "ATOM", "ATOMS", "RED", "REDG", "LDC", "LDL", "STL"}
PIPES = ["alu", "fma", "fp64/conv", "mem", "ctrl", "uniform", "other"]

LINE = re.compile(r"\s*/\*([0-9a-f]{4,})\*/\s+(@!?U?P[T0-9]+\s+)?([A-Z0-9_]+)((?:\.[A-Z0-9_]+)*)\s*([^;]*);")


def pipe(op):
    if op in ALU:
        return "alu"
    if op in FMA:
        return "fma"
    if op in FP64:
        return "fp64/conv"
    if op in MEM:
        return "mem"
    if op in {"BRA", "BSSY", "BSYNC", "EXIT", "NOP", "WARPSYNC", "YIELD", "BAR", "PREEXIT", "CALL", "RET", "BPT"}:
        return "ctrl"
    if op.startswith("U") or op in {"S2UR", "R2UR", "S2R", "CS2R"}:
        return "uniform"
    return "other"


def sass_of(path, kernel):
    out = subprocess.run(["cuobjdump", "-sass", "-fun", kernel, path], capture_output=True, text=True)
    if out.returncode != 0 or "Function" not in out.stdout:
        sys.exit(f"cuobjdump found no function {kernel} in {path}:\n{out.stderr}")
    ins = []
    for line in out.stdout.splitlines():
        m = LINE.match(line)
        if m:
            ins.append((int(m.group(1), 16), m.group(3), m.group(3) + m.group(4), m.group(5), bool(m.group(2))))
    return ins   # (address, mnemonic, mnemonic with modifiers, operands, predicated)


def regions(ins):
    idx = {a[0]: k for k, a in enumerate(ins)}
    # grid-stride loop: the conditional backward branch with the longest span (an unconditional one jumps back from an
    # out-of-line slow path, such as the retry of a barrier wait)
    best = None
    for a, op, full, arg, pred in ins:
        if op == "BRA" and pred:
            m = re.search(r"0x([0-9a-f]+)", arg)
            tgt = int(m.group(1), 16) if m else None
            if tgt is not None and tgt < a and tgt in idx and (best is None or a - tgt > best[1] - best[0]):
                best = (tgt, a)
    if best is None:
        sys.exit("no loop found")
    lo, hi = idx[best[0]], idx[best[1]]
    first_st = next((k for k in range(lo, hi + 1) if ins[k][1] in ("STG", "ST")), hi + 1)
    # BSSY blocks opened between the loop head and the first store; the largest is the reset branch
    blocks = []
    for k in range(lo, first_st):
        a, op, full, arg, pred = ins[k]
        if op == "BSSY":
            m = re.search(r"(B\d+),\s*0x([0-9a-f]+)", arg)
            end = int(m.group(2), 16)
            if end in idx and idx[end] <= first_st:
                blocks.append((k, idx[end]))
    reset = max(blocks, key=lambda b: b[1] - b[0], default=None)
    in_reset = set(range(reset[0], reset[1] + 1)) if reset else set()
    return {"main": [ins[k] for k in range(lo, first_st) if k not in in_reset],
            "reset": [ins[k] for k in sorted(in_reset)],
            "tail": [ins[k] for k in range(first_st, hi + 1)]}


def main():
    args = [a for a in sys.argv[1:] if a != "-v"]
    verbose = "-v" in sys.argv[1:]
    path = args[0] if args else DEFAULT_LIB
    kernels = args[1:] or DEFAULT_KERNELS
    for kern in kernels:
        regs = regions(sass_of(path, kern))
        print(f"{kern}")
        print(f"{'region':8s} {'instrs':>6s} " + " ".join(f"{p:>9s}" for p in PIPES))
        tot = collections.Counter()
        for name, body in regs.items():
            c = collections.Counter(pipe(x[1]) for x in body)
            tot.update(c)
            print(f"{name:8s} {len(body):6d} " + " ".join(f"{c[p]:9d}" for p in PIPES))
        print(f"{'loop':8s} {sum(tot.values()):6d} " + " ".join(f"{tot[p]:9d}" for p in PIPES))
        if verbose:
            for name, body in regs.items():
                c = collections.Counter(x[2] for x in body)
                print(f"  {name}: " + ", ".join(f"{k} {v}" for k, v in c.most_common()))


if __name__ == "__main__":
    main()
