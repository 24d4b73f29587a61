"""Static rehearsal of the 1-lane hot loop: python scripts/chain_path.py [lib.so] [kernel-name-substring] [--path]

Reads `cuobjdump -sass` of the library (default: the in-tree libecdna_b200.so), takes the kernel (default: the C2
build, ssa_kernel<1, false, false, 2, 5, SPEC 1, UNR 1>), finds its hot loop - the straight-line step, the one
backward branch whose body holds no other branch - and prints
  * the loop's instructions per pipe (ALU / FMA-heavy / FP32 / LSU / other), and
  * the longest register-dependency path through one iteration, with the latencies of LATENCY below.

Assumptions (a model, not a measurement):
  * every opcode has the fixed latency of LATENCY (cycles from issue to a dependent issue); LDS stands for the
    shared-memory round trip, MUFU and POPC for their variable-latency units;
  * shared-memory instructions leave the LSU in program order, so an LDS or ATOMS starts no earlier than the one
    before it (this ties the next event's loads to the current event's red.shared.add - a dependency through
    memory, not through registers);
  * a predicated instruction depends on its guard; a register written by it depends on the guard and sources.
The path is followed through consecutive iterations (the registers a loop carries into the next one), and the
figure reported is the growth of the critical path per iteration in steady state: the loop-carried recurrence
that bounds a warp alone on its scheduler.  A second figure adds in-order issue: one instruction per cycle, and
ISSUE_CYCLES between two instructions of the same pipe.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_LIB = os.path.join(ROOT, "ecdna-evo_b200", "libecdna_b200.so")
DEFAULT_KERNEL = "_ZN5ecdna10ssa_kernelILi1ELb0ELb0ELi2ELi5ELi1ELi1EEE"

PIPES = {
    "ALU": {"LOP3", "ISETP", "SEL", "IADD3", "FSETP", "VIADD", "SHF", "PLOP3", "VIMNMX", "IMNMX", "BMSK", "FSEL",
            "LEA", "POPC", "FLO", "BREV", "PRMT", "SHL", "SHR", "IABS", "P2R", "R2P", "FMNMX", "LOP", "IADD", "MOV",
            "ISCADD", "SGXT", "ICMP", "FCHK"},
    "FMA-heavy": {"IMAD", "IMUL", "IMADSP", "IDP", "IMNMX3"},
    "FP32": {"FFMA", "FMUL", "FADD", "FMNMX3", "FADD2", "FFMA2", "FMUL2"},
    "LSU": {"LDS", "STS", "ATOMS", "LD", "ST", "LDG", "STG", "ATOM", "ATOMG", "RED", "LDL", "STL", "LDC", "LDSM"},
}
# cycles from issue to a dependent issue (assumed, see above)
LATENCY = {"ALU": 4, "FMA-heavy": 4, "FP32": 4, "IMAD.WIDE": 6, "IMAD.HI": 6, "POPC": 6, "MUFU": 18, "I2FP": 6,
           "F2I": 6, "I2F": 6, "F2F": 6, "LDS": 30, "LDC": 30, "ATOMS": 30, "VOTE": 4, "S2R": 20, "S2UR": 20,
           "CS2R": 4, "R2UR": 8}
DEFAULT_LAT = 4
# cycles a warp instruction occupies its pipe (16-lane ALU and FMA-heavy pipes: two cycles per warp instruction)
ISSUE_CYCLES = {"ALU": 2, "FMA-heavy": 2}
REG = re.compile(r"\b(U?R\d+|U?P\d+)\b")


def pipe(op):
    base = op.split(".")[0]
    for p, ops in PIPES.items():
        if base in ops:
            return p
    return "other"


def latency(op):
    base = op.split(".")[0]
    for key in (".".join(op.split(".")[:2]), base):
        if key in LATENCY:
            return LATENCY[key]
    return LATENCY.get(pipe(op), DEFAULT_LAT)


def width(op):
    """registers a destination register name stands for"""
    if ".128" in op:
        return 4
    if ".64" in op or ".WIDE" in op:
        return 2
    return 1


def parse(text):
    """(op, dests, srcs) of one SASS instruction; a guard predicate counts as a source"""
    guard = None
    if text.startswith("@"):
        guard, text = text.split(None, 1)
        guard = guard.lstrip("@!")
    parts = text.split(None, 1)
    op = parts[0]
    ops = [o.strip() for o in parts[1].split(",")] if len(parts) > 1 else []
    base = op.split(".")[0]
    # instructions without a register result: stores, reductions, branches, votes into a predicate only
    no_dest = base in {"STS", "ST", "STG", "STL", "RED", "BRA", "EXIT", "BAR", "WARPSYNC", "NOP", "BSYNC", "BSSY"} or (
        base == "ATOMS" and len(ops) >= 1 and ops[0].startswith("["))
    dests, srcs = [], []
    for i, o in enumerate(ops):
        names = REG.findall(o)
        if not names:
            continue
        if not no_dest and i == 0 and not o.startswith("["):
            n0 = names[0]
            w = width(op) if "P" not in n0 else 1
            if n0.startswith(("R", "UR")):
                pre = "UR" if n0.startswith("UR") else "R"
                num = int(n0[len(pre):])
                dests += [f"{pre}{num + j}" for j in range(w)]
            else:
                dests.append(n0)
            continue
        # a second result in the second position: ISETP / FSETP / PLOP3 P0, P1, ...; IADD3 / LOP3 / LEA R, P0, ...
        if not no_dest and i == 1 and base in {"ISETP", "FSETP", "PLOP3", "IADD3", "LOP3", "LEA"} \
                and re.fullmatch(r"U?P\d+", o):
            dests.append(names[0])
            continue
        for nm in names:
            srcs.append(nm)
            # the 64-bit addend of IMAD.WIDE
            if ".WIDE" in op and i == 3 and nm.startswith("R"):
                srcs.append(f"R{int(nm[1:]) + 1}")
    if guard:
        srcs.append(guard)
    return op, [d for d in dests if d not in ("RZ", "PT", "URZ", "UPT")], [s for s in srcs if s not in ("RZ", "PT", "URZ", "UPT")]


def functions(lib):
    txt = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    for f in re.split(r"\n\s*Function : ", txt)[1:]:
        name = f.split("\n", 1)[0].strip()
        ins = []
        for line in f.split("\n"):
            m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
            if m:
                ins.append((int(m.group(1), 16), m.group(2).strip()))
        yield name, ins


BRANCH = re.compile(r"\b(BRA|BRX|JMP|CALL|RET|EXIT|BSSY|BSYNC|BREAK|WARPSYNC)\b")


def hot_loop(ins):
    """the largest backward branch whose body holds no other control flow"""
    idx = {a: i for i, (a, _) in enumerate(ins)}
    best = None
    for i, (a, t) in enumerate(ins):
        m = re.search(r"\bBRA(?:\.\w+)*\s+(?:\S+,\s*)?`?\(?0x([0-9a-f]+)", t)
        if not m:
            continue
        tgt = int(m.group(1), 16)
        if tgt > a or tgt not in idx:
            continue
        body = ins[idx[tgt]:i]
        if any(BRANCH.search(x) for _, x in body):
            continue
        if best is None or len(body) > best[1] - best[0]:
            best = (idx[tgt], i + 1)
    if best is None:
        raise SystemExit("no branch-free backward-branch loop found")
    return ins[best[0]:best[1]]


def critical_path(loop, iterations=4, in_order=False):
    """list of per-iteration finish times and the critical path (instruction indices) of the last iteration
    (in_order: also one issue per cycle in program order, and ISSUE_CYCLES between two instructions of one pipe)"""
    parsed = [parse(t) for _, t in loop]
    last_issue = -1
    pipe_free = collections.defaultdict(int)
    ready = collections.defaultdict(int)   # register -> cycle its value is available
    who = {}                               # register -> (iteration, instruction) that wrote it
    prev_lsu = (0, None)
    finish = []
    pred = {}
    for it in range(iterations):
        end_max = 0
        for j, (op, dests, srcs) in enumerate(parsed):
            start, src = 0, None
            for s in srcs:
                if ready[s] > start:
                    start, src = ready[s], who.get(s)
            if pipe(op) == "LSU" and prev_lsu[0] > start:
                start, src = prev_lsu[0], prev_lsu[1]
            if in_order:
                start = max(start, last_issue + 1, pipe_free[pipe(op)])
                last_issue = start
                pipe_free[pipe(op)] = start + ISSUE_CYCLES.get(pipe(op), 1)
            if pipe(op) == "LSU":
                prev_lsu = (start + 1, (it, j))
            end = start + latency(op)
            pred[(it, j)] = (src, end)
            for d in dests:
                ready[d] = end
                who[d] = (it, j)
            end_max = max(end_max, end)
        finish.append(end_max)
    # walk back from the latest-finishing instruction of the last iteration to where it enters that iteration
    last = iterations - 1
    node = max(((last, j) for j in range(len(parsed))), key=lambda n: pred[n][1])
    path = []
    while node is not None and node[0] == last:
        path.append(node[1])
        node = pred[node][0]
    return finish, path[::-1], node


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    lib = args[0] if args else DEFAULT_LIB
    key = args[1] if len(args) > 1 else DEFAULT_KERNEL
    found = False
    for name, ins in functions(lib):
        if key not in name:
            continue
        found = True
        loop = hot_loop(ins)
        print(f"{name}")
        print(f"  hot loop 0x{loop[0][0]:x} .. 0x{loop[-1][0]:x}: {len(loop)} instructions")
        per_pipe = collections.Counter(pipe(parse(t)[0]) for _, t in loop)
        print("  per pipe: " + ", ".join(f"{p} {per_pipe.get(p, 0)}" for p in ("ALU", "FMA-heavy", "FP32", "LSU", "other")))
        ops = collections.Counter(parse(t)[0].split(".")[0] for _, t in loop)
        print("  opcodes:  " + ", ".join(f"{k} {v}" for k, v in ops.most_common()))
        finish, path, entry = critical_path(loop)
        steps = [b - a for a, b in zip(finish, finish[1:])]
        print(f"  longest dependency path: {finish[0]} cycles in a first iteration; "
              f"{steps[-1]} cycles per iteration in steady state (growth over iterations: {steps})")
        print(f"  steady-state critical path: {len(path)} instructions, entering from "
              f"{'the previous iteration' if entry is not None else 'a loop-invariant value'}")
        io, _, _ = critical_path(loop, in_order=True)
        print(f"  with in-order issue (one instruction per cycle, ALU and FMA-heavy pipes two cycles per instruction): "
              f"{io[-1] - io[-2]} cycles per iteration")
        if "--path" in sys.argv:
            for j in path:
                a, t = loop[j]
                print(f"    0x{a:05x} {latency(parse(t)[0]):3d}  {t}")
    if not found:
        raise SystemExit(f"no kernel matching {key} in {lib}")


if __name__ == "__main__":
    main()
