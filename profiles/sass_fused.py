#!/usr/bin/env python
"""SASS budget of the fused GMW forward (no GPU needed).

Compiles dcd_b200/csrc/gmw_mlp_fused.cu for sm_100a with the library's flags (dcd_b200/build.py), disassembles it and prints,
for every instantiation mlp_fused_kernel<UPO>: registers, stack frame, spills, total instructions, and for each converter step
loop — the innermost loop that holds a cluster of F2FP.F16.F32.PACK_AB (the FP16 hi/-lo split of one unit) — its static size,
its common path per step and its opcode histogram.

    python profiles/sass_fused.py [--json FILE] [--hist N] [-D MACRO[=VALUE] ...]

Common path = the fewest instructions from the loop head to its back edge, forward branches only, divided by the steps one
loop iteration converts (its F2FP clusters; the loop is unrolled): an inner spin loop counts once, a block that a forward
branch can skip (object boundary, partial post) counts as skipped.  That is what a steady-state step issues when no wait has
to repeat — but only where every step runs its statistics unconditionally: in the full-slice kind0 and kind2 loops.  In
the tail loops (`nv > 0`, `st_load`) and in the first layer (`t >= 2`) the shortest path skips the statistics, so no common
path is reported for them.  The budget (12 units x 150 / 4 schedulers = 450 issue cycles, under the 576 tensor cycles of a
48-edge tile) is stated against the full kind0 / kind2 figure.

Step loop kinds: "kind0" (residual update -> folded preconv.conv1: reads X and applies ReLU), "first" (the net's first layer:
reads X, no accumulators), "kind2" (conv2); "full" is the variant without tail masks (all CTAs whose slice has no padding),
"tail" the other one.
"""
import argparse
import collections
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dcd_b200 import build as B  # noqa: E402

SRC = os.path.join(B.CSRC, "gmw_mlp_fused.cu")
INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)(.*?);")
BRANCH = re.compile(r"(0x[0-9a-f]+)\s*$")
PACK = "F2FP.F16.F32.PACK_AB"


def nvcc_path():
    n = B._nvcc()
    return n if os.path.isabs(n) else shutil.which(n)


def compile_and_dump(defines):
    nvcc = nvcc_path()
    if not nvcc:
        raise FileNotFoundError("nvcc not found")
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    with tempfile.TemporaryDirectory() as tmp:
        cubin = os.path.join(tmp, "fused.cubin")
        flags = [f for f in B.NVCC_FLAGS if f not in ("-Xcompiler", "-fPIC", "-fvisibility=hidden")]
        cmd = [nvcc] + flags + ["-D" + d for d in defines] + ["-Xptxas", "-v", "-cubin", "-o", cubin, SRC]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(res.stdout + res.stderr)
        sass = subprocess.run([cuobjdump, "-sass", cubin], capture_output=True, text=True, check=True).stdout
    return res.stdout + res.stderr, sass


def ptxas_info(log):
    """{mangled name: {registers, stack, spill_stores, spill_loads}} from -Xptxas -v."""
    out, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), {})
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur is not None:
            cur.update(stack=int(m.group(1)), spill_stores=int(m.group(2)), spill_loads=int(m.group(3)))
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and cur is not None:
            cur["registers"] = int(m.group(1))
    return out


def functions(sass):
    """{mangled name: [(addr, opcode, operands)]}, NOPs dropped."""
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        m = INSN.match(line)
        if m and cur is not None and m.group(3) != "NOP":
            cur.append((int(m.group(1), 16), m.group(3), (m.group(2) or "") + m.group(4)))
    return out


def is_branch(op):
    return op.split(".")[0] in ("BRA", "JMP")


def branch_target(operands):
    m = BRANCH.search(operands.strip())
    return int(m.group(1), 16) if m else None


def step_loops(ins):
    """(head index, back-edge index) of every innermost loop holding at least 8 PACKs."""
    idx = {a: i for i, (a, _, _) in enumerate(ins)}
    loops = []
    for i, (a, op, opr) in enumerate(ins):
        if is_branch(op):
            t = branch_target(opr)
            if t is not None and t <= a and t in idx:
                h = idx[t]
                if sum(1 for _, o, _ in ins[h:i + 1] if o == PACK) >= 8:
                    loops.append((h, i))
    return [(h, e) for h, e in loops if not any((h2, e2) != (h, e) and h <= h2 and e2 <= e for h2, e2 in loops)]


def common_path(ins, h, e):
    """Fewest instructions from ins[h] to the back edge ins[e], following forward edges inside the loop only."""
    INF = float("inf")
    addr = {a: i for i, (a, _, _) in enumerate(ins)}
    best = [INF] * (e + 1)
    best[h] = 1
    for i in range(h, e):
        if best[i] == INF:
            continue
        _, op, opr = ins[i]
        # guarded: a predicate in front ("@P0 BRA") or a predicate operand ("BRA.U !UP0, 0x...")
        guarded = opr.lstrip().startswith("@") or "," in opr.split("0x")[0]
        unconditional = (is_branch(op) or op == "EXIT") and not guarded
        if is_branch(op):
            t = branch_target(opr)
            if t is not None and t in addr and addr[t] > i and addr[t] <= e:
                best[addr[t]] = min(best[addr[t]], best[i] + 1)
        if not unconditional:
            best[i + 1] = min(best[i + 1], best[i] + 1)
    return best[e]


def classify(ins, h, e):
    c = collections.Counter(op for _, op, _ in ins[h:e + 1])
    x_loads = sum(v for k, v in c.items() if k.startswith("LDS.128"))
    if x_loads >= 4:
        return "kind0" if c.get("FMNMX", 0) >= 16 else "first"
    return "kind2"


def analyse(defines=(), hist=12):
    log, sass = compile_and_dump(defines)
    info = ptxas_info(log)
    report = {}
    for name, ins in functions(sass).items():
        m = re.search(r"mlp_fused_kernelILi(\d+)E", name)
        if not m:
            continue
        upo = int(m.group(1))
        loops = []
        for h, e in step_loops(ins):
            body = ins[h:e + 1]
            steps = max(1, sum(1 for _, o, _ in body if o == PACK) // 16)
            loops.append({"kind": classify(ins, h, e), "start": "0x%x" % ins[h][0], "static": len(body), "steps": steps,
                          "common_path": common_path(ins, h, e) / steps,
                          "local_memory": sum(1 for _, o, _ in body if o.startswith(("LDL", "STL"))),
                          "opcodes": dict(collections.Counter(o for _, o, _ in body).most_common())})
        by_kind = collections.defaultdict(list)
        for lp in loops:
            by_kind[lp["kind"]].append(lp)
        for lst in by_kind.values():
            lst.sort(key=lambda lp: lp["static"])
            for j, lp in enumerate(lst):
                lp["variant"] = "full" if j == 0 and len(lst) > 1 else ("tail" if len(lst) > 1 else "-")
                if lp["variant"] != "full" or lp["kind"] == "first":
                    lp["common_path"] = None      # (the shortest path skips the statistics: not a steady-state step)
        report[upo] = dict(info.get(name, {}), instructions=len(ins), step_loops=loops)
    return dict(sorted(report.items()))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--json", help="also write the report as JSON")
    ap.add_argument("--hist", type=int, default=12, help="opcodes shown per step loop")
    ap.add_argument("-D", dest="defines", action="append", default=[], help="extra macro for the compile")
    args = ap.parse_args()
    rep = analyse(args.defines, args.hist)
    for upo, r in rep.items():
        print("UPO=%d  registers %s  stack %s B  spills %s/%s B  instructions %d" % (
            upo, r.get("registers"), r.get("stack"), r.get("spill_stores"), r.get("spill_loads"), r["instructions"]))
        for lp in sorted(r["step_loops"], key=lambda lp: (lp["kind"], lp["variant"])):
            top = ", ".join("%s %d" % kv for kv in list(lp["opcodes"].items())[:args.hist])
            cp = "%6.1f" % lp["common_path"] if lp["common_path"] is not None else "     -"
            print("   %-6s %-4s @%-6s static %4d (%d steps)  common path per step %s  local %d | %s" % (
                lp["kind"], lp["variant"], lp["start"], lp["static"], lp["steps"], cp, lp["local_memory"], top))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
