"""Static SASS statistics of one kernel of a built libuavca: instruction count up to the first unconditional EXIT
(the common path of the step kernels), per-opcode and per-source-line (needs -lineinfo).
    python tools/sass_stats.py LIB.so KERNEL_SUBSTRING [--lines] [--list]
    python tools/sass_stats.py LIB.so KERNEL_SUBSTRING --loop [--via OPCODE]

--loop reports each outermost loop of the kernel (a backward branch and the code between its target and itself; the
K loop of a rollout kernel, once per warp specialisation).  Its common path is the shortest path through the loop's
control-flow graph from the head to the back edge: rare work (auto-reset, counters, degenerate angles) sits behind
branches that skip it, and divergence fallbacks (BRA.DIV) are never shorter.  --via OPCODE makes the path pass an
instruction of that opcode (e.g. LDGSTS: the action-block prefetch of a kernel whose loop also holds the Philox path).
For the path it prints the instruction count, the opcode mix and every S2R, S2UR, LDC*, LDL and STL; for the whole loop
range, the count of those."""
import heapq, re, subprocess, sys, tempfile, os
from collections import Counter

WATCH = ("S2R", "S2UR", "LDC", "LDCU", "LDL", "STL")


def disassemble(lib, pat):
    d = tempfile.mkdtemp()
    subprocess.check_call(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=d, stdout=subprocess.DEVNULL)
    cub = [f for f in os.listdir(d) if f.startswith("uavca_kernels.")][0]
    txt = subprocess.run(["nvdisasm", "--print-line-info", os.path.join(d, cub)], capture_output=True, text=True).stdout
    insts, labels = [], {}  # (line info, text); label -> instruction index
    inside = False; cur = None; name = None
    for l in txt.split("\n"):
        if l.startswith(".text."):
            if inside: break  # the first kernel whose name contains pat
            inside = pat in l
            name = l[6:].rstrip(":")
            continue
        if not inside: continue
        m = re.match(r"(\.L_x_\d+):", l)
        if m:
            labels[m.group(1)] = len(insts); continue
        m = re.search(r'//## File "([^"]+)", line (\d+)', l)
        if m:
            cur = (m.group(1).split("/")[-1], int(m.group(2))); continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
        if m: insts.append((cur, m.group(2)))
    return name, insts, labels


def opcode(t):
    op = t.split()
    if op[0].startswith("@"): op = op[1:]
    return op[0].split(".")[0]


def successors(i, t, labels):
    """control-flow successors of instruction i (text t)"""
    op = opcode(t)
    pred = t.startswith("@")
    m = re.search(r"`\((\.L_x_\d+)\)", t)
    if op in ("BRA", "JMP") and m:
        tgt = labels[m.group(1)]
        # conditional: a guard predicate, a uniform/predicate operand (BRA.U !UP0, BRA P3), or a divergence test
        cond = pred or ".DIV" in t.split()[0 if not pred else 1] or re.search(r"BRA(\.\w+)*\s+!?U?P\d", t) is not None
        return [tgt, i + 1] if cond else [tgt]
    if op in ("EXIT", "RET") and not pred: return []
    return [i + 1]


def shortest(insts, labels, lo, hi, src, dst):
    """fewest instructions on a path src -> dst inside [lo, hi] (both ends counted); None when unreachable"""
    dist = {src: 1}; prev = {}; q = [(1, src)]
    while q:
        d, i = heapq.heappop(q)
        if i == dst: break
        if d > dist.get(i, 1 << 30): continue
        for j in successors(i, insts[i][1], labels):
            if lo <= j <= hi and d + 1 < dist.get(j, 1 << 30):
                dist[j] = d + 1; prev[j] = i; heapq.heappush(q, (d + 1, j))
    if dst not in dist: return None
    path = [dst]
    while path[-1] != src: path.append(prev[path[-1]])
    return path[::-1]


def loops(insts, labels):
    """outermost loops: (head, back edge) of every backward branch not inside a larger one"""
    spans = []
    for i, (_, t) in enumerate(insts):
        m = re.search(r"`\((\.L_x_\d+)\)", t)
        # a loop's back edge tests the loop condition; the unconditional backward branches are out-of-line blocks
        # (divergence fallbacks, rare paths) returning to the code they left
        if m and opcode(t) == "BRA" and labels[m.group(1)] <= i and len(successors(i, t, labels)) == 2:
            spans.append((labels[m.group(1)], i))
    spans.sort(key=lambda s: (s[0], -s[1]))
    out = []
    for s in spans:
        if not any(o[0] <= s[0] and s[1] <= o[1] for o in out): out.append(s)
    return out


def loop_report(name, insts, labels, via):
    print(f"kernel {name}")
    for n, (h, b) in enumerate(loops(insts, labels)):
        if via:
            best = None
            for v in range(h, b + 1):
                if opcode(insts[v][1]) != via: continue
                p1 = shortest(insts, labels, h, b, h, v); p2 = shortest(insts, labels, h, b, v, b)
                if p1 and p2 and (best is None or len(p1) + len(p2) - 1 < len(best)): best = p1 + p2[1:]
            path = best
        else:
            path = shortest(insts, labels, h, b, h, b)
        body = insts[h:b + 1]
        print(f"loop {n}: instructions {h}..{b} ({len(body)} in the loop range)")
        if path is None:
            print("  no path" + (f" through {via}" if via else "")); continue
        ops = Counter(opcode(insts[i][1]) for i in path)
        print(f"  common path: {len(path)} instructions" + (f" (through {via})" if via else ""))
        print("  " + " ".join(f"{k}:{v}" for k, v in ops.most_common()))
        watched = [i for i in path if opcode(insts[i][1]) in WATCH]
        print(f"  S2R/S2UR/LDC*/LDL/STL on the path: {len(watched)}")
        for i in watched:
            c, t = insts[i]
            print(f"    {c[0]}:{c[1]:<5d} {t}" if c else f"    {t}")
        rng = Counter(opcode(t) for _, t in body if opcode(t) in WATCH)
        print("  in the whole loop range: " + (" ".join(f"{k}:{v}" for k, v in sorted(rng.items())) or "none"))


def main():
    lib, pat = sys.argv[1], sys.argv[2]
    name, insts, labels = disassemble(lib, pat)
    if "--loop" in sys.argv:
        via = sys.argv[sys.argv.index("--via") + 1] if "--via" in sys.argv else None
        loop_report(name, insts, labels, via)
        return
    n = 0; ops = Counter(); cnt = Counter(); listing = []
    for cur, t in insts:
        n += 1
        ops[opcode(t)] += 1
        cnt[cur] += 1
        listing.append((cur, t))
        if opcode(t) == "EXIT" and not t.startswith("@"): break
    print("instructions to first EXIT:", n)
    print(" ".join(f"{k}:{v}" for k, v in ops.most_common()))
    if "--lines" in sys.argv:
        for k, v in sorted(cnt.items(), key=lambda kv: (kv[0] or ("", 0))): print(k, v)
    if "--list" in sys.argv:
        for c, t in listing: print(f"{c[0]}:{c[1]:<5d} {t}" if c else t)


if __name__ == "__main__":
    main()
