"""Static SASS instruction counts of one kernel of libtsg.so, per device function and per source function.

usage: sass_size.py DIS [KERNEL]
  DIS     `nvdisasm -gi` output of the library's cubin (tools/README.md)
  KERNEL  substring of the mangled kernel name; default: the step kernel (MODE = 0) of the production shape,
          tb_env_kernel<P64, 0, 6, 10>

Every instruction carries its inline chain, innermost source line first.  Each source line is mapped to the TB_FN /
TB_NOINL / __global__ function of csrc/ whose definition precedes it.  `self` counts an instruction for the innermost
function of its chain, `incl` for every function of the chain once: a stage of phys() reports its own size under
`incl`, the helpers inlined into it included."""
import bisect
import collections
import os
import re
import sys

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tensegrity_rl_b200", "csrc")
DEF = re.compile(r"^(?:template\s*<.*?>\s*)?(?:TB_FN|TB_NOINL|__global__)\b.*?(\w+)\s*\(")


def definitions():
    """{file name: (sorted start lines, function names)} of the function definitions in csrc/"""
    out = {}
    for fname in sorted(os.listdir(CSRC)):
        starts, names = [], []
        for i, line in enumerate(open(os.path.join(CSRC, fname))):
            m = DEF.match(re.sub(r"__launch_bounds__\s*\(.*?\)", "", line))
            if m:
                starts.append(i + 1); names.append(m.group(1))
        out[fname] = (starts, names)
    return out


def function_of(defs, path, line):
    fname = os.path.basename(path)
    if fname not in defs:
        return fname
    starts, names = defs[fname]
    k = bisect.bisect_right(starts, line) - 1
    return names[k] if k >= 0 else fname


def device_function(symbol):
    m = re.search(r"\$_ZN2tb(\d+)(\w+)$", symbol)
    return m.group(2)[:int(m.group(1))] if m else symbol.split("$")[-1][:60]


def main():
    dis = sys.argv[1]
    want = sys.argv[2] if len(sys.argv) > 2 else "tb_env_kernelIN2tb3P64ELi0ELi6ELi10E"
    defs = definitions()
    loc = re.compile(r'//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?')
    sec, dev, chain = None, None, []
    per_dev, self_cnt, incl_cnt = collections.Counter(), collections.Counter(), collections.Counter()
    for l in open(dis):
        s = l.strip()
        if s.startswith(".section"):
            m = re.match(r"\.section\s+\.text\.([^,\s]+)", s)
            sec = m.group(1) if m and want in m.group(1) else None
            dev, chain = "kernel", []
            continue
        if sec is None:
            continue
        m = re.match(r"\.type\s+(\S+),@function", s)
        if m:
            dev = "kernel" if m.group(1) == sec else device_function(m.group(1))
            continue
        m = loc.search(s)
        if m:
            here = (m.group(1), int(m.group(2)))
            outer = (m.group(3), int(m.group(4))) if m.group(3) else None
            if chain and chain[-1][1] == here:   # the next level of the current chain
                chain.append((here, outer))
            else:
                chain = [(here, outer)]
            continue
        if re.match(r"/\*[0-9a-f]{4,}\*/\s+\S", s):
            per_dev[dev] += 1
            fns = [function_of(defs, p, n) for (p, n), _ in chain] or ["?"]
            self_cnt[fns[0]] += 1
            for f in set(fns):
                incl_cnt[f] += 1
    total = sum(per_dev.values())
    if not total:
        sys.exit("no instructions of a kernel matching %r in %s" % (want, dis))
    print("kernel *%s*: %d instructions" % (want, total))
    print("device functions:", ", ".join("%s %d" % kv for kv in per_dev.most_common()))
    print("%8s %8s  source function" % ("incl", "self"))
    for f, n in incl_cnt.most_common():
        print("%8d %8d  %s" % (n, self_cnt[f], f))


if __name__ == "__main__":
    main()
