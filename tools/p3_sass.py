"""SASS instructions per position of the nibble kernel's P3 (frisk_nibble.cu), counted from the compiler's output.

    python tools/p3_sass.py [K PP ALLK MODE]        default: 8 20 1 0 (the C2 instantiation score_windows_nibble_kernel<8,20,0,1,0>)

Compiles frisk_nibble.cu for sm_100a into a temporary cubin, disassembles that instantiation with line information and
prints, for every loop that holds the 256-bit pair gathers (LDG.E.ENL2.256): its instructions, those on the side-list
source lines (rarely run: a short word of K-1 / K-2 bases below the K-mer's bin), and the rest per position (one gather
serves two positions).  No GPU needed."""
import os, re, subprocess, sys, tempfile

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "frisk_b200", "csrc")
SIDE = re.compile(r"n_side|ss\.side\[|side_add\(|sv = e >> 16|code == |code >> 2")      # the side-list code of P3


def main(argv):
    K, PP, ALLK, MODE = (argv + ["8", "20", "1", "0"][len(argv):])[:4]
    src = os.path.join(CSRC, "frisk_nibble.cu")
    text = open(src).read().splitlines()
    with tempfile.TemporaryDirectory() as tmp:
        cubin = os.path.join(tmp, "nib.cubin")
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo",
                               "-diag-suppress", "186", "-cubin", src, "-o", cubin], cwd=CSRC)
        sass = subprocess.check_output(["nvdisasm", "-g", "-c", cubin], text=True).splitlines()
    tag = "score_windows_nibble_kernelILi%sELi%sELb0ELb%sELi%sEE" % (K, PP, ALLK, MODE)
    start = next(i for i, l in enumerate(sass) if l.startswith(".text.") and tag in l)
    ins, labels, line = [], {}, None
    for l in sass[start + 1:]:
        if l.startswith(".text.") or l.startswith("\t.section"):
            break
        m = re.match(r"^(\.L_x_\d+):", l)
        if m:
            labels[m.group(1)] = len(ins)
        elif l.strip().startswith("//##"):
            m = re.search(r'File "([^"]+)", line (\d+)', l)
            line = (os.path.basename(m.group(1)), int(m.group(2))) if m else None
        else:
            m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
            if m:
                side = line is not None and line[0] == "frisk_nibble.cu" and bool(SIDE.search(text[line[1] - 1]))
                ins.append((m.group(2), side))
    print("score_windows_nibble_kernel<%s,%s,0,%s,%s>: %d instructions" % (K, PP, ALLK, MODE, len(ins)))
    loops = []                                       # (head, back branch) of every loop that holds a pair gather
    for i, (op, _) in enumerate(ins):
        m = re.search(r"BRA.*`\((\.L_x_\d+)\)", op)
        if m and labels.get(m.group(1), len(ins)) <= i and any("ENL2.256" in o for o, _ in ins[labels[m.group(1)]:i + 1]):
            loops.append((labels[m.group(1)], i))
    for a, b in loops:                               # the round loops: those without another such loop inside
        if not any((a, b) != (c, d) and a <= c and d <= b for c, d in loops):
            body = ins[a:b + 1]
            gathers = sum("ENL2.256" in op for op, _ in body)
            side = sum(s for _, s in body)
            print("loop of %d instructions, %d pair gathers: %d on side-list lines, %.1f per position otherwise"
                  % (len(body), gathers, side, (len(body) - side) / (2.0 * gathers)))


if __name__ == "__main__":
    main(sys.argv[1:])
