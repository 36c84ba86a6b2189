"""Static instruction budget of the flat-scene bounce kernels the Cornell workload (C2) launches. Needs no GPU.

    python tools/flat_sass_budget.py [--src DIR] [--cubin FILE] [--form uniform|shared]

Compiles DIR/2019global_b200/csrc/path_kernels.cu (default: this checkout) with the build's flags (build.py) into a
cubin, or reads --cubin, disassembles it with nvdisasm's inlining line info, and prints for

    bounce_flat_fused_kernel<false, false, false>  camera segment + first vertex (bounce 0)
    bounce_flat_kernel<false>                      the middle bounces
    bounce_flat_kernel<true>                       the bounce before the last, which shades the last vertex (FOLD)

the registers and spill bytes (ptxas), and the static instructions of the vertex loop (the loop over queue entries in
bounce_flat_body) split by the innermost project function they come from. The primitive-pair code is counted per call of
trace_flat and per kind group: a loop body once, or the unrolled copies (FlatPairsU capacity). Per planar pair counts
both planar groups (parallelograms, triangles) together over their copies, since the line table may credit one group's
instructions to the other's call line. "C2 trip" = the loop without pair code + per trace call 3 parallelogram pairs (five walls
and the light) + 1 sphere pair (the two spheres): a static estimate of the instructions one queue entry costs.
--form picks the kernels that read the pairs from their FlatPairsU launch parameter (uniform, the default where they
exist) or the shared-memory loops (shared).
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = "/usr/local/cuda/bin/"
C2_KERNELS = [
    ("fused (bounce 0)", r"bounce_flat_fused_kernel<false, false, false(, %s)?(, false)?>"),
    ("plain (middle bounces)", r"bounce_flat_kernel<false, %s>"),
    ("FOLD (bounce before the last)", r"bounce_flat_kernel<true, %s>"),
]
# pair code: planar pair functions / sphere pair functions (the parent's sphere loop body lived in trace_flat itself)
PLANAR = {"plane_pairs", "plane_pairs_u", "plane_pair", "plane_origin2", "plane_uvt2", "plane_inside"}
SPHERE = {"sphere_pair", "sphere_roots2"}


def compile_cubin(src_root, out):
    sys.path.insert(0, os.path.join(src_root, "2019global_b200"))
    import build  # the build's flags
    sys.path.pop(0)
    extra = dict(build.UNITS)["path_kernels.cu"]
    common = [f.replace(os.path.join(ROOT, "include"), os.path.join(src_root, "include")) for f in build.COMMON]
    cmd = ([build.NVCC] + build.ARCH + common + extra + ["-I", os.path.join(src_root, "include"), "-I",
           os.path.join(src_root, "2019global_b200", "csrc"), "-cubin", "-x", "cu",
           os.path.join(src_root, "2019global_b200", "csrc", "path_kernels.cu"), "-o", out])
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stderr)
        raise SystemExit("nvcc failed")
    return r.stderr


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    return {n: re.sub(r"g19::\(anonymous namespace\)::", "", d) for n, d in zip(names, out)}


def ptxas_usage(log):
    use = {}
    for m in re.finditer(r"Compiling entry function '(\S+)' for 'sm_100a'\n.*\n\s+(\d+) bytes stack frame, (\d+) bytes spill "
                         r"stores, (\d+) bytes spill loads\n.*Used (\d+) registers", log):
        use[m.group(1)] = (int(m.group(5)), int(m.group(3)), int(m.group(4)))
    return use


def functions(path):
    """(first line, last line, name) of every function definition in a source file, by brace matching."""
    lines = open(path).read().split("\n")
    spans = []
    pat = re.compile(r"^(?:template <[^>]*>\s*)?(?:__device__|__global__|static)[^;{]*?\b(\w+)\s*\(")
    i = 0
    while i < len(lines):
        m = pat.match(lines[i]) if not lines[i].startswith(" ") else None
        if m is None and lines[i].startswith("    __device__"):  # member functions
            m = re.match(r"^\s+__device__[^;{]*?\b(\w+)\s*\(", lines[i])
        if m:
            depth, j, opened = 0, i, False
            while j < len(lines):
                depth += lines[j].count("{") - lines[j].count("}")
                opened = opened or "{" in lines[j]
                if opened and depth <= 0:
                    break
                if not opened and lines[j].rstrip().endswith(";"):
                    break
                j += 1
            if opened:
                spans.append((i + 1, j + 1, m.group(1)))
        i += 1
    return lines, spans


def find_fn(spans, line):
    best = None
    for a, b, n in spans:
        if a <= line <= b and (best is None or b - a < best[1] - best[0]):
            best = (a, b, n)
    return best


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--src", default=ROOT, help="repository tree whose path_kernels.cu is compiled")
    ap.add_argument("--cubin", help="read this cubin instead of compiling (registers / spills then not shown)")
    ap.add_argument("--form", choices=("uniform", "shared"), default="uniform")
    args = ap.parse_args()
    src = os.path.join(os.path.abspath(args.src), "2019global_b200", "csrc", "path_kernels.cu")
    with tempfile.TemporaryDirectory() as tmp:
        cubin, log = args.cubin, ""
        if not cubin:
            cubin = os.path.join(tmp, "path_kernels.cubin")
            log = compile_cubin(os.path.abspath(args.src), cubin)
        dis = subprocess.run([CUDA + "nvdisasm", "-gi", cubin], capture_output=True, text=True).stdout
    usage = ptxas_usage(log)
    lines, spans = functions(src)
    # the vertex loop of bounce_flat_body and, in trace_flat, the call lines of the kind groups
    body = next(s for s in spans if s[2] == "bounce_flat_body")
    loop_a = next(i for i in range(body[0], body[1]) if re.search(r"for \(; q - lane < n; q \+= stride\)", lines[i - 1]))
    depth, loop_b = 0, loop_a
    for loop_b in range(loop_a, body[1] + 1):
        depth += lines[loop_b - 1].count("{") - lines[loop_b - 1].count("}")
        if depth == 0:
            break
    tf = next(s for s in spans if s[2] == "trace_flat")
    sph_loop, sph_loop_u = set(), set()  # trace_flat lines of the sphere loops (all / the unrolled one)
    for i in range(tf[0], tf[1] + 1):
        text = lines[i - 1]
        if "j < p_sph" in text or "j < uint32_t(kUniSpherePairs)" in text:
            span, d, k = {i}, 0, i
            if not text.rstrip().endswith(";"):
                while True:
                    d += lines[k - 1].count("{") - lines[k - 1].count("}")
                    span.add(k)
                    if d <= 0 and k > i:
                        break
                    k += 1
            sph_loop |= span
            if "kUniSpherePairs" in text:
                sph_loop_u |= span
    hdr = open(os.path.join(os.path.dirname(src), "path.h")).read()
    m1, m2 = re.search(r"kUniPlanarPairs = (\d+)", hdr), re.search(r"kUniSpherePairs = (\d+)", hdr)

    # split the disassembly into kernels: name -> list of (opcode, chain of source lines, innermost first)
    kernels, cur, chain, pending = {}, None, [], []
    for ln in dis.split("\n"):
        m = re.match(r"^(_Z\w+):$", ln)
        if m:
            cur = kernels.setdefault(m.group(1), [])
            chain, pending = [], []
            continue
        if cur is None:
            continue
        m = re.match(r'\s*//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?', ln)
        if m:
            pending.append((m.group(1), int(m.group(2))))
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", ln)
        if m:
            if pending:
                chain, pending = pending, []
            cur.append((m.group(1), [l for f, l in chain if f.endswith("path_kernels.cu")]))
    names = demangle(list(kernels))
    form_tag = "true" if args.form == "uniform" else "false"
    print("source: %s  form: %s" % (src, args.form))
    for label, pat in C2_KERNELS:
        cands = [k for k, d in names.items() if re.fullmatch(r"void " + (pat % form_tag) + r"\(g19::PassArgs(, int)?(, g19::FlatPairsU)?\)", d)]
        cands.sort(key=lambda k: len(names[k]), reverse=(args.form == "uniform"))
        if not cands:
            print("\n%s: not found" % label)
            continue
        k = cands[0]
        ins = kernels[k]
        regs = usage.get(k)
        print("\n%s  %s" % (label, names[k].split("(")[0]))
        if regs:
            print("  registers %d, spill stores %d B, spill loads %d B" % regs)
        print("  static instructions: kernel %d" % len(ins))
        outside = collections.Counter()
        pairs = collections.Counter()  # (call line, group) -> instructions
        unrolled = collections.defaultdict(bool)
        for op, ch in ins:
            if not any(loop_a <= l <= loop_b and find_fn(spans, l)[2] == "bounce_flat_body" for l in ch):
                continue
            fns = [(l, find_fn(spans, l)) for l in ch]
            fns = [(l, f[2] if f else "?") for l, f in fns]
            call = next((l for l, f in fns if f == "bounce_flat_body"), 0)
            group = None
            tf_line = next((l for l, f in fns if f == "trace_flat"), None)
            if any(f in SPHERE for _, f in fns) or (tf_line in sph_loop):
                group = "sphere"
            elif any(f in PLANAR for _, f in fns) and tf_line is not None:
                group = "planar@%d" % tf_line
            if group:
                pairs[(call, group)] += 1
                if any(f == "plane_pairs_u" for _, f in fns) or (group == "sphere" and tf_line in sph_loop_u):
                    unrolled[(call, group)] = True
                continue
            outside[fns[0][1] if fns else "?"] += 1
        n_out = sum(outside.values())
        print("  vertex loop (lines %d-%d): %d static, %d of them outside the pair code" % (
            loop_a, loop_b, n_out + sum(pairs.values()), n_out))
        for f, n in outside.most_common(12):
            print("    %-28s %5d" % (f, n))
        rest = n_out - sum(n for _, n in outside.most_common(12))
        if rest:
            print("    %-28s %5d" % ("(other functions)", rest))
        trip = n_out
        calls = sorted({c for c, _ in pairs})
        for c in calls:
            desc, planar_n, planar_copies = [], 0, 0
            for g in sorted(g for cc, g in pairs if cc == c):
                n = pairs[(c, g)]
                copies = (int(m2.group(1)) if g == "sphere" else int(m1.group(1))) if unrolled[(c, g)] else 1
                desc.append("%s %d static%s" % ("sphere" if g == "sphere" else "planar group (line %s)" % g.split("@")[1], n,
                                                 " in %d unrolled copies" % copies if copies > 1 else ""))
                if g == "sphere":
                    trip += n / copies
                else:
                    planar_n, planar_copies = planar_n + n, planar_copies + copies
            # per planar pair: both planar groups together (the compiler may credit one group's instructions to the
            # other's line), over their copies
            if planar_copies:
                trip += 3 * planar_n / planar_copies
                desc.append("-> %.1f per planar pair" % (planar_n / planar_copies))
            print("  trace_flat called at line %d: %s" % (c, "; ".join(desc)))
        print("  C2 trip (loop outside pairs + per call 3 parallelogram pairs + 1 sphere pair): %.0f" % trip)


if __name__ == "__main__":
    main()
