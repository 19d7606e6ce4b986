"""Per-function SASS comparison of two builds of libnmpc_b200.so (runs on any machine with the CUDA toolkit; no GPU needed).

    python tools/sass_diff.py OLD.so NEW.so [REGEX]

Extracts the sm_100a cubin of both libraries (cuobjdump -xelf), disassembles it with nvdisasm, and splits every kernel into
its functions: the kernel body and each device function it calls (the solver's noinline passes).  Instruction addresses and
encodings are stripped, return addresses loaded into registers are made relative to their function, branch labels are
renumbered within each function, and the compiler's numbering of specialised
copies (`_$_specialized_$_N`) and of the CUDA math helpers (`__internal_N_$__cuda_sm20_div_rn_f64_full`, numbered in the order
the file's kernels use them, so a kernel added to the file renumbers them everywhere) is dropped, so that two builds compare equal when every function has the same instructions,
wherever the linker placed it.  Kernel and function names are compared with a trailing `false` template argument removed, so
that WarpSolver<NR, OBS> / solve_kernel<NR, OBS> of an older build pair with <NR, OBS, false> of a newer one.
REGEX selects kernels by mangled name (default: the warp-path solve kernels without the tracking flag, solve_kernel<1..10,
false> and solve_kernel<1..4, true>).  Exit code 0 when every selected kernel is the same, 1 otherwise."""
import glob
import os
import re
import subprocess
import sys
import tempfile

DEFAULT = r"^_Z12solve_kernelILi\d+ELb[01]EEv15NmpcSolveParams$"


def _norm(name):
    name = re.sub(r"(ILi\d+ELb[01])ELb0EE", r"\1EE", name)
    name = re.sub(r"__internal_\d+_", "__internal_", name)
    return re.sub(r"_\$_specialized_\$_\d+", "_$_specialized", name)


def kernels(so):
    """{kernel: {function: sorted list of instruction lists}} of the library's sm_100a cubin."""
    with tempfile.TemporaryDirectory() as d:
        subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(so)], cwd=d, check=True, capture_output=True)
        cubins = sorted(glob.glob(d + "/*sm_100a*.cubin"))
        if not cubins:
            raise SystemExit("%s: no sm_100a cubin" % so)
        txt = "".join(subprocess.run(["nvdisasm", "-c", c], check=True, capture_output=True, text=True).stdout for c in cubins)
    out, fn, body = {}, None, []

    def flush():
        if fn is not None and body:
            labels = {}
            lo, hi = body[0][0], body[-1][0]

            def local(m):     # an address inside this function (a return address put in a register): relative to its start
                v = int(m.group(1), 16)
                return "+0x%x" % (v - lo) if lo <= v <= hi + 16 else m.group(0)
            ins = [re.sub(r"\.L_x_\d+", lambda m: "L%d" % labels.setdefault(m.group(0), len(labels)), b) for _, b in body]
            ins = [re.sub(r"0x([0-9a-f]+)", local, b) if b.startswith("MOV ") else b for b in ins]
            out.setdefault(fn[0], {}).setdefault(fn[1], []).append(ins)
    for line in txt.splitlines():
        m = re.match(r"^(\$?)([A-Za-z_][\w$]*):\s*$", line)
        if m and not line.startswith(".text"):
            flush()
            lab = m.group(2)
            if m.group(1):      # $kernel$function
                k, f = lab.split("$", 1)
            else:
                k, f = lab, lab
            fn, body = (_norm(k), _norm(f)), []
            continue
        m = re.match(r"^\s*/\*([0-9a-f]+)\*/(.*)$", line)
        if fn is not None and m:
            ins = re.sub(r"/\* 0x[0-9a-f]{16} \*/", "", m.group(2)).strip()
            if ins:
                body.append((int(m.group(1), 16), _norm(ins)))
    flush()
    for k in out:
        for f in out[k]:
            out[k][f].sort()
    return out


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    pat = re.compile(sys.argv[3] if len(sys.argv) > 3 else DEFAULT)
    sel = sorted(k for k in old if pat.search(k))
    bad = 0
    for k in sel:
        if k not in new:
            print("MISSING in new build:", k)
            bad += 1
            continue
        diff = sorted(f for f in set(old[k]) | set(new[k]) if old[k].get(f) != new[k].get(f))
        n = sum(len(b) for bs in old[k].values() for b in bs)
        if diff:
            print("DIFFERS: %s in %d function(s): %s" % (k, len(diff), ", ".join(diff[:4])))
            bad += 1
        else:
            print("same:    %s (%d functions, %d instructions)" % (k, sum(len(v) for v in old[k].values()), n))
    print("%d kernel(s) compared, %d differ" % (len(sel), bad))
    return 1 if bad or not sel else 0


if __name__ == "__main__":
    sys.exit(main())
