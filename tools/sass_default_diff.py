"""Compare the SASS of the default (non-deterministic) kernel instantiations of two builds of the library.

    python tools/sass_default_diff.py PARENT.so NEW.so [--out report.txt]

The deterministic mode adds a trailing `bool DET` template argument (false = the atomic path) to the kernels it touches and
adds instantiations with DET = true. This tool dumps `cuobjdump -sass` of both libraries, demangles the function names,
maps `kernel<..., false>` of the new build onto `kernel<...>` of the old one (a kernel that gained its first template
argument maps `kernel<false>` onto `kernel`), and diffs the instruction streams with addresses and constant-bank parameter
offsets left in. Exit code 1 when a checked kernel differs or is missing."""
from __future__ import annotations

import argparse
import re
import subprocess
import sys

CHECKED = ("wgrad_kernel", "conv_igemm_kernel", "bn_stats_kernel", "bn_act_bwd_reduce_kernel", "bn_act_bwd_apply_kernel",
           "bn_act_kernel", "nchw_to_p8_ex_kernel", "conv_c1_wgrad", "loss_kernel")


def sass_functions(path):
    txt = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    funcs, name, body = {}, None, []
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = body
            name, body = m.group(1), []
            continue
        if name is None:
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m:
            body.append(m.group(1).strip())
    if name:
        funcs[name] = body
    names = list(funcs)
    dem = subprocess.run(["cu++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {d: funcs[n] for n, d in zip(names, dem)}


def key(name):
    """Demangled name without the parameter list (the deterministic kernels append a workspace parameter)."""
    name = name.split(" ", 1)[1] if name.startswith("void ") else name
    depth = 0
    for i, ch in enumerate(name):
        depth += {"<": 1, ">": -1}.get(ch, 0)
        if ch == "(" and depth == 0:
            return name[:i]
    return name


def split_last_arg(k):
    """(name without its last template argument, that argument) or (k, None)."""
    if not k.endswith(">"):
        return k, None
    depth = 0
    for i in range(len(k) - 1, -1, -1):
        depth += {">": 1, "<": -1}.get(k[i], 0)
        if depth == 0:
            args = k[i + 1:-1]
            break
    parts = [a.strip() for a in re.split(r",(?![^<]*>)", args)]
    head = k[:i]
    return head + ("<" + ", ".join(parts[:-1]) + ">" if len(parts) > 1 else ""), parts[-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    old = {key(n): b for n, b in sass_functions(a.old).items()}
    new = {key(n): b for n, b in sass_functions(a.new).items()}
    lines, bad = [], 0
    for name, body in sorted(new.items()):
        if not any(k in name for k in CHECKED):
            continue
        ref = old.get(name)
        if ref is None:
            base, last = split_last_arg(name)
            if last == "(bool)1" and name[:-len("(bool)1>")] + "(bool)0>" in new:      # the DET = true sibling of a default kernel
                lines.append(f"new (deterministic)  {name}")
                continue
            ref = old.get(base) if last == "(bool)0" else None
        if ref is None:
            lines.append(f"MISSING in old       {name}")
            bad += 1
        elif ref != body:
            lines.append(f"DIFFERENT            {name}  ({len(ref)} -> {len(body)} instructions)")
            bad += 1
        else:
            lines.append(f"identical            {name}  ({len(body)} instructions)")
    lines.append(f"{bad} checked default kernel(s) differ or are missing")
    report = "\n".join(lines)
    print(report)
    if a.out:
        with open(a.out, "w") as f:
            f.write(report + "\n")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
