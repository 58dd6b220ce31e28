#!/usr/bin/env python3
"""Apply INTEGRATION.md option B to the reference's own main-cli.c and (optionally) build it.

    python integration/apply_dropin.py REFERENCE_DIR/main-cli.c OUT.c              # splice only
    python integration/apply_dropin.py --build REFERENCE_DIR [OUT_DIR]             # splice + gcc -> OUT_DIR/smvp-toolkit-cli-dropin

REFERENCE_DIR is a checkout of circletile/smvp-toolkit (main-cli.c and mmio/ at its top level).

What changes in the reference's file (nothing else is touched):
  * `#include "smvp_cuda.h"` after `#include "mmio/mmio.h"`;
  * the body of `smvp_csr_compute`  (main-cli.c:325 ... :469)  -> integration/dropin_bodies.c, first block;
  * the body of `smvp_tjds_compute` (main-cli.c:734 ... :1162) -> integration/dropin_bodies.c, second block.
The functions are found by their signatures and brace matching, so this repository holds no line of the reference
(a unified diff would carry ~1200 removed lines of it).  The build uses plain gcc on the patched file + the
reference's mmio.c where they lie, the argv-only stub popt.h of oracle/stub (libpopt is not installed in this image),
and links libsmvp_cuda.so."""
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)


def body_of(text, name):
    """(start, end) offsets of the brace block that follows the definition `double *<name>(`."""
    m = re.search(r"^double \*%s\(" % re.escape(name), text, re.M)
    if not m:
        raise SystemExit("definition of %s not found: is this the reference's main-cli.c?" % name)
    i = text.index("{", m.end())
    depth, j = 0, i
    in_str = in_chr = in_line = in_block = False
    while j < len(text):
        ch, nxt = text[j], text[j + 1:j + 2]
        if in_line:
            in_line = ch != "\n"
        elif in_block:
            if ch == "*" and nxt == "/":
                in_block = False
                j += 1
        elif in_str:
            if ch == "\\":
                j += 1
            elif ch == '"':
                in_str = False
        elif in_chr:
            if ch == "\\":
                j += 1
            elif ch == "'":
                in_chr = False
        elif ch == "/" and nxt == "/":
            in_line = True
        elif ch == "/" and nxt == "*":
            in_block = True
        elif ch == '"':
            in_str = True
        elif ch == "'":
            in_chr = True
        elif ch == "{":
            depth += 1
        elif ch == "}":
            depth -= 1
            if depth == 0:
                return i, j + 1
        j += 1
    raise SystemExit("unbalanced braces after %s" % name)


def new_body(name):
    with open(os.path.join(HERE, "dropin_bodies.c")) as f:
        src = f.read()
    a = src.index("/* >>> %s */" % name) + len("/* >>> %s */" % name)
    b = src.index("/* <<< %s */" % name)
    return src[a:b].strip() + "\n"


def splice(ref_path, out_path):
    with open(ref_path) as f:
        text = f.read()
    for name in ("smvp_tjds_compute", "smvp_csr_compute"):  # back to front: offsets of the earlier one stay valid
        a, b = body_of(text, name)
        text = text[:a] + new_body(name).rstrip("\n") + text[b:]
    inc = '#include "mmio/mmio.h"'
    if inc not in text:
        raise SystemExit("include anchor not found")
    text = text.replace(inc, inc + '\n#include "smvp_cuda.h" /* smvp_coo has the layout of MMRawData (main-cli.c:42-47) */', 1)
    with open(out_path, "w") as f:
        f.write(text)
    return out_path


def build(ref_dir, out_dir=None):
    out_dir = out_dir or os.path.join(HERE, "_build")
    os.makedirs(out_dir, exist_ok=True)
    patched = splice(os.path.join(ref_dir, "main-cli.c"), os.path.join(out_dir, "main-cli.dropin.c"))
    lib = os.path.join(REPO, "smvp-toolkit_b200", "lib")
    exe = os.path.join(out_dir, "smvp-toolkit-cli-dropin")
    cmd = ["gcc", "-O2", "-w", "-D_XOPEN_SOURCE=700", "-I" + os.path.join(REPO, "oracle", "stub"), "-I" + os.path.join(REPO, "include"),
           "-I" + ref_dir, patched, os.path.join(ref_dir, "mmio", "mmio.c"), "-o", exe, "-L" + lib, "-lsmvp_cuda",
           "-Wl,-rpath," + lib, "-Wl,-rpath,$ORIGIN/../../smvp-toolkit_b200/lib", "-lm"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    os.remove(patched)  # the spliced file is mostly the reference's text: it is not kept
    if r.returncode != 0:
        raise SystemExit("drop-in build failed:\n" + r.stdout + r.stderr)
    return exe


if __name__ == "__main__":
    if len(sys.argv) in (3, 4) and sys.argv[1] == "--build":
        print(build(*sys.argv[2:4]))
    elif len(sys.argv) == 3:
        print(splice(sys.argv[1], sys.argv[2]))
    else:
        raise SystemExit(__doc__)
