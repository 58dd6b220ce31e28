"""INTEGRATION.md option B: integration/apply_dropin.py splices the two bodies of integration/dropin_bodies.c into the
upstream smvp-toolkit main-cli.c.  The repository holds no line of that file, so the splice is checked on a stand-in:
a C file with the two functions, taking the parameters the bodies use, and braces hidden in strings, character
literals and comments."""
import importlib.util
import os
import subprocess

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HEAD = r'''#include <stdio.h>
#include <stdlib.h>
#include "mmio/mmio.h"
#define ANSI_COLOR_RED "\x1b[31m"
#define ANSI_COLOR_YELLOW "\x1b[33m"
#define ANSI_COLOR_RESET "\x1b[0m"
typedef struct { int row, col; double val; } MMRawData;
struct _time_data_ { double time_total, time_avg, time_stdev, time_min, time_max; double time_each[]; };
/* double *smvp_csr_compute( in a comment is not a definition */
'''
CSR_SIG = "double *smvp_csr_compute(MMRawData *mmImportData, int fInputRows, int fInputNonZeros, int compiter,\n" \
          "                         struct _time_data_ *csr_time)\n"
CSR_OLD = r'''{
    const char *s = "}{\"}"; /* } */
    char c = '}', d = '\'';
    // }
    (void)mmImportData; (void)fInputRows; (void)fInputNonZeros; (void)compiter; (void)csr_time; (void)s; (void)c; (void)d;
    { return NULL; }
}'''
MID = "\n\nstatic int kept(void) { return '{'; }\n\n"
TJDS_SIG = "double *smvp_tjds_compute(MMRawData *mmImportData, int fInputRows, int fInputColumns, int fInputNonZeros,\n" \
           "                          int compiter, struct _time_data_ *tjds_time)\n"
TJDS_OLD = r'''{
    /* { */
    (void)mmImportData; (void)fInputRows; (void)fInputColumns; (void)fInputNonZeros; (void)compiter; (void)tjds_time;
    return NULL;
}'''
TAIL = "\n\nint main(void) { return kept() == '}'; }\n"


def _apply():
    spec = importlib.util.spec_from_file_location("apply_dropin", os.path.join(REPO, "integration", "apply_dropin.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_splice_replaces_exactly_the_two_bodies_and_compiles(tmp_path):
    mod = _apply()
    src = tmp_path / "main-cli.c"
    src.write_text(HEAD + CSR_SIG + CSR_OLD + MID + TJDS_SIG + TJDS_OLD + TAIL)
    out = mod.splice(str(src), str(tmp_path / "main-cli.dropin.c"))
    text = open(out).read()
    inc = '\n#include "smvp_cuda.h" /* smvp_coo has the layout of MMRawData (main-cli.c:42-47) */'
    assert '#include "mmio/mmio.h"' + inc + "\n" in text
    want = (HEAD + CSR_SIG + mod.new_body("smvp_csr_compute").rstrip("\n") + MID + TJDS_SIG +
            mod.new_body("smvp_tjds_compute").rstrip("\n") + TAIL)
    # everything outside the two bodies is the input's text, plus that one include
    assert text.replace(inc, "", 1) == want
    (tmp_path / "mmio").mkdir()
    (tmp_path / "mmio" / "mmio.h").write_text("")
    r = subprocess.run(["gcc", "-std=gnu11", "-fsyntax-only", "-I" + os.path.join(REPO, "include"), "-I" + str(tmp_path), out],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "smvp_csr_mult(" in text and "smvp_tjds_mult(" in text and "return NULL" not in text
