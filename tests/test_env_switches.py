"""CPU checks of the environment switches of libsmvp_cuda (no build needed): the library reads the environment only
through the helpers in csrc/api.cu, the INTEGRATION.md table lists exactly the switches it reads, and the tuning
switches retired with their kernel instantiations stay gone."""
import os
import re

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(REPO, "smvp-toolkit_b200", "csrc")
HELPERS = ("env_str", "env_set", "env_int", "env_tristate")
HELPER_CALL = re.compile(r"\b(%s)\(\s*([^)\s,]*)" % "|".join(HELPERS))

# compile-time switches, tuning hooks and configuration tables that selected swept kernel variants, and the plan-level
# and host-side switches that selected a losing or neutral arm; the measurements that retired them are in DESIGN.md
# §5.2 / §5.3 / §5.4 / §6
REMOVED = ("SMVP_ASM_LDS", "SMVP_SCAN_EXIT", "SMVP_UNIFORM_TILES", "SMVP_X_EVICT_LAST", "SMVP_TJDS_STREAM", "SMVP_MERGE_CFG",
           "SMVP_WMERGE_CFGS", "SMVP_PATTERN_CFG", "SMVP_PATTERN_CFGS", "SMVP_VECTOR_WIDE", "SMVP_TJDS_DET_CFG",
           "SMVP_TJDS_UNROLL", "SMVP_MERGE_CHUNK", "SMVP_MERGE_ALIGNED", "SMVP_PHASED_PLAIN", "SMVP_CUDA_LIB",
           "SMVP_CSR_SPLIT", "SMVP_L2_PERSIST_MB", "SMVP_RANKED_HINTS", "SMVP_HOT_L1", "SMVP_HOT_L2", "SMVP_PIPE_PROFILE",
           "SMVP_PIPE_STREAMS", "SMVP_PIPE_RANGES", "SMVP_PIPE_XCHUNKS")


def _sources():
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".h")):
            yield f, open(os.path.join(CSRC, f)).read()


def _code(text):
    """text without its comments"""
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return re.sub(r"//[^\n]*", "", text)


def test_getenv_only_inside_the_helpers():
    helper_def = re.compile(r"\b(%s)\(const char \*name[^)]*\)\s*\{[^{}]*\}" % "|".join(HELPERS))
    found = []
    for f, text in _sources():
        code = _code(text)
        if f == "api.cu":
            assert len(helper_def.findall(code)) == len(HELPERS), "the env helpers are defined in api.cu"
            code = helper_def.sub("", code)
        found += ["%s: %d" % (f, code[:m.start()].count("\n") + 1) for m in re.finditer(r"\bgetenv\s*\(", code)]
    assert not found, "getenv outside the env helpers of api.cu: %s" % found


def _switches_read():
    names = set()
    for f, text in _sources():
        for helper, arg in HELPER_CALL.findall(_code(text)):
            if arg.startswith('"'):
                names.add(arg.strip('"'))
            else:  # only the helpers themselves pass a name on
                assert f in ("api.cu", "common.cuh"), (f, helper, arg)
    return names


def _switches_documented():
    names = set()
    for line in open(os.path.join(REPO, "INTEGRATION.md")):
        cells = [c.strip() for c in re.split(r"(?<!\\)\|", line)[1:-1]]
        if len(cells) >= 2 and "libsmvp_cuda" in cells[1]:
            names |= set(re.findall(r"SMVP_[A-Z0-9_]+", cells[0]))
    return names


def test_table_lists_exactly_the_switches_read():
    read, documented = _switches_read(), _switches_documented()
    assert read, "no env helper calls found"
    assert read == documented, {"read, not in INTEGRATION.md": sorted(read - documented),
                                "in INTEGRATION.md, never read": sorted(documented - read)}


def test_removed_switches_stay_removed():
    pattern = re.compile(r"\b(%s)\b" % "|".join(REMOVED))
    me = os.path.abspath(__file__)
    hits = []
    for top in ("smvp-toolkit_b200", "tests", "tools"):
        for root, dirs, files in os.walk(os.path.join(REPO, top)):
            dirs[:] = [d for d in dirs if d not in ("lib", "__pycache__", "golden")]
            for f in files:
                path = os.path.join(root, f)
                if path == me:
                    continue
                try:
                    text = open(path, encoding="utf-8").read()
                except (UnicodeDecodeError, OSError):
                    continue
                hits += ["%s: %s" % (os.path.relpath(path, REPO), m) for m in sorted(set(pattern.findall(text)))]
    assert not hits, hits
