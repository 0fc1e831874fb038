"""Every entry point of the C-ABI (include/dreamlab_b200.h) is exercised by name in the suite.

A kernel reached only through whole pipelines is judged at the pipelines' bars (2e-2, a PSNR, a
golden), where an edge row, a tail element or a rounding step can be wrong unnoticed.  So each
exported `dl_*` function must be named in some tests/test_*.py, either through its binding
(`lib.<name>(`) or as `dl_<name>` (the fp32 entry points are reached through the dtype-dispatching
bindings, and the test that calls them names them).  The allowlist holds only queries and
diagnostics, which launch no arithmetic of their own."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "dreamlab_b200.h")

ALLOWLIST = {
    "dl_abi_version": "constant query, no launch",
    "dl_last_error": "returns the text of the last failure, no launch",
    "dl_device_sm_count": "device attribute query, no launch",
    "dl_debug_attention_trace": "debug aid: switches clock-stamp tracing on or off",
    "dl_fill_identity": "fills the constant identity operand that every residual igemm test uses",
    "dl_igemm_plan_bn": "host-only tile plan query, used by lib.igemm(row_stats=True)",
    "dl_groupnorm_workspace_bytes": "workspace size query, no launch",
    "dl_groupnorm_split_workspace_bytes": "workspace size query, no launch",
    "dl_png_stored_workspace_bytes": "workspace size query, no launch",
}


def header_entry_points():
    """Names of the functions declared in the header (a declaration starts a line with its return type)."""
    text = open(HEADER).read()
    return sorted(set(re.findall(r"^(?:const\s+)?(?:int|size_t|long long|char\s*\*|void)\s*\*?\s*(dl_\w+)\s*\(",
                                 text, re.M)))


def test_header_parses():
    names = header_entry_points()
    # a few landmarks of each group, so that a parser that silently matches nothing cannot pass
    for n in ("dl_abi_version", "dl_last_error", "dl_igemm", "dl_igemm_f32", "dl_attention", "dl_conv_tapsum",
              "dl_png_stored_size", "dl_groupnorm_workspace_bytes"):
        assert n in names, n
    assert len(names) >= 40, names


def test_allowlist_is_current():
    stale = sorted(set(ALLOWLIST) - set(header_entry_points()))
    assert not stale, f"allowlisted names no longer in the header: {stale}"


def test_every_entry_point_is_named_in_a_test():
    here = os.path.abspath(__file__)
    texts = [open(f).read() for f in sorted(glob.glob(os.path.join(ROOT, "tests", "test_*.py")))
             if os.path.abspath(f) != here]
    corpus = "\n".join(texts)
    missing = []
    for name in header_entry_points():
        if name in ALLOWLIST:
            continue
        short = name[len("dl_"):]
        if re.search(r"\blib\." + re.escape(short) + r"\(", corpus) or re.search(r"\b" + re.escape(name) + r"\b",
                                                                                  corpus):
            continue
        missing.append(name)
    assert not missing, f"C-ABI entry points with no test naming them: {missing}"
