"""Every compiled attention kernel variant has a parity case in tests/test_attention_edges_gpu.py.

The variants are read out of the CUDA sources: the `DL_ATTN_ATTR(...)` list of attention.cu and the
`DL_PP_ATTR(...)` list of attention_pp.cu (each instantiation gets its shared-memory attribute there), the
`attn_x_kernel<...>` launches of attention_x.cu and the wide and SIMT kernels.  Each must be named by the case
table (default dispatch) or the knob table (DL_ATTN_* child processes) of the GPU module, whose tables are plain
module data.  So a new template instantiation without a case fails here, without a GPU."""
import importlib.util
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "stable-diffusion-1.5-lcm-onnx-rknn2_b200", "csrc")


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _edges():
    spec = importlib.util.spec_from_file_location(
        "attention_edges_tables", os.path.join(ROOT, "tests", "test_attention_edges_gpu.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _bool(a):
    a = a.strip()
    return {"true": "1", "false": "0"}.get(a, a)


def _template_defaults(src, kernel):
    """Default values of the trailing template parameters of `kernel` (e.g. kPoly = 0)."""
    m = re.search(r"template\s*<([^>]*)>\s*__global__[^\n]*\n?\s*" + kernel + r"\s*\(", src)
    assert m, f"template declaration of {kernel} not found"
    params = [p.strip() for p in m.group(1).split(",")]
    return params, [p.split("=")[1].strip() if "=" in p else None for p in params]


def tc_variants():
    src = _src("attention.cu")
    params, defaults = _template_defaults(src, "attn_tc_kernel")
    attr = set()
    for args in re.findall(r"^\s*DL_ATTN_ATTR\(([^)]*)\);", src, re.M):
        a = [_bool(x) for x in args.split(",")]
        a += defaults[len(a):]
        assert None not in a and len(a) == len(params), (args, params)
        attr.add("attn_tc<" + ",".join(a) + ">")
    launched = set()
    for args in re.findall(r"attn_tc_kernel<([^>]*)><<<", src):
        a = [_bool(x) for x in args.split(",")]
        launched.add("attn_tc<" + ",".join(a + defaults[len(a):]) + ">")
    return attr, launched


def pp_variants():
    src = _src("attention_pp.cu")
    attr = {"attn_pp<" + ",".join(x.strip() for x in args.split(",")) + ">"
            for args in re.findall(r"DL_PP_ATTR\(([^)]*)\);", src)}
    return attr


def x_variants():
    return {f"attn_x<{kt}>" for kt in re.findall(r"attn_x_kernel<(\d+)><<<", _src("attention_x.cu"))}


def plain_variants():
    out = set()
    if re.search(r"attn_wide_kernel<<<", _src("attention_wide.cu")):
        out.add("attn_wide")
    if re.search(r"attn_simt_kernel<<<", _src("attention_simt.cu")):
        out.add("attn_simt")
    return out


def all_variants():
    attr, _ = tc_variants()
    return attr | pp_variants() | x_variants() | plain_variants()


def test_parsers_find_the_landmarks():
    attr, launched = tc_variants()
    # a few known variants of each family, so that a parser that silently matches nothing cannot pass
    for tag in ("attn_tc<1,1,3,128,2>", "attn_tc<1,1,0,0,0>", "attn_tc<0,0,0,0,0>", "attn_tc<1,1,4,128,0>"):
        assert tag in attr, (tag, sorted(attr))
    assert {"attn_pp<3,2,1>", "attn_pp<4,0,2>"} <= pp_variants()
    assert x_variants() == {"attn_x<80>", "attn_x<128>"}
    assert plain_variants() == {"attn_wide", "attn_simt"}
    assert len(attr) >= 9 and len(pp_variants()) >= 12, (sorted(attr), sorted(pp_variants()))


def test_every_launched_tc_variant_gets_its_smem_attribute():
    attr, launched = tc_variants()
    assert len(launched) >= 9, sorted(launched)
    assert launched == attr, f"launched without an attribute: {sorted(launched - attr)}; " \
                             f"attribute for a variant never launched: {sorted(attr - launched)}"


def test_every_variant_has_a_case():
    edges = _edges()
    named = {c["kernel"] for c in edges.CASES}
    for knob in edges.KNOBS:
        named |= {kernel for kernel, _ in knob["cases"].values()}
    missing = sorted(all_variants() - named)
    assert not missing, f"attention kernel variants with no case in test_attention_edges_gpu.py: {missing}"
    stale = sorted(named - all_variants())
    assert not stale, f"cases name kernels the sources no longer compile: {stale}"


def test_tables_name_known_cases_and_tags():
    edges = _edges()
    for knob in edges.KNOBS:
        assert knob["env"] and all(k.startswith("DL_ATTN_") for k in knob["env"]), knob["env"]
        for name, (_, kt) in knob["cases"].items():
            assert name in edges.CASE, name
            assert kt in (32, 64, 80, 96, 128), (name, kt)
    # the profiler's spellings of one name normalise to the tag the tables use
    for raw in ("void dl::attn_tc_kernel<true, true, 3, 128, 2>(dl::AttnParams)",
                "void dl::attn_tc_kernel<(bool)1, (bool)1, (int)3, (int)128, (int)2>(dl::AttnParams)"):
        assert edges.kernel_tag(raw) == "attn_tc<1,1,3,128,2>", raw
    assert edges.kernel_tag("dl::attn_wide_kernel(dl::AttnWParams)") == "attn_wide"
    assert edges.kernel_tag("void dl::attn_x_kernel<(int)80>(dl::AttnXParams)") == "attn_x<80>"
    assert edges.kernel_tag("void dl::igemm_kernel<1>(dl::IgemmParams)") is None
