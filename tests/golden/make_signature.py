"""Extract the parameter lists of PyramidCorrelationView's constructor and of pyramid_correlate() from the reference header
(Stereo/CorrelationView.h:48-69, :195-218) into tests/golden/pyramid_correlate_signature.json -- the fixture
tests/test_cpp_shim.py compares the shim with.

  python tests/golden/make_signature.py <Vision Workbench source tree>/src/vw/Stereo/CorrelationView.h"""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def split_params(txt):
    out, depth, cur = [], 0, ""
    for ch in txt:
        if ch in "<(":
            depth += 1
        elif ch in ">)":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur)
            cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur)
    res = []
    for p in out:
        p = " ".join(p.split())
        default = None
        if "=" in p:
            p, default = [s.strip() for s in p.split("=", 1)]
            default = default.replace(" ", "")
        m = re.match(r"(.*?)([A-Za-z_][A-Za-z0-9_]*)$", p)
        typ = m.group(1).strip().replace(" ", "").replace("stereo::", "")
        res.append({"type": typ, "name": m.group(2), "default": default})
    return res


def param_list(src, opener):
    i = src.index(opener) + len(opener)
    depth, j = 1, i
    while depth:
        depth += {"(": 1, ")": -1}.get(src[j], 0)
        j += 1
    return split_params(src[i:j - 1])


def extract(header_text):
    return {"constructor": param_list(header_text, "PyramidCorrelationView("),
            "factory": param_list(header_text, "pyramid_correlate(")}


if __name__ == "__main__":
    sig = extract(open(sys.argv[1]).read())
    json.dump(sig, open(os.path.join(HERE, "pyramid_correlate_signature.json"), "w"), indent=1)
    print(len(sig["constructor"]), len(sig["factory"]))
