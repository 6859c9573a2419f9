"""Writes tests/golden/cfg_parser_golden.json from the REFERENCE's own ``parse_model_config``
(src/models/dark_net.py:243-261): the two cfg texts of tests/test_cfg_parser.py (the synthetic 79-block trunk and
a cfg with comments, blank lines and fringe whitespace) with the module-definition lists the reference returns.

    python tests/golden/make_cfg_parser_golden.py <checkout of the original project>   (or AVDN_REFERENCE_DIR)
"""
import importlib.util
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from avdn_b200.utils import synthetic  # noqa: E402
from test_cfg_parser import TRICKY  # noqa: E402


def reference_parser(checkout):
    spec = importlib.util.spec_from_file_location("ref_dark_net", os.path.join(checkout, "src", "models", "dark_net.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.parse_model_config


if __name__ == "__main__":
    checkout = sys.argv[1] if len(sys.argv) > 1 else os.environ["AVDN_REFERENCE_DIR"]
    parse = reference_parser(checkout)
    out = {}
    for case, text in (("trunk", synthetic.yolov3_trunk_cfg()), ("tricky", TRICKY)):
        with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
            f.write(text)
        try:
            out[case] = {"text": text, "module_defs": parse(f.name)}
        finally:
            os.unlink(f.name)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cfg_parser_golden.json")
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print("wrote", path, os.path.getsize(path))
