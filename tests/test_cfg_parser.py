"""CPU: D1 -- the product's cfg parser (models/dark_net.py) against the reference's own ``parse_model_config``
(src/models/dark_net.py:243-261), on the synthetic 79-block trunk cfg and on a cfg with comments, blank lines and
fringe whitespace.  tests/golden/cfg_parser_golden.json stores both cfg texts with the module-definition lists the
reference parser returns for them (values stay strings, ``batch_normalize`` defaults to the int 0)."""
import json
import os
import tempfile

TRICKY = """# leading comment
[net]
channels=3
height = 416

[convolutional]
batch_normalize=1
filters=32
size=3
stride=1
pad=1
activation=leaky
# a comment between blocks
[convolutional]
filters = 64
size=3
stride=2
pad=1
activation=leaky

[shortcut]
from=-2
activation=linear
[yolo]
mask = 0,1,2
anchors = 10,13,  16,30
"""


def _parse(text):
    from avdn_b200.models.dark_net import parse_model_config
    with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
        f.write(text)
    try:
        return parse_model_config(f.name)
    finally:
        os.unlink(f.name)


def test_parse_model_config_matches_reference(built_lib, golden_dir):
    from avdn_b200.utils import synthetic
    with open(os.path.join(golden_dir, "cfg_parser_golden.json")) as f:
        golden = json.load(f)
    assert golden["tricky"]["text"] == TRICKY
    for case in ("trunk", "tricky"):
        assert _parse(golden[case]["text"]) == golden[case]["module_defs"], case
    # the synthetic cfg is the truncated-79 trunk: [net] + 80 blocks (57 convolutions, 23 shortcuts)
    defs = _parse(synthetic.yolov3_trunk_cfg())
    kinds = [d["type"] for d in defs]
    assert kinds[0] == "net" and kinds.count("convolutional") == 57 and kinds.count("shortcut") == 23
