"""Regenerate inceptionv4_reference.json from the original project's Inception-v4 (lzhangbv/dear_pytorch,
dear/inceptionv4.py):

    python tests/golden/make_inceptionv4_reference.py <checkout of lzhangbv/dear_pytorch>/dear/inceptionv4.py

Stores the shapes of its state dict, in order, and its eval-mode logits for the seeded weights and inputs that
tests/test_models.py::test_inceptionv4_matches_the_reference_file gives our model.
"""
import importlib.util
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(HERE), os.path.dirname(os.path.dirname(HERE))]
from test_models import inceptionv4_input, seeded_state_dict  # noqa: E402


def main(path):
    spec = importlib.util.spec_from_file_location("reference_inceptionv4", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    ref = mod.InceptionV4(num_classes=1000).eval()
    sd = ref.state_dict()
    ref.load_state_dict(seeded_state_dict(sd))
    with torch.no_grad():
        logits = ref(inceptionv4_input())
    out = {"source": "lzhangbv/dear_pytorch dear/inceptionv4.py, InceptionV4(num_classes=1000), eval mode, float32 on the CPU",
           "state_dict_shapes": [list(v.shape) for v in sd.values()],
           "logits": logits.tolist()}
    with open(os.path.join(HERE, "inceptionv4_reference.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
