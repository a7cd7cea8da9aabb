"""Generates tests/golden/flava_golden.pt by running the UNMODIFIED reference `flava_model` (a TorchMultimodal checkout,
given as the argument) on the cases of tests/flava_cases.py.

    python tests/golden/make_flava_golden.py <path to the TorchMultimodal checkout>

Stored per case: the inputs, a parameter checksum (weights are re-created from seeds by the tests) and every output of
`FLAVAModel.forward(image, text, image_patches_mask, text_masked, skip_unmasked_mm_encoder=False)` in fp32, sequence
outputs at the token positions of `flava_cases.golden_view`.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle", "iopath_shim"))
sys.path.insert(0, os.path.abspath(sys.argv[1]))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from torchmultimodal.models.flava.model import flava_model  # noqa: E402

import flava_cases as FC  # noqa: E402


def main():
    torch.set_num_threads(8)
    out = {}
    for name in FC.CASES:
        m = FC.build(flava_model, name)
        inp = FC.inputs(name)
        with torch.no_grad():
            o = m(image=inp["image"], text=inp["text"], image_patches_mask=inp["image_patches_mask"],
                  text_masked=inp["text_masked"], skip_unmasked_mm_encoder=False)
        out[name] = {"inputs": inp, "param_checksum": FC.param_checksum(m),
                     "outputs": {k: FC.golden_view(v) for k, v in FC.flatten_output(o).items()}}
        print(name, {k: tuple(v.shape) for k, v in out[name]["outputs"].items() if "hidden_states" not in k})
    path = os.path.join(HERE, "flava_golden.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path) / 1e6, "MB")


if __name__ == "__main__":
    main()
