"""Generates tests/golden/dino_v1.npz by running the REFERENCE'S OWN ViTExtractor
(/root/reference/dino_extractor.py, imported verbatim through oracle/dino_v1_reference.py) over the
restated DINOv1 model (oracle/dino_v1_restated.py, perturbed seeded weights) on the seeded images of
tests/dino_v1_cases.py.  Run in the build container only:

    python tests/golden/make_golden_dino_v1.py

Per case: the four facets at layers 11 and 5, `include_cls`, and bin=True for token and key (layer 11),
all stored as digests (tests/util.py: shape, sums and seeded samples; 512 samples for the layer-11 key
descriptors, 64 otherwise), which keeps the file small.  Also the reference's `_log_bin` alone on random
maps of the grids in LOG_BIN_GRIDS (stored in full: at most 35 x 136 values)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import dino_v1_reference as r1          # noqa: E402
from tests import dino_v1_cases as cases            # noqa: E402
from tests.util import digest                       # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    mod = r1.load_reference_dino_extractor()
    z = {}
    with torch.no_grad():
        for tag, (name, stride, H, W, B) in cases.CASES.items():
            ext = mod.ViTExtractor(name, stride, model=cases.model_for(name), device="cpu")
            img = cases.image_for(tag)
            for layer in cases.LAYERS:
                for facet in cases.FACETS:
                    out = ext.extract_descriptors(img, layer, facet).numpy()
                    # the d1 facet (layer-11 key) is pinned at 512 sampled entries, the others at 64
                    n = 512 if (layer, facet) == (11, "key") else 64
                    for k, v in digest(out, n).items():
                        z[f"{tag}/L{layer}_{facet}_{k}"] = v
            z[f"{tag}/num_patches"] = np.array(ext.num_patches)
            z[f"{tag}/load_size"] = np.array(ext.load_size)
            for k, v in digest(ext.extract_descriptors(img, 11, "value", include_cls=True).numpy()).items():
                z[f"{tag}/L11_value_cls_{k}"] = v
            for facet in ("token", "key"):
                for k, v in digest(ext.extract_descriptors(img, 11, facet, bin=True).numpy()).items():
                    z[f"{tag}/L11_{facet}_bin_{k}"] = v
        ext = mod.ViTExtractor("dino_vits8", 8, model=cases.model_for("dino_vits8"), device="cpu")
        for gh, gw in cases.LOG_BIN_GRIDS:
            x = cases.log_bin_input(gh, gw)
            ext.num_patches = (gh, gw)
            # _log_bin takes the [B,h,t,d] hook layout; [B,1,t,C] is the token facet's
            z[f"logbin_{gh}x{gw}/out"] = ext._log_bin(x.unsqueeze(1)).squeeze(1).numpy()
    path = os.path.join(OUT, "dino_v1.npz")
    np.savez_compressed(path, **z)
    print(f"{path}: {os.path.getsize(path) / 1e6:.2f} MB, {len(z)} arrays")


if __name__ == "__main__":
    main()
