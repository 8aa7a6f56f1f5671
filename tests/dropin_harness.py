"""TEST INFRASTRUCTURE -- the synthetic dataset and calling pattern of the reference's driver, `build_vlads` of
scripts/dino_v2_vlad.py (extract loop :164-188, vocabulary :195-213, database / query VLADs :219-264).

`run_driver` restates that calling pattern against any module with the reference's `utilities` API; the tests drive
this repo's drop-in shim (anyloc_b200/dropin/utilities.py) with it and compare against vectors committed from the
reference's own run.  `load_script` imports the unmodified script itself, with a chosen module answering
`from utilities import ...`; only tests/golden/make_golden.py uses it, where the reference tree is present.
Third-party modules the script imports but never uses on this path (natsort, matplotlib, faiss in the dataset
loaders) are stubbed.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

from oracle import reference_import as ri

SCRIPT = os.path.join(ri.REFERENCE_ROOT, "scripts", "dino_v2_vlad.py")


MODEL, LAYER, K = "dinov2_vits14", 2, 4


def hub_model(name):
    """the hub model the driver runs are made with: restated, 3 blocks, perturbed weights"""
    from oracle import dinov2_restated as dr
    return dr.perturb(dr.build(name, seed=0, depth_override=LAYER + 1), seed=3)


def cache_subdir(cache_root, model=MODEL, layer=LAYER, facet="value", clusters=K):
    """where the driver's --cache-vlad-descs puts one configuration's vocabulary and per-image files"""
    return f"{cache_root}/vlad_descs/Dino/17places/{model}-{facet}-L{layer}-C{clusters}"


def residual_api_inputs():
    """-> x [2, 40, 64], centres [5, 64] of the VLAD.generate_multi_res_vec comparison"""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 40, 64, generator=g)
    return x, 0.7 * torch.nn.functional.normalize(torch.randn(5, 64, generator=g), dim=1)


class SyntheticVprDataset:
    """What build_vlads needs from a BaseDataset (dvgl_benchmark/datasets_ws.py:222-239): `database_num`, `len()`,
    `ds[i][0]` = normalised image tensor [3,h,w], `get_image_relpaths(indices)`, `soft_positives_per_query`."""

    def __init__(self, n_db=6, n_qu=3, h=60, w=75, seed=5):
        g = torch.Generator().manual_seed(seed)
        self.database_num, self.queries_num = n_db, n_qu
        db = torch.randn(n_db, 3, h, w, generator=g)
        qu = db[:n_qu] + 0.05 * torch.randn(n_qu, 3, h, w, generator=g)       # query i shows database place i
        self.images = torch.cat([db, qu])
        self.soft_positives_per_query = np.empty(n_qu, dtype=object)
        for i in range(n_qu):
            self.soft_positives_per_query[i] = np.array([i])

    def __len__(self):
        return self.images.shape[0]

    def __getitem__(self, i):
        return self.images[i], i

    def get_image_relpaths(self, i):
        if isinstance(i, (int, np.integer)):
            return f"synth/img_{int(i):04d}.jpg"
        return [f"synth/img_{int(k):04d}.jpg" for k in i]


def load_script(utilities_module):
    """Imports scripts/dino_v2_vlad.py (unmodified) with `utilities` resolving to `utilities_module`."""
    ri._install_stubs()
    if "natsort" not in sys.modules:
        ns = types.ModuleType("natsort")
        ns.natsorted = sorted
        sys.modules["natsort"] = ns
    if ri.REFERENCE_ROOT not in sys.path:
        sys.path.append(ri.REFERENCE_ROOT)
    old = sys.modules.get("utilities")
    sys.modules["utilities"] = utilities_module
    # the dataset loaders do `from utilities import CustomDataset` at import time: drop cached copies bound to another module
    for name in [m for m in sys.modules if m.startswith("custom_datasets") or m.startswith("dvgl_benchmark")]:
        del sys.modules[name]
    try:
        spec = importlib.util.spec_from_file_location("_ref_dino_v2_vlad_" + utilities_module.__name__.replace(".", "_"), SCRIPT)
        mod = importlib.util.module_from_spec(spec)
        st = (np.random.get_state(), torch.random.get_rng_state())
        spec.loader.exec_module(mod)
        np.random.set_state(st[0]); torch.random.set_rng_state(st[1])
    finally:
        if old is not None:
            sys.modules["utilities"] = old
        else:
            sys.modules.pop("utilities", None)
    return mod


def run_driver(utilities_module, ds, cache_root, model=MODEL, layer=LAYER, facet="value", clusters=K, cache=False,
               soft=False, device="cpu"):
    """The driver's calling pattern, restated: batch-1 centre-cropped images through DinoV2ExtractFeatures with
    `.cpu()` per image; the vocabulary from a complete cache (`fit(None)`) or fitted on the database features;
    database then query VLADs via `generate_multi`, from `[None] * n` when the cache holds every image.
    -> (db_vlads, qu_vlads)"""
    u = utilities_module
    vlad = u.VLAD(clusters, None, vlad_mode="soft" if soft else "hard", soft_temp=1.0,
                  cache_dir=cache_subdir(cache_root, model, layer, facet, clusters) if cache else None)
    dino = u.DinoV2ExtractFeatures(model, layer, facet, device=device)

    def extract(indices):
        descs = []
        for i in indices:
            img = ds[i][0].to(device)
            h, w = (img.shape[1] // 14) * 14, (img.shape[2] // 14) * 14
            top, left = int(round((img.shape[1] - h) / 2.0)), int(round((img.shape[2] - w) / 2.0))  # T.CenterCrop
            descs.append(dino(img[:, top:top + h, left:left + w][None]).cpu())
        return torch.cat(descs, dim=0)

    num_db = ds.database_num
    if vlad.can_use_cache_vlad():
        vlad.fit(None)
    else:
        full = extract(np.arange(num_db))
        vlad.fit(full.reshape(-1, full.shape[2]))

    def vlads(indices):
        names = ds.get_image_relpaths(indices)
        if vlad.can_use_cache_ids(names):
            return vlad.generate_multi([None] * len(indices), names)
        return vlad.generate_multi(extract(indices), names)
    return vlads(np.arange(num_db)), vlads(np.arange(num_db, len(ds)))


def make_largs(mod, cache_dir, model="dinov2_vits14", layer=2, facet="value", clusters=4, cache=False, soft=False):
    prog = type(mod.LocalArgs().prog)(cache_dir=cache_dir, vg_dataset_name="17places", use_wandb=False)
    return mod.LocalArgs(prog=prog, model_type=model, desc_layer=layer, desc_facet=facet, num_clusters=clusters,
                         cache_vlad_descs=cache, vlad_assignment="soft" if soft else "hard")
