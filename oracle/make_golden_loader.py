"""ORACLE TEST INFRASTRUCTURE: golden results of the UNMODIFIED tensor-parallel checkpoint loader
(accessory/util/tensor_parallel.py) on the folders checkpoint.save_tensor_parallel_shards writes.

Needs the reference tree (see oracle/ref_import.py).  For the seeded tiny LLaMA saved as two shards in each folder format
it records what the reference loader reports: the inferred (format, model-parallel size), the shard file names, the merged
TP = 1 state dict (dtype, shape and sha256 of every tensor) and the parameter names of the reference Transformer the merged
dict is loaded into; for an empty folder and a folder holding two formats, the exception the loader raises.
tests/test_checkpoint_cpu.py compares the package's loader with this record.

    python -m oracle.make_golden_loader   ->  tests/golden/reference_tp_loader.json
"""
import contextlib
import importlib
import io
import json
import os
import sys
import tempfile

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from llama2_accessory_b200 import checkpoint as ck  # noqa: E402
from oracle import cases, ref_import  # noqa: E402
from oracle.weights import tensor_digest  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_tp_loader.json")
SEED = 3
MP_SIZE = 2


def main():
    assert ref_import.available(), "needs the reference tree"
    ref_import.load("llama")
    tp = importlib.import_module("accessory.util.tensor_parallel")
    args = cases.TINY_LLAMA
    sd = cases.master_state_dict("llama", args, seed=SEED)
    model = ref_import.build_reference_model("llama", dict(args), sd, torch.float16)
    holder = torch.nn.Module()
    holder.llma = model
    out = {"model": f"TINY_LLAMA master weights (oracle.cases, seed {SEED}), {MP_SIZE} shards",
           "model_keys": sorted(holder.state_dict()), "formats": {}, "refused": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for fmt in ("consolidated", "meta_ori"):
            d = os.path.join(tmp, fmt)
            ck.save_tensor_parallel_shards(sd, d, MP_SIZE, fmt)
            with contextlib.redirect_stdout(io.StringIO()):
                ref_sd = tp.load_tensor_parallel_model_state_dict(holder, d, fmt)
            out["formats"][fmt] = {"inferred": list(tp.infer_checkpoint_format_and_mp_size(d)),
                                   "shard_file_names": list(tp.get_tensor_parallel_shards_file_name(fmt, MP_SIZE)),
                                   "merged": {k: tensor_digest(v) for k, v in sorted(ref_sd.items())}}
        for bad in ("empty", "mixed"):
            d = os.path.join(tmp, bad)
            os.makedirs(d)
            if bad == "mixed":
                ck.save_tensor_parallel_shards(sd, d, 1, "consolidated")
                ck.save_tensor_parallel_shards(sd, d, 1, "meta_ori")
            else:
                with open(os.path.join(d, "x.txt"), "w") as f:
                    f.write("x")
            try:
                tp.infer_checkpoint_format_and_mp_size(d)
                out["refused"][bad] = None
            except Exception as e:  # noqa: BLE001 -- the exception type is what is recorded
                out["refused"][bad] = type(e).__name__
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", OUT)


if __name__ == "__main__":
    main()
