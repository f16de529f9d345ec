"""ORACLE TEST INFRASTRUCTURE: what the UNMODIFIED MetaModel (accessory/model/meta.py) returns when it is constructed with
``llama_type="llama_b200"`` and drives this package's engine through its own generate() / stream_generate().

Needs a GPU and the reference tree (see oracle/ref_import.py).  The modules meta.py imports but this path never touches
(util.misc / util.tensor_parallel / model.tokenizer) are stubbed; the tokenizer is the toy whitespace tokenizer of
tests/golden/generate.json; the weights are the seeded tiny LLaMA of oracle.cases.  Recorded for wbits = 4: the greedy
texts, the texts with eos set to row 0's third token, with a two-token stop symbol, the stream of one prompt and that
prompt's batch text; for wbits = 16: the greedy texts.  tests/test_metamodel_gpu.py runs the package's statement of the loop
(generation.generate / stream_generate) over the same engine and compares with this record.

    python -m oracle.make_golden_metamodel [OUT]   ->  tests/golden/metamodel_generate.json
"""
import importlib
import json
import os
import sys
import tempfile
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import llama2_accessory_b200 as pkg  # noqa: E402
from llama2_accessory_b200.model import llama_b200  # noqa: E402
from oracle import cases, ref_import  # noqa: E402
from oracle.toy_tokenizer import ToyTokenizer  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "metamodel_generate.json")
PROMPTS = ["the quick brown fox", "hello world", "a b c d e f g"]


class _PathTokenizer(ToyTokenizer):
    """accessory/model/tokenizer.py::Tokenizer(model_path=...) stand-in: 'toy:<n_words>:<eos_id>'."""

    def __init__(self, model_path):
        _, n, eos = model_path.split(":")
        super().__init__(int(n), int(eos))


def _import_meta():
    ref_import.load("llama")  # registers the accessory namespace packages + the fairscale shim
    stubs = (("accessory.util.misc", {"mark_mp_params": lambda model: None}),
             ("accessory.util.tensor_parallel", {}),
             ("accessory.model.tokenizer", {"Tokenizer": _PathTokenizer, "probe_tokenizer_path_from_pretrained": None}))
    for name, attrs in stubs:
        m = sys.modules.get(name)
        if m is None:
            m = types.ModuleType(name)
            sys.modules[name] = m
            parent, leaf = name.rsplit(".", 1)
            setattr(sys.modules[parent], leaf, m)
        for k, v in attrs.items():
            setattr(m, k, v)
    # the two-line plug-in file of INTEGRATION.md section 3 (accessory/model/LLM/llama_b200.py), registered in memory
    plug = types.ModuleType("accessory.model.LLM.llama_b200")
    plug.ModelArgs, plug.Transformer = llama_b200.ModelArgs, llama_b200.Transformer
    sys.modules["accessory.model.LLM.llama_b200"] = plug
    meta = importlib.import_module("accessory.model.meta")
    meta.Tokenizer = _PathTokenizer
    return meta


def _metamodel(meta, tmp, wbits, eos_id=2):
    args = dict(cases.TINY_LLAMA)
    cfg = {k: v for k, v in args.items() if k not in ("vocab_size", "max_seq_len", "max_batch_size")}
    cfg["wbits"] = wbits
    p = os.path.join(tmp, f"config_w{wbits}.json")
    with open(p, "w") as f:
        json.dump(cfg, f)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float16)
    try:
        with torch.device("cuda"):
            model = meta.MetaModel("llama_b200", p, f"toy:{args['vocab_size']}:{eos_id}", with_visual=False,
                                   max_seq_len=args["max_seq_len"])
    finally:
        torch.set_default_dtype(old)
    sd = cases.master_state_dict("llama", args)
    missing, unexpected = model.load_state_dict({"llma." + k: v.cuda() for k, v in sd.items()}, strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    return model.eval()


def main(out_path=OUT):
    assert torch.cuda.is_available() and ref_import.available(), "needs a GPU and the reference tree"
    pkg.build()
    meta = _import_meta()
    out = {"model": "TINY_LLAMA (oracle.cases, seed 0), MetaModel('llama_b200') on cuda:0", "prompts": PROMPTS}
    with tempfile.TemporaryDirectory() as tmp:
        model = _metamodel(meta, tmp, wbits=4)
        texts = model.generate(list(PROMPTS), max_gen_len=6)
        row0 = [int(w[1:]) for w in texts[0].split()]
        model.tokenizer.eos_id = row0[2]
        cut = model.generate(list(PROMPTS), max_gen_len=6)
        model.tokenizer.eos_id = 2
        stops = [f"w{row0[1]} w{row0[2]}"]
        stop = model.generate(list(PROMPTS), max_gen_len=6, additional_stop_symbols=tuple(stops))
        stream = list(model.stream_generate(PROMPTS[0], max_gen_len=5))
        single = model.generate([PROMPTS[0]], max_gen_len=5)
        out["w4"] = {"greedy": texts, "eos_id_cut": row0[2], "eos_cut": cut, "stop_symbols": stops, "stop": stop,
                     "stream_prompt0": stream, "single_prompt0": single}
        del model
        model = _metamodel(meta, tmp, wbits=16)
        out["w16"] = {"greedy": model.generate(list(PROMPTS), max_gen_len=6)}
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", out_path)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main(*sys.argv[1:])
