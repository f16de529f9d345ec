"""CPU: the generate loop (SURVEY.md 8f rank 2) against golden outputs of the UNMODIFIED MetaModel.generate /
stream_generate (tests/golden/generate.json, made by oracle/make_golden_generate.py from accessory/model/meta.py).

The engine's host loop is driven here with the oracle port (fp32, bit-exact to the reference model) as the model and
an injected arg-max as token selection -- on the GPU the same loop selects tokens with b200_argmax / b200_sample_top_p
and the device loop is compared to it (tests/test_zz_generation_gpu.py).
"""
import json
import os
import types

import pytest
import torch

from llama2_accessory_b200 import generation
from oracle import cases
from oracle.llama_port import PortModel
from oracle.toy_tokenizer import ToyTokenizer

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "generate.json")))


@pytest.fixture(scope="module")
def model():
    args = dict(cases.TINY_LLAMA)
    port = PortModel("llama", args, cases.master_state_dict("llama", args), dtype=torch.float32)
    # parameters(): the loop keeps its token buffers where the model's weights are (the CPU), on a GPU host as well
    return types.SimpleNamespace(args=types.SimpleNamespace(max_seq_len=args["max_seq_len"], max_batch_size=args["max_batch_size"]),
                                 forward_inference=port.forward_inference, parameters=lambda: iter(port.sd.values()))


def _argmax(logits, temperature, top_p):
    assert temperature == 0
    return torch.argmax(logits, dim=-1)


@pytest.mark.parametrize("case", GOLD["cases"], ids=[c["name"] for c in GOLD["cases"]])
def test_generate_matches_reference_loop(model, case):
    tok = ToyTokenizer(cases.TINY_LLAMA["vocab_size"], case["eos_id"])
    kw = dict(case["kwargs"])
    prompts = case.get("prompts", GOLD["prompts"])
    got = generation.generate(model, tok, list(prompts), select=_argmax, device_loop=False, **kw)
    assert got == case["texts"]


@pytest.mark.parametrize("case", GOLD["stream_cases"], ids=[c["name"] for c in GOLD["stream_cases"]])
def test_stream_generate_matches_reference_loop(model, case):
    tok = ToyTokenizer(cases.TINY_LLAMA["vocab_size"], case["eos_id"])
    got = list(generation.stream_generate(model, tok, GOLD["prompts"][0], select=_argmax, **case["kwargs"]))
    assert got == case["yields"]


def test_generate_matches_reference_loop_mixtral():
    args = dict(cases.TINY_MIXTRAL)
    port = PortModel("mixtral", args, cases.master_state_dict("mixtral", args), dtype=torch.float32)
    m = types.SimpleNamespace(args=types.SimpleNamespace(max_seq_len=args["max_seq_len"], max_batch_size=args["max_batch_size"]),
                              forward_inference=port.forward_inference, parameters=lambda: iter(port.sd.values()))
    for case in GOLD["mixtral_cases"]:
        tok = ToyTokenizer(args["vocab_size"], case["eos_id"])
        assert generation.generate(m, tok, list(GOLD["prompts"]), select=_argmax, device_loop=False, **case["kwargs"]) == case["texts"]


def test_argument_errors_follow_the_reference(model):
    tok = ToyTokenizer()
    with pytest.raises(ValueError, match="LIST of prompts"):
        generation.generate(model, tok, "a single string", select=_argmax, device_loop=False)
    with pytest.raises(AssertionError):
        generation.generate(model, tok, ["x"] * 5, select=_argmax, device_loop=False)  # max_batch_size 4
    with pytest.raises(NotImplementedError):
        generation.generate(model, tok, ["x"], images=torch.zeros(1, 3, 2, 2), select=_argmax, device_loop=False)
    with pytest.raises(RuntimeError, match="no CPU path"):
        generation.generate(model, tok, ["x"], max_gen_len=2, device_loop=False)  # default selection is GPU-only
