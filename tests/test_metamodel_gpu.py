"""GPU: the UNMODIFIED reference `MetaModel` (accessory/model/meta.py) constructed with ``llama_type="llama_b200"`` and
driven through its own ``generate()`` -- the integration level 3 of INTEGRATION.md -- against this package's statement of
that loop over the same engine.

`MetaModel.__init__` (meta.py:20-78) resolves ``accessory.model.LLM.llama_b200``, reads the JSON config into our
``ModelArgs`` (max_batch_size 32, vocab size from the tokenizer) and builds our ``Transformer``; a checkpoint-shaped state
dict is loaded into it; ``MetaModel.generate`` (meta.py:372-468) then calls ``forward_inference`` once per token, every one
of those calls running in libb200decode.so.  What it returned on a B200 is stored in tests/golden/metamodel_generate.json
(oracle/make_golden_metamodel.py); here the same ``Transformer`` is built from the same config, and generation.generate /
stream_generate must return those texts.  The tokenizer is the toy whitespace tokenizer the generate-loop goldens use.
"""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

import llama2_accessory_b200 as pkg  # noqa: E402
from llama2_accessory_b200 import generation  # noqa: E402
from llama2_accessory_b200.model import llama_b200  # noqa: E402
from oracle import cases  # noqa: E402
from oracle.toy_tokenizer import ToyTokenizer  # noqa: E402

GOLD_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLD = os.path.join(GOLD_DIR, "generate.json")
PROMPTS = ["the quick brown fox", "hello world", "a b c d e f g"]


def _meta_gold():
    with open(os.path.join(GOLD_DIR, "metamodel_generate.json")) as f:
        g = json.load(f)
    assert g["prompts"] == PROMPTS
    return g


@pytest.fixture(scope="module", autouse=True)
def _built():
    pkg.build()


def _metamodel(wbits, eos_id=2):
    """The Transformer and tokenizer MetaModel('llama_b200', <config with wbits>, 'toy:<vocab>:<eos>') holds (meta.py:33-56)."""
    args = dict(cases.TINY_LLAMA)
    cfg = {k: v for k, v in args.items() if k not in ("vocab_size", "max_seq_len", "max_batch_size")}
    cfg["wbits"] = wbits
    tok = ToyTokenizer(args["vocab_size"], eos_id)
    margs = llama_b200.ModelArgs(**cfg, max_seq_len=args["max_seq_len"], max_batch_size=32,
                                 vocab_size=tok.n_words)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float16)
    try:
        with torch.device("cuda"):
            model = llama_b200.Transformer(margs, with_visual=False)
    finally:
        torch.set_default_dtype(old)
    assert model.args.max_batch_size == 32
    sd = cases.master_state_dict("llama", args)
    missing, unexpected = model.load_state_dict({k: v.cuda() for k, v in sd.items()}, strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    return model.eval(), tok


def test_generate_reproduces_the_unmodified_metamodel_on_the_b200_engine():
    g = _meta_gold()["w4"]
    model, tok = _metamodel(wbits=4)
    texts = generation.generate(model, tok, list(PROMPTS), max_gen_len=6, device_loop=False)
    assert model.engine is not None and model.engine.cfg.bits == 4  # forward_inference built the packed engine
    assert texts == g["greedy"], (texts, g["greedy"])
    # the loop runs to max(prompt length) + max_gen_len for every row (meta.py:415-433): shorter prompts generate more tokens
    plens = [len(tok.encode(x, bos=True, eos=False)) for x in PROMPTS]
    assert [len(t.split()) for t in texts] == [max(plens) + 6 - n for n in plens], texts
    # same tokens from the device-resident driver of the loop over the same engine
    assert generation.generate(model, tok, list(PROMPTS), max_gen_len=6, device_loop=True) == texts
    # eos / stop-symbol handling of the reference loop over our logits
    row0 = [int(w[1:]) for w in texts[0].split()]
    assert g["eos_id_cut"] == row0[2]
    tok.eos_id = row0[2]
    cut = generation.generate(model, tok, list(PROMPTS), max_gen_len=6, device_loop=False)
    first = row0.index(row0[2])  # the reference stops a row at the FIRST occurrence of eos among its generated tokens
    assert cut == g["eos_cut"] and cut[0] == " ".join(texts[0].split()[:first]), (cut, g["eos_cut"], texts)
    tok.eos_id = 2
    stops = (f"w{row0[1]} w{row0[2]}",)
    assert list(stops) == g["stop_symbols"]
    stop = generation.generate(model, tok, list(PROMPTS), max_gen_len=6, additional_stop_symbols=stops, device_loop=False)
    assert stop == g["stop"], (stop, g["stop"])
    assert len(stop[0].split()) < len(texts[0].split()), (stop, texts)
    ys = list(generation.stream_generate(model, tok, PROMPTS[0], max_gen_len=5))
    assert ys == g["stream_prompt0"], (ys, g["stream_prompt0"])
    single = generation.generate(model, tok, [PROMPTS[0]], max_gen_len=5)
    assert single == g["single_prompt0"] and ys[-1]["end_of_content"] and ys[-1]["text"] == single[0]


def test_metamodel_fp16_engine_against_the_reference_goldens():
    """wbits = 16: the same weights the fp32 goldens of the unmodified reference model were generated from
    (tests/golden/generate.json); fp16 logits can flip a near-tie, so agreement is counted, not demanded token for token.
    The texts are those the unmodified MetaModel returned over the fp16 engine."""
    model, tok = _metamodel(wbits=16)
    texts = generation.generate(model, tok, list(PROMPTS), max_gen_len=6)
    assert texts == _meta_gold()["w16"]["greedy"], texts
    gold = next(c for c in json.load(open(GOLD))["cases"] if c["name"] == "greedy")["texts"]
    first = sum(a.split()[0] == b.split()[0] for a, b in zip(texts, gold))
    n_tok = sum(len(b.split()) for b in gold)
    n_same = sum(x == y for a, b in zip(texts, gold) for x, y in zip(a.split(), b.split()))
    print(f"\n[MetaModel(llama_b200, fp16) vs reference fp32 goldens] first tokens {first}/3, all tokens {n_same}/{n_tok}")
    assert first >= 2 and n_same >= n_tok // 2, (texts, gold)
