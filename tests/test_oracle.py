"""CPU: pin the oracle port (oracle/llama_port.py) to outputs of the UNMODIFIED reference.

tests/golden/*.npz were produced by oracle/make_golden.py from
accessory/model/LLM/{llama,mixtral}.py (imported byte-for-byte); on the host that wrote them the port
matched the live reference bit for bit in fp16 and fp32.
"""
import os

import numpy as np
import pytest
import torch

from oracle import cases, omniquant, weights
from oracle.make_golden import sd_digest
from oracle.llama_port import PortModel

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _gold(name):
    return np.load(os.path.join(GOLD, f"{name}.npz"))


# The reference's fp32 CPU run is reproducible across hosts to a few ulps (same torch build); its fp16 run is NOT: oneDNN picks the
# fp16 GEMM kernel by host ISA (avx512_fp16 / amx hosts accumulate differently from avx512f-only hosts), and two build
# containers of this repo differed by one fp16 ulp of a logit (1.95e-3 in [2, 4)).  So the committed fp16 vectors are
# compared within FP16_HOST_TOL here and within one fp16 ulp per logit in test_port_equals_reference_bits.
FP16_HOST_TOL = 4e-3
# fp32 is not bit for bit across hosts either: the CPU of a B200 host reproduced mixtral_w4 to 3.0e-7 (little more than one
# ulp of its largest logit, 2.19) and the other cases bit for bit.
FP32_HOST_ULPS = 8


@pytest.mark.parametrize("name", list(cases.CASES))
def test_port_matches_reference_golden(name):
    g = _gold(name)
    for dt, tag, tol in ((torch.float32, "fp32", 2e-5), (torch.float16, "fp16", FP16_HOST_TOL)):
        got = cases.port_logits(name, dtype=dt).numpy()
        ref = g[f"logits_{tag}"]
        assert got.shape == ref.shape
        # fp32: bit for bit on every host seen so far (same torch build); the BLAS kernel choice is nevertheless the host's,
        # so the assertion is a tolerance two orders below the fp16 effects under test -- the bit-for-bit pin is
        # test_port_equals_reference_bits
        assert np.abs(got - ref).max() <= tol, (name, tag, np.abs(got - ref).max())
        if tag == "fp32":
            assert (got.argmax(-1) == ref.argmax(-1)).all()


@pytest.mark.parametrize("name", list(cases.CASES))
def test_port_equals_reference_bits(name):
    """The pin: the port reproduces the stored logits of the UNMODIFIED reference modules to within FP32_HOST_ULPS fp32 ulps
    of the largest logit, and in fp16 to within one fp16 ulp of every logit (the host's GEMM kernels decide those last
    bits, see FP16_HOST_TOL; on the host that wrote the fixtures port and reference agreed bit for bit in both)."""
    g = _gold(name)
    port32, ref32 = cases.port_logits(name, dtype=torch.float32).numpy(), g["logits_fp32"]
    tol32 = FP32_HOST_ULPS * np.spacing(np.abs(ref32).max())
    assert np.abs(port32 - ref32).max() <= tol32, (name, np.abs(port32 - ref32).max(), tol32)
    port16 = cases.port_logits(name, dtype=torch.float16).numpy()
    ref16 = g["logits_fp16"]
    ulp = np.spacing(np.abs(ref16).astype(np.float16)).astype(np.float32)
    assert (np.abs(port16 - ref16) <= ulp).all(), (name, np.abs(port16 - ref16).max())


@pytest.mark.parametrize("name", list(cases.CASES))
def test_reference_golden_was_made_from_the_case_inputs(name):
    """The stored reference logits belong to the inputs cases.build_case draws today: same fake-quantised weights
    (sha256), same tokens, same prefill / decode schedule."""
    kind, args, bits, gs, bsz, plen, ndec = cases.CASES[name]
    kind, args, sd, sd_ref, recs, toks = cases.build_case(name)
    g = _gold(name)
    assert str(g["weights_sha256"]) == sd_digest(sd_ref)
    assert np.array_equal(g["tokens"], toks.numpy())
    assert (int(g["prefill_len"]), int(g["n_decode"])) == (plen, ndec)
    assert g["logits_fp32"].shape == g["logits_fp16"].shape == (ndec + 1, bsz, args["vocab_size"])


@pytest.mark.parametrize("bits,gs", [(4, 0), (4, 128), (3, 128), (2, 64)])
def test_quantiser_contract(bits, gs):
    """w_hat == fp16(fp16(q - z) * s16), q in range, group extremes hit the end codes."""
    g = torch.Generator().manual_seed(7)
    w = ((torch.rand(48, 512, generator=g) * 2 - 1) / 16).half()
    r = omniquant.quantize_weight(w, bits, gs)
    q, s, z = r["q"], r["scale"], r["zero"]
    assert q.dtype == torch.uint8 and int(q.max()) <= 2 ** bits - 1
    assert torch.equal(omniquant.dequantize(q, s, z, r["group_size"]), r["w_hat"])
    G = 512 // r["group_size"]
    qg = q.reshape(48, G, -1)
    assert (qg.amin(-1) == 0).all() and (qg.amax(-1) == 2 ** bits - 1).all()
    err = (r["w_hat"].float() - w.float()).abs().reshape(48, G, -1).amax(-1)
    assert (err <= 0.5 * s.float() * 1.01 + 1e-6).all()


@pytest.mark.parametrize("name,tp", [("llama_w4", 2), ("mixtral_w4", 2), ("mixtral_fp16", 2)])
def test_port_tensor_parallel_algebra(name, tp):
    """Sharding per tensor_parallel.py:34-38 / mixtral.py:237 and summing partials == TP=1 up to fp16 rounding."""
    a = cases.port_logits(name, dtype=torch.float32, tp=1)
    b = cases.port_logits(name, dtype=torch.float32, tp=tp)
    assert (a - b).abs().max() < 2e-5
    assert (a.argmax(-1) == b.argmax(-1)).all()


def test_incremental_equals_full_prefill():
    """SURVEY.md Appendix A.7: KV-cache decode == full causal forward (fp32)."""
    kind, args, sd, sd_ref, recs, toks = cases.build_case("llama_w4")
    m = PortModel(kind, args, sd_ref, dtype=torch.float32)
    full = m.forward_inference(toks[:, :8], 0)
    m2 = PortModel(kind, args, sd_ref, dtype=torch.float32)
    m2.forward_inference(toks[:, :5], 0)
    for j in range(5, 8):
        inc = m2.forward_inference(toks[:, j:j + 1], j)
    assert (full - inc).abs().max() < 1e-5


def test_shard_shapes():
    sd = weights.llama_state_dict(cases.TINY_LLAMA)
    s0 = weights.shard_state_dict(sd, 0, 2)
    assert s0["layers.0.attention.wq.weight"].shape == (256, 512)
    assert s0["layers.0.attention.wo.weight"].shape == (512, 256)
    assert s0["tok_embeddings.weight"].shape == (1024, 256)
    assert s0["output.weight"].shape == (512, 512)
    assert s0["norm.weight"].shape == (512,)
