"""Pins the oracle to the UNMODIFIED reference and writes the golden vectors.

Needs a checkout of the reference project (no GPU, no compiled extension):
    python oracle/make_golden.py PATH/TO/flash-cosine-sim-attention

For each case it (1) loads the reference's flash_cosine_sim_attention.py by path (the package
import itself fails without the compiled extension, reference __init__.py:1), (2) runs
`plain_cosine_sim_attention` in float64 with autograd on seeded inputs, (3) asserts that
oracle/cosine_sim_attention_oracle.py reproduces the outputs and all gradients to 1e-9, and
(4) stores inputs + reference outputs in tests/golden/<case>.npz.  Shapes are kept small enough that
every file stays under 1 MB.
TEST INFRASTRUCTURE ONLY.
"""
import contextlib
import importlib.util
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import cosine_sim_attention_oracle as oracle  # noqa: E402

REF_PY = os.path.join("flash_cosine_sim_attention", "flash_cosine_sim_attention.py")     # inside the reference

# name -> (q shape, k/v shape, kwargs, has_mask)
CASES = {
    "c1_noncausal_f32": dict(q=(1, 2, 128, 64), kv=(1, 2, 128, 64), kw=dict()),
    "causal_square": dict(q=(2, 2, 96, 64), kv=(2, 2, 96, 64), kw=dict(causal=True)),
    "causal_cross_40_72": dict(q=(1, 2, 40, 64), kv=(1, 2, 72, 64), kw=dict(causal=True)),
    "causal_cross_72_40": dict(q=(1, 2, 72, 64), kv=(1, 2, 40, 64), kw=dict(causal=True, scale=4)),
    "mask_single_head_kv_groups2": dict(q=(2, 4, 50, 64), kv=(2, 70, 64), kw=dict(groups=2), mask=True),
    "merged_bh_groups4_scale1": dict(q=(6, 33, 64), kv=(6, 33, 64), kw=dict(groups=4, scale=1)),
    "d128_causal_scale10": dict(q=(1, 2, 64, 128), kv=(1, 2, 64, 128), kw=dict(causal=True, scale=10)),
    "no_l2norm": dict(q=(1, 2, 48, 64), kv=(1, 2, 48, 64), kw=dict(l2norm_qk=False, scale=1), small=True),
    # attn_bias (reference tests/test.py:58-61): per head, and with a batch dimension on merged batch-heads
    "bias_heads_causal": dict(q=(2, 2, 80, 64), kv=(2, 2, 80, 64), kw=dict(causal=True), bias=(2, 80, 80)),
    "bias_heads_mask_cross": dict(q=(2, 2, 40, 64), kv=(2, 2, 72, 64), kw=dict(), mask=True, bias=(2, 40, 72)),
    "bias_batch_dim_merged": dict(q=(4, 56, 64), kv=(4, 56, 64), kw=dict(attn_bias_batch_dim=True), bias=(4, 56, 56)),
}


def load_reference(ref_root):
    spec = importlib.util.spec_from_file_location("ref_fcsa", os.path.join(ref_root, REF_PY))
    mod = importlib.util.module_from_spec(spec)
    with contextlib.redirect_stdout(io.StringIO()):   # it prints a "not compiled" hint
        spec.loader.exec_module(mod)
    return mod


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python oracle/make_golden.py PATH/TO/flash-cosine-sim-attention")
    ref = load_reference(sys.argv[1])
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    for idx, (name, c) in enumerate(CASES.items()):
        g = torch.Generator().manual_seed(1000 + idx)
        amp = 0.2 if c.get("small") else 1.0
        # inputs are bf16-representable so that 16-bit GPU runs consume exactly these values
        r16 = lambda t: t.to(torch.bfloat16).to(torch.float64)
        q = r16(torch.randn(c["q"], generator=g, dtype=torch.float64) * amp).requires_grad_()
        k = r16(torch.randn(c["kv"], generator=g, dtype=torch.float64) * amp).requires_grad_()
        v = r16(torch.randn(c["kv"], generator=g, dtype=torch.float64)).requires_grad_()
        mask = None
        if c.get("mask"):
            mask = torch.rand((c["q"][0], c["kv"][-2]), generator=g) > 0.3
            mask[:, 0] = True   # no fully-masked rows (plain and fused differ there by design)
        bias = None
        if c.get("bias"):
            bias = r16(torch.randn(c["bias"], generator=g, dtype=torch.float64)).requires_grad_()
        kw_ref = dict(c["kw"], attn_bias=bias) if bias is not None else c["kw"]
        o = ref.plain_cosine_sim_attention(q, k, v, mask=mask, **kw_ref)
        do = r16(torch.randn(o.shape, generator=g, dtype=torch.float64))
        (o * do).sum().backward()

        args = dict(mask=None if mask is None else mask.numpy(), d_out=do.numpy(), **c["kw"])
        if bias is not None:
            args["attn_bias"] = bias.detach().numpy()
        res = oracle.attention(q.detach().numpy(), k.detach().numpy(), v.detach().numpy(), **args)
        oo, dq, dk, dv = res[:4]
        errs = [np.abs(oo - o.detach().numpy()).max(), np.abs(dq - q.grad.numpy()).max(),
                np.abs(dk - k.grad.numpy()).max(), np.abs(dv - v.grad.numpy()).max()]
        if bias is not None:
            errs.append(np.abs(res[4] - bias.grad.numpy()).max())
        assert max(errs) < 1e-9, (name, errs)
        np.savez_compressed(
            os.path.join(out_dir, name + ".npz"),
            q=q.detach().numpy().astype(np.float32), k=k.detach().numpy().astype(np.float32),
            v=v.detach().numpy().astype(np.float32), d_out=do.numpy().astype(np.float32),
            mask=np.zeros(0, dtype=bool) if mask is None else mask.numpy(),
            o=o.detach().numpy(), dq=q.grad.numpy(), dk=k.grad.numpy(), dv=v.grad.numpy(),
            kwargs=np.array(repr(c["kw"])),
            **({} if bias is None else dict(attn_bias=bias.detach().numpy().astype(np.float32),
                                            d_bias=bias.grad.numpy())),
        )
        print(f"{name}: oracle vs reference max err fwd/dq/dk/dv(/dbias) = " + " ".join(f"{e:.2e}" for e in errs))


if __name__ == "__main__":
    main()
