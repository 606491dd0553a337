"""Loading of the reference-generated fixtures in tests/golden/ (written by tools/make_golden.py).

sla_a.pt does not store its inputs (they would take the file past 1 MB): q, k, v are drawn again here exactly as
tools/make_golden.py drew them and checked against the int16-bit-pattern checksum stored with the reference's outputs."""
import os

import torch

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
SEED = 20260922   # tools/make_golden.py seeds torch's global generator once, then draws the norm fixtures and then sla_a


def checksum(*tensors):
    return torch.stack([t.view(torch.int16).to(torch.int64).sum() for t in tensors])


def sla_a_inputs():
    g = torch.Generator().manual_seed(SEED)
    for n in (1536, 5120, 256):                    # the norm fixtures' draws come first: x, w, b per size
        torch.randn(32 if n <= 512 else 6, n, generator=g)
        torch.rand(n, generator=g)
        torch.randn(n, generator=g)
    bsz, l, h, d = 1, 600, 2, 128
    q = torch.randn(bsz, l, h, d, generator=g).bfloat16()
    k = (torch.randn(bsz, l, h, d, generator=g) + torch.randn(1, 1, h, d, generator=g) * 2.0).bfloat16()
    v = torch.randn(bsz, l, h, d, generator=g).bfloat16()
    return q, k, v


def load(name):
    g = torch.load(os.path.join(GOLD, name + ".pt"))
    if name == "sla_a":
        q, k, v = sla_a_inputs()
        assert torch.equal(checksum(q, k, v), g["checksum"]), "regenerated sla_a inputs differ from the ones the golden was made from"
        g.update(q=q, k=k, v=v)
    return g
