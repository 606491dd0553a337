"""Block-map parity at the FULL block counts (Nblk = 512 for Wan-1.3B 480p, 1182 for Wan-14B 720p) against the reference's own
`get_block_map` (SLA/utils.py:55-67), run on the CPU by tools/make_golden.py (Triton interpreter for mean_pool, torch.topk).

The fixtures hold the reference's key mean and pooled keys, and for a seeded sample of query blocks (the first and the ragged
last one always included; one head of the two at Nblk = 1182) its pooled queries, bf16 scores and selected key blocks; the
inputs are regenerated here from the same seeded CPU generator (checksum-verified).  Asserted on the stored heads and rows:
  * pooled query/key means and the key mean: bit-equal to the reference except a counted handful of 1-ulp differences
    (fp32 summation order);
  * fed the REFERENCE's pooled vectors, our score + exact top-k selects exactly the reference's set in every row where the
    reference's k-th and (k+1)-th bf16 scores differ ("no tie at the threshold"); rows with a tie at the threshold are
    counted separately and must still select a valid top-k of the reference's scores;
  * end to end from q,k the maps agree except at entries whose reference score is within one bf16 ulp of the row threshold.
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def blockmap_inputs(l, h, d, seed):
    """Byte-identical to tools/make_golden.py:blockmap_inputs."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(1, h, l, d, generator=g).bfloat16()
    k = (torch.randn(1, h, l, d, generator=g) + torch.randn(1, h, 1, d, generator=g) * 2.0).bfloat16()
    return q, k


def _ulps(a, b):
    return (a.view(torch.int16).to(torch.int32) - b.view(torch.int16).to(torch.int32)).abs()


@pytest.mark.parametrize("name", ["blockmap_n512", "blockmap_n1182", "blockmap_n512_d64"])
def test_block_map_vs_reference_full_block_counts(cuda, name):
    from turbodiffusion_b200.SLA.utils import block_map_from_pools, get_block_map
    g = torch.load(os.path.join(GOLD, name + ".pt"))
    l, h, d, topk = g["l"], g["h"], g["d"], g["topk"]
    qh, kh = blockmap_inputs(l, h, d, g["seed"])
    csum = torch.stack([qh.view(torch.int16).to(torch.int64).sum(), kh.view(torch.int16).to(torch.int64).sum()])
    assert torch.equal(csum, g["checksum"]), "regenerated inputs differ from the ones the golden was made from"
    heads, rows = torch.tensor(g["heads"]), g["rows"]

    def sampled(t):                                              # [B, H, Mblk, ...] of every head and query block -> stored ones
        return t[:, heads][:, :, rows]

    score = g["score"].float()                                   # the reference's bf16 pooled scores
    nblk = score.shape[-1]
    ref_map = torch.zeros(score.shape, dtype=torch.bool).scatter_(-1, g["lut"].long(), True)
    assert topk == min(nblk, int(g["topk_ratio"] * nblk)) and (ref_map.sum(-1) == topk).all()
    srt = torch.sort(score, dim=-1, descending=True).values
    thr, nxt = srt[..., topk - 1], srt[..., topk]                # k-th and (k+1)-th score of every row
    tie_rows = thr == nxt

    # ---- (1) score + top-k alone, on the reference's pooled vectors
    pq, pk = g["pooled_q"].to(cuda), g["pooled_k"].to(cuda)
    ours_map, lut = block_map_from_pools(pq, pk, topk)
    ours = ours_map.cpu().bool()
    assert (ours.sum(-1) == topk).all()
    row_equal = (ours == ref_map).all(-1)
    bad_rows = ~row_equal & ~tie_rows
    # a no-tie row can still differ if OUR fp32 accumulation order rounds one score to the neighbouring bf16 value:
    # every differing entry must then sit within one bf16 ulp of the threshold
    diff = ours ^ ref_map
    near = (score - thr[..., None]).abs() <= 2.0 ** -7 * thr[..., None].abs() + 1e-30
    assert (near | ~diff).all(), "selection differs away from the threshold"
    # rows with a tie at the threshold: any choice among the tied blocks is a valid torch.topk(sorted=False) result
    lo = torch.where(ours, score, torch.full_like(score, float("inf"))).amin(-1)
    hi = torch.where(~ours, score, torch.full_like(score, float("-inf"))).amax(-1)
    valid_topk = lo >= hi
    n_rows = row_equal.numel()
    print(f"{name}: rows {n_rows}, identical {int(row_equal.sum())}, threshold-tie rows {int(tie_rows.sum())}, "
          f"no-tie rows differing (1-ulp score) {int(bad_rows.sum())}, rows that are not a valid top-k of the reference "
          f"scores {int((~valid_topk).sum())}")
    assert bad_rows.float().mean() <= 0.02
    assert (valid_topk | bad_rows).all()

    # ---- (2) pooled means + key mean from q,k
    from turbodiffusion_b200.SLA.utils import quant_qk
    qt, kt = qh.transpose(1, 2).contiguous().to(cuda), kh.transpose(1, 2).contiguous().to(cuda)   # module layout [B,L,H,D]
    prep = quant_qk(qt, kt)
    our_pq, our_pk = sampled(prep.q_pool.cpu()[..., :d]), prep.k_pool.cpu()[:, heads][..., :d]
    uq, uk = _ulps(our_pq, g["pooled_q"]), _ulps(our_pk, g["pooled_k"])
    print(f"{name}: pooled_q !=: {int((uq > 0).sum())}/{uq.numel()} (max {int(uq.max())} ulp), "
          f"pooled_k !=: {int((uk > 0).sum())}/{uk.numel()} (max {int(uk.max())} ulp)")
    assert uq.max() <= 1 and (uq > 0).float().mean() < 2e-3
    # pooled_k inherits the rounding of the 16-bit key mean (k - T(mean)): allow 1 ulp of the LARGEST element of the vector
    kmean_ref = g["kmean"].float()
    assert (prep.kmean.cpu()[:, heads][..., :d] - kmean_ref).abs().max() <= 2.0 ** -8 * kmean_ref.abs().max()
    assert ((our_pk.float() - g["pooled_k"].float()).abs() <= 2.0 ** -7 * g["pooled_k"].float().abs().amax(-1, keepdim=True)).all()

    # ---- (3) end to end
    e2e_map, _, e2e_topk = get_block_map(qh.to(cuda), kh.to(cuda), g["topk_ratio"], 128, 64)
    assert e2e_topk == topk
    e2e = sampled(e2e_map.cpu().bool())
    diff = e2e ^ ref_map
    near = (score - thr[..., None]).abs() <= 2.0 ** -6 * thr[..., None].abs() + 2.0 ** -6 * score.abs().amax(-1, keepdim=True)
    print(f"{name}: end-to-end differing entries {int(diff.sum())} of {diff.numel()} ({int((~(e2e == ref_map).all(-1)).sum())} rows)")
    assert (near | ~diff).all(), "end-to-end block map differs away from the selection threshold"
    assert diff.float().mean() < 2e-3
