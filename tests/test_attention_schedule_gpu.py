"""Attention against the fp64 reference where the other attention tests do not reach:

  * the persistent forward (attn_fwd5_kernel) with many work items per CTA, i.e. rounds r >= 1 of its item list, where
    the K / V ring, the P-chunk and S phases and the two XU-token barrier sets carry state from item to item; and the
    backward at the same shapes. Besides the fp64 comparison, a launch over a single (sequence, kv head) slice must give
    bit for bit what the big launch gave for that slice: an item's arithmetic does not depend on where it is scheduled;
  * score distributions that take the forward's lazy O rescale (running max up by more than 2^8 in a later kv tile),
    rows that stay below that threshold with P > 1, warps mixing both, tiles that underflow and a +300 score offset;
  * edge shapes: S < 128 and S = 1, GQA 8, Hq = Hkv = 1, prefix lengths 0, S and above S, head_dim 64 with documents and
    per-sequence prefixes, a non-default softmax scale, 1-token documents at tile borders.

The reference is R.attention_ref_grouped (dense fp64, one (sequence, kv head) at a time, on the GPU for the big shapes);
test_grouped_reference_matches_autograd_oracle checks it against the autograd oracle on the CPU. The input builders and
the replay of the rescale rule run on the CPU too, so that the structure these tests rely on is checked without a GPU."""
import math

import pytest
import torch

from llamax_b200 import ops
from oracle import ref_ops as R

gpu = pytest.mark.gpu
LOG2E = 1.4426950408889634
TILE = 128           # query and kv tile of both forward kernels
B200_SMS = 148       # the persistent forward's grid is min(items, SMs)
TOL = 1e-2


def _split(t, Hq, Hkv, Dh):
    return t[:, : Hq * Dh], t[:, Hq * Dh : (Hq + Hkv) * Dh], t[:, (Hq + Hkv) * Dh :]


def _heads(t, B, S, H, Dh):
    """[B*S, H*Dh] row view -> [B, H, S, Dh] view"""
    return t.reshape(B, S, H, Dh).transpose(1, 2)


def _doc_ids(B, S, lengths):
    assert sum(lengths) == S
    return torch.repeat_interleave(torch.arange(len(lengths)), torch.tensor(lengths))[None].expand(B, S).contiguous()


def _prefix_arg(P, device="cuda"):
    return torch.tensor(P, device=device, dtype=torch.int32) if isinstance(P, list) else P


def _slice_err(a, ref, Hkv):
    """Worst (sequence, kv head) slice of max|a - ref| / max|ref| (max|a| where the reference slice is exactly 0) and
    which slice it is. a, ref: [B, H, S, D] with H = Hkv * group."""
    B = ref.shape[0]
    d = (a.double() - ref).abs().reshape(B, Hkv, -1).amax(-1)
    r = ref.abs().reshape(B, Hkv, -1).amax(-1)
    e = torch.where(r > 0, d / r.clamp_min(1e-300), d)
    i = int(e.argmax())
    return e.max().item(), divmod(i, Hkv)


def _lse_err(a, ref):
    return (a.double() - ref).abs().max().item()


def _run_kernels(g, gd, B, S, Hq, Hkv, Dh, P, lengths=None, scale=None):
    """Forward and both backwards on the device buffers g = q|k|v [B*S, (Hq + 2 Hkv) Dh], gd = dO [B*S, Hq Dh]."""
    ds = de = None
    if lengths is not None:
        ds, de = ops.doc_bounds(_doc_ids(B, S, lengths).cuda())
    Pd = _prefix_arg(P)
    q, k, v = _split(g, Hq, Hkv, Dh)
    o, lse = ops.attn_fwd(q, k, v, B, S, Hq, Hkv, Dh, Pd, scale=scale, doc_start=ds)
    out = {"o": o, "lse": lse}
    for det in (False, True):
        dqkv = torch.zeros_like(g)
        dq, dk, dv = _split(dqkv, Hq, Hkv, Dh)
        ops.attn_bwd(q, k, v, o, lse, gd, dq, dk, dv, B, S, Hq, Hkv, Dh, Pd, scale=scale, doc_start=ds, doc_end=de,
                     deterministic=det)
        sfx = "_det" if det else ""
        out.update({"dq" + sfx: dq, "dk" + sfx: dk, "dv" + sfx: dv})
    torch.cuda.synchronize()
    return out


def _reference(g, gd, B, S, Hq, Hkv, Dh, P, lengths=None, scale=None, delta_from_bf16_o=False):
    q, k, v = _split(g, Hq, Hkv, Dh)
    doc_ids = None if lengths is None else _doc_ids(B, S, lengths).to(g.device)
    return R.attention_ref_grouped(_heads(q, B, S, Hq, Dh), _heads(k, B, S, Hkv, Dh), _heads(v, B, S, Hkv, Dh),
                                   _heads(gd, B, S, Hq, Dh), P, doc_ids=doc_ids, scale=scale,
                                   delta_from_bf16_o=delta_from_bf16_o)


def _errors(out, ref, B, S, Hq, Hkv, Dh):
    """name -> (worst slice error, (b, kv head)) for o, dq, dk, dv of both backwards; 'lse' -> max abs error."""
    o_r, lse_r, dq_r, dk_r, dv_r = ref
    errs = {"o": _slice_err(_heads(out["o"], B, S, Hq, Dh), o_r, Hkv), "lse": (_lse_err(out["lse"], lse_r), None)}
    for sfx in ("", "_det"):
        errs["dq" + sfx] = _slice_err(_heads(out["dq" + sfx], B, S, Hq, Dh), dq_r, Hkv)
        errs["dk" + sfx] = _slice_err(_heads(out["dk" + sfx], B, S, Hkv, Dh), dk_r, Hkv)
        errs["dv" + sfx] = _slice_err(_heads(out["dv" + sfx], B, S, Hkv, Dh), dv_r, Hkv)
    return errs


# ------------------------------------------------------------------------------------------------ reference helper (CPU)
@pytest.mark.parametrize("B,S,Hq,Hkv,P,lengths,scale", [
    (2, 200, 4, 2, 70, None, None),                  # scalar prefix, ragged S
    (3, 150, 4, 1, [0, 77, 400], None, None),        # per-sequence prefix (one above S)
    (2, 160, 2, 1, 0, [40, 1, 119], None),           # packed documents with a 1-token document
    (1, 130, 8, 1, 20, None, 0.3),                   # GQA 8, non-default scale
])
def test_grouped_reference_matches_autograd_oracle(B, S, Hq, Hkv, P, lengths, scale):
    Dh = 64
    torch.manual_seed(S)
    q, dout = torch.randn(B, Hq, S, Dh).bfloat16(), torch.randn(B, Hq, S, Dh).bfloat16()
    k, v = torch.randn(B, Hkv, S, Dh).bfloat16(), torch.randn(B, Hkv, S, Dh).bfloat16()
    doc_ids = None if lengths is None else _doc_ids(B, S, lengths)
    o, lse, dq, dk, dv = R.attention_ref_grouped(q, k, v, dout, P, doc_ids=doc_ids, scale=scale)
    for b in range(B):
        Pb = P[b] if isinstance(P, list) else P
        sl = slice(b, b + 1)
        # the autograd oracle has the fixed 1/sqrt(D) scale: fold a different scale into q (exact in fp64)
        qs = q[sl].double() * (1.0 if scale is None else scale * math.sqrt(Dh))
        o_r, dq_r, dk_r, dv_r = R.attention_ref_grads(qs, k[sl], v[sl], dout[sl], Pb,
                                                      doc_ids=None if doc_ids is None else doc_ids[sl])
        if scale is not None:
            dq_r = dq_r * (scale * math.sqrt(Dh))
        s = (qs @ k[sl].double().repeat_interleave(Hq // Hkv, 1).transpose(-1, -2)) / math.sqrt(Dh)
        mask = R.prefix_lm_mask(S, Pb) if doc_ids is None else R.document_causal_mask(doc_ids[sl])
        lse_r = torch.logsumexp(s.masked_fill(~mask, float("-inf")), -1)
        for name, a, r in (("o", o[sl], o_r), ("lse", lse[sl], lse_r), ("dq", dq[sl], dq_r), ("dk", dk[sl], dk_r),
                           ("dv", dv[sl], dv_r)):
            assert a.dtype is torch.float64 and a.shape == r.shape, name
            assert torch.allclose(a, r, rtol=1e-10, atol=1e-12), (name, b, (a - r).abs().max().item())
    # delta from the bf16-rounded output changes the gradients of q and k only, by a little
    o2, lse2, dq2, dk2, dv2 = R.attention_ref_grouped(q, k, v, dout, P, doc_ids=doc_ids, scale=scale,
                                                      delta_from_bf16_o=True)
    assert torch.equal(o2, o) and torch.equal(lse2, lse) and torch.equal(dv2, dv)
    assert 0 < (dq2 - dq).abs().max() <= 1e-2 * dq.abs().max()


# ------------------------------------------------------------------------------------------------ B: multi-item launches
# (B, S, Hq, Hkv, prefix, head_dim): the config-5 size, the benchmark's text step, the speech shape with mixed prefix
# lengths, an odd number of query tiles (the last pair's second tile is past the end), head_dim 64 with GQA 4
SCHEDULE_CASES = [
    (2, 4096, 32, 8, 0, 128),
    (8, 2048, 32, 8, 0, 128),
    (4, 1756, 32, 8, [1500, 0, 1756, 300], 128),
    (3, 1900, 16, 2, 100, 128),
    (4, 2048, 16, 4, 0, 64),
]


def _n_pairs(S):
    return (math.ceil(S / TILE) + 1) // 2


def _item_slice(k, B, S, Hq, Hkv):
    """(sequence, kv head, pair index) of work item k of the persistent forward (its decode())."""
    per_pair = B * Hq
    rem = k % per_pair
    return rem // Hq, (rem % Hq) // (Hq // Hkv), _n_pairs(S) - 1 - k // per_pair


def _probe_slices(B, S, Hq, Hkv, sms):
    """Slices holding items 0, G - 1, G and n_items - 1 (G = grid size: the first and last items of round 0, the first
    item of round 1 and the last item of all), plus one seeded random slice."""
    n_items = _n_pairs(S) * B * Hq
    G = min(n_items, sms)
    ks = [0, G - 1, G, n_items - 1]
    out = []
    for k in ks:
        b, hk, _ = _item_slice(k, B, S, Hq, Hkv)
        if (b, hk) not in out:
            out.append((b, hk))
    gen = torch.Generator().manual_seed(B * S + Hq)
    extra = (int(torch.randint(B, (1,), generator=gen)), int(torch.randint(Hkv, (1,), generator=gen)))
    if extra not in out:
        out.append(extra)
    return out


@pytest.mark.parametrize("B,S,Hq,Hkv,P,Dh", SCHEDULE_CASES)
def test_schedule_cases_run_several_rounds(B, S, Hq, Hkv, P, Dh):
    """CPU: every multi-item case gives each CTA of a full B200 at least two rounds, and the probe slices hold the items
    at the round boundaries."""
    n_items = _n_pairs(S) * B * Hq
    assert n_items > 2 * B200_SMS
    slices = _probe_slices(B, S, Hq, Hkv, B200_SMS)
    assert all(0 <= b < B and 0 <= hk < Hkv for b, hk in slices)
    for k in (0, B200_SMS - 1, B200_SMS, n_items - 1):
        assert _item_slice(k, B, S, Hq, Hkv)[:2] in slices
    if S == 1900:   # 15 query tiles: the last pair index has one tile only
        assert math.ceil(S / TILE) % 2 == 1


def _inputs(B, S, Hq, Hkv, Dh, seed):
    torch.manual_seed(seed)
    g = torch.randn(B * S, (Hq + 2 * Hkv) * Dh, device="cuda").bfloat16()
    gd = torch.randn(B * S, Hq * Dh, device="cuda").bfloat16()
    return g, gd


def _print_table(title, errs, extra=None):
    print(f"\n{title}")
    for name, (e, where) in errs.items():
        col = "" if extra is None or name not in extra else f"   emulated-delta {extra[name]:9.3e}"
        print(f"  {name:7s} {e:9.3e}" + ("" if where is None else f"  worst slice (b, kv head) = {where}") + col)


@gpu
@pytest.mark.parametrize("B,S,Hq,Hkv,P,Dh", SCHEDULE_CASES)
def test_multi_item_launch_vs_fp64(B, S, Hq, Hkv, P, Dh):
    """Every (sequence, kv head) slice of o, lse and of dq / dk / dv from the atomic and the deterministic backward
    against dense fp64 attention, at shapes where each CTA of the persistent forward runs several items."""
    g, gd = _inputs(B, S, Hq, Hkv, Dh, seed=S + Hq)
    out = _run_kernels(g, gd, B, S, Hq, Hkv, Dh, P)
    ref = _reference(g, gd, B, S, Hq, Hkv, Dh, P)
    errs = _errors(out, ref, B, S, Hq, Hkv, Dh)
    n_items = _n_pairs(S) * B * Hq
    _print_table(f"multi-item B={B} S={S} Hq={Hq} Hkv={Hkv} P={P} Dh={Dh} ({n_items} items, "
                 f"{math.ceil(n_items / min(n_items, torch.cuda.get_device_properties(0).multi_processor_count))} "
                 f"rounds)", errs)
    bad = {n: e for n, e in errs.items() if e[0] > (1e-3 if n == "lse" else TOL)}
    assert not bad, bad


def _slice_views(t, b, S, c0, c1):
    return t[b * S : (b + 1) * S, c0:c1]


@gpu
@pytest.mark.parametrize("B,S,Hq,Hkv,P,Dh", SCHEDULE_CASES)
def test_multi_item_launch_is_schedule_independent(B, S, Hq, Hkv, P, Dh):
    """A launch over one (sequence, kv head) slice (B = 1, Hq = group, Hkv = 1: a handful of items, all in round 0) on
    column views of the same buffers reproduces that slice of the big launch bit for bit: o and lse of the forward, dk
    and dv of the atomic backward, dq, dk and dv of the deterministic one. A read of another item's Q, K, V or P, or a
    hand-off on a wrong barrier phase, shows up here even where it would hide inside the 1e-2 bar."""
    g, gd = _inputs(B, S, Hq, Hkv, Dh, seed=S + Hq + 1)
    out = _run_kernels(g, gd, B, S, Hq, Hkv, Dh, P)
    Gq = Hq // Hkv
    q, k, v = _split(g, Hq, Hkv, Dh)
    slices = _probe_slices(B, S, Hq, Hkv, torch.cuda.get_device_properties(0).multi_processor_count)
    for b, hk in slices:
        qc, oc = (hk * Gq * Dh, (hk + 1) * Gq * Dh), (hk * Dh, (hk + 1) * Dh)
        qs, ks, vs = _slice_views(q, b, S, *qc), _slice_views(k, b, S, *oc), _slice_views(v, b, S, *oc)
        dos = _slice_views(gd, b, S, *qc)
        Ps = torch.tensor(P[b : b + 1], device="cuda", dtype=torch.int32) if isinstance(P, list) else P
        o1, lse1 = ops.attn_fwd(qs, ks, vs, 1, S, Gq, 1, Dh, Ps)
        assert torch.equal(o1, _slice_views(out["o"], b, S, *qc)), ("o", b, hk)
        assert torch.equal(lse1[0], out["lse"][b, hk * Gq : (hk + 1) * Gq]), ("lse", b, hk)
        # the backwards of the slice read the big launch's o and lse
        o_big = _slice_views(out["o"], b, S, *qc)
        lse_big = out["lse"][b : b + 1, hk * Gq : (hk + 1) * Gq]
        assert lse_big.is_contiguous()
        for det in (False, True):
            dq1 = torch.zeros(S, Gq * Dh, device="cuda", dtype=torch.bfloat16)
            dk1 = torch.zeros(S, Dh, device="cuda", dtype=torch.bfloat16)
            dv1 = torch.zeros_like(dk1)
            ops.attn_bwd(qs, ks, vs, o_big, lse_big, dos, dq1, dk1, dv1, 1, S, Gq, 1, Dh, Ps, deterministic=det)
            sfx = "_det" if det else ""
            assert torch.equal(dk1, _slice_views(out["dk" + sfx], b, S, *oc)), ("dk" + sfx, b, hk)
            assert torch.equal(dv1, _slice_views(out["dv" + sfx], b, S, *oc)), ("dv" + sfx, b, hk)
            if det:   # the atomic dQ sums in completion order: only the deterministic one is reproducible
                assert torch.equal(dq1, _slice_views(out["dq_det"], b, S, *qc)), ("dq_det", b, hk)
    print(f"\nschedule independence B={B} S={S} Hq={Hq} Hkv={Hkv} P={P} Dh={Dh}: slices {slices} bitwise equal")


# ------------------------------------------------------------------------------------------------ C: lazy O rescale
# Score structure planted in q and k (coordinates 0 .. 2 + kv tiles; the rest is N(0, 0.5^2) noise):
#   coordinate 0: k = 4 x position / 128 (a ramp), q = per-head slope in log2 units per kv tile (x 0.75-1.25 per row);
#   coordinate 1: k = 16, q sets a common offset of the row's scores (natural units, x 0.75-1.25 per row);
#   coordinate 2: k = 32 from 128 positions into the key's document on, q = a drop of 150-250 (log2 units) there:
#                 later tiles underflow;
#   coordinate 3 + t: k = 16 at one "spike" key inside kv tile t, q = spike height (log2 units) for the rows that spike
#                     there — a third of the rows of a spiking head: none, rise 1-6 (P > 1, no rescale), rise 10-30.
# Every planted q value varies per row: with one value per head, dk of that coordinate would be the value times a column
# sum of dS, which cancels to a small difference of large bf16-rounded terms (1000x at head_dim 64 with a ramp of -150
# per tile), and measure the rounding of the MMA accumulation rather than the kernel.
# Modes by head (h % 8): (slope per kv tile, offset, drop after tile 0, spikes)
_MODES = [(0.0, 0.0, 0.0, True), (12.0, 0.0, 0.0, False), (3.0, 0.0, 0.0, False), (0.0, 0.0, 200.0, False),
          (0.0, 300.0, 0.0, True), (3.0, 300.0, 0.0, False), (12.0, 0.0, 0.0, True), (-5.0, 0.0, 0.0, True)]


def _first_tiles(B, S, lengths):
    """[B, S] first kv tile the forward visits for each row: 0 (attn_fwd5_kernel), or with packed documents the tile of
    the first row's document start of the row's query tile (attn_fwd2_kernel)."""
    if lengths is None:
        return torch.zeros(B, S, dtype=torch.long)
    ds, _ = ops.doc_bounds(_doc_ids(B, S, lengths))
    q0 = (torch.arange(S) // TILE) * TILE
    return (ds[:, q0] // TILE).long()


def _visible(S, Pb, doc):
    idx = torch.arange(S)
    if doc is None:
        return (idx[None, :] < Pb) | (idx[:, None] >= idx[None, :])
    return (doc[:, None] == doc[None, :]) & (idx[:, None] >= idx[None, :])


def _peaked_inputs(B, S, Hq, Hkv, Dh, P, lengths, seed):
    """CPU bf16 (q|k|v [B*S, (Hq + 2 Hkv) Dh], dO [B*S, Hq Dh]) with the structure above."""
    gen = torch.Generator().manual_seed(seed)
    n_t = math.ceil(S / TILE)
    assert 3 + n_t <= Dh
    sl2 = Dh ** -0.5 * LOG2E              # raw dot product -> the kernels' log2 score units (default scale)
    q = 0.5 * torch.randn(B, S, Hq, Dh, generator=gen)
    k = 0.5 * torch.randn(B, S, Hkv, Dh, generator=gen)
    v = torch.randn(B, S, Hkv, Dh, generator=gen)
    dout = torch.randn(B, S, Hq, Dh, generator=gen)
    q[..., : 3 + n_t] = 0
    k[..., : 3 + n_t] = 0
    k[..., 0] = 4.0 * (torch.arange(S) / TILE)[None, :, None]
    k[..., 1] = 16.0
    starts = ops.doc_bounds(_doc_ids(B, S, lengths))[0] if lengths is not None else torch.zeros(B, S, dtype=torch.int32)
    k[..., 2] = 32.0 * (torch.arange(S)[None, :] - starts >= TILE).float()[..., None]
    spike = [None] + [t * TILE + int(torch.randint(min(TILE, S - t * TILE), (1,), generator=gen)) for t in range(1, n_t)]
    for t in range(1, n_t):
        k[:, spike[t], :, 3 + t] = 16.0
    first = _first_tiles(B, S, lengths)
    doc_ids = None if lengths is None else _doc_ids(B, S, lengths)
    for b in range(B):
        Pb = P[b] if isinstance(P, list) else P
        vis = _visible(S, Pb, None if doc_ids is None else doc_ids[b])
        for h in range(Hq):
            slope, offset, drop, spikes = _MODES[h % len(_MODES)]
            q[b, :, h, 0] = slope / sl2 / 4.0 * (0.75 + 0.5 * torch.rand(S, generator=gen))
            q[b, :, h, 1] = offset / Dh ** -0.5 / 16.0 * (0.75 + 0.5 * torch.rand(S, generator=gen))
            q[b, :, h, 2] = -drop / sl2 / 32.0 * (0.75 + 0.5 * torch.rand(S, generator=gen))
            if not spikes:
                continue
            kind = torch.randint(3, (S,), generator=gen)
            height = torch.where(kind == 1, 1 + 5 * torch.rand(S, generator=gen), 10 + 20 * torch.rand(S, generator=gen))
            pick = torch.rand(S, generator=gen)
            for i in range(S):
                if kind[i] == 0:
                    continue
                ts = [t for t in range(int(first[b, i]) + 1, n_t) if vis[i, spike[t]]]
                if ts:
                    t = ts[int(pick[i] * len(ts))]
                    q[b, i, h, 3 + t] = height[i] / sl2 / 16.0
    qkv = torch.cat([q.reshape(B * S, -1), k.reshape(B * S, -1), v.reshape(B * S, -1)], 1).bfloat16()
    return qkv, dout.reshape(B * S, -1).bfloat16()


def _rescale_stats(qkv, B, S, Hq, Hkv, Dh, P, lengths):
    """Replays the forwards' lazy rescale rule (m_tile > m_used + 8 in log2 units, kv tiles of 128 from the row's first
    visited tile) on fp64 scores of the bf16 inputs. Returns the fraction of rows that rescale after their first visited
    tile, the fraction that see a later tile raise their max by 1 .. 8 without a rescale (P up to 2^8 in bf16), the
    number of (32-row warp, kv step) pairs in which some rows rescale and others do not, the number of rows with a later
    visited tile that underflows as a whole (its max below the running max - 126) and the largest lse in natural units."""
    q, k, _ = _split(qkv, Hq, Hkv, Dh)
    q4, k4 = _heads(q, B, S, Hq, Dh), _heads(k, B, S, Hkv, Dh)
    n_t = math.ceil(S / TILE)
    sl2 = Dh ** -0.5 * LOG2E
    first = _first_tiles(B, S, lengths)
    doc_ids = None if lengths is None else _doc_ids(B, S, lengths)
    rows = resc_rows = pover_rows = mixed = under_rows = 0
    max_lse = -math.inf
    for b in range(B):
        Pb = P[b] if isinstance(P, list) else P
        vis = _visible(S, Pb, None if doc_ids is None else doc_ids[b])
        fb = first[b]
        for h in range(Hq):
            s = (q4[b, h].double() @ k4[b, h // (Hq // Hkv)].double().T) * sl2
            s = s.masked_fill(~vis, -math.inf)
            max_lse = max(max_lse, (torch.logsumexp(s, -1) / LOG2E).max().item())
            tmax = torch.nn.functional.pad(s, (0, n_t * TILE - S), value=-math.inf).reshape(S, n_t, TILE).amax(-1)
            m = torch.full((S,), -math.inf, dtype=torch.float64)
            resc = torch.zeros(S, n_t, dtype=torch.bool)
            pover = torch.zeros(S, dtype=torch.bool)
            under = torch.zeros(S, dtype=torch.bool)
            for t in range(n_t):
                active = t >= fb
                mt = tmax[:, t]
                up = active & (mt > m + 8)
                finite = torch.isfinite(m)
                resc[:, t] = up & finite
                pover |= active & finite & ~up & (mt > m + 1)
                m = torch.where(up, mt, m)
                under |= active & (t > fb) & torch.isfinite(mt) & (mt < m - 126)
            rows += S
            resc_rows += int(resc.any(1).sum())
            pover_rows += int(pover.sum())
            under_rows += int(under.sum())
            w = torch.nn.functional.pad(resc, (0, 0, 0, (-S) % 32)).reshape(-1, 32, n_t)
            lim = torch.nn.functional.pad(torch.ones(S, dtype=torch.bool), (0, (-S) % 32)).reshape(-1, 32, 1)
            mixed += int((w.any(1) & ~(w | ~lim).all(1)).sum())
    return resc_rows / rows, pover_rows / rows, mixed, under_rows, max_lse


# (B, S, Hq, Hkv, prefix, document lengths, head_dim): attn_fwd5_kernel with a scalar and a per-sequence prefix,
# attn_fwd2_kernel (packed documents), head_dim 128 and 64
RESCALE_CASES = [
    (2, 1536, 8, 2, 200, None, 128),
    (3, 1024, 8, 2, [0, 700, 1024], None, 128),
    (1, 2048, 8, 2, 0, [300, 1, 1000, 747], 128),
    (2, 1024, 8, 2, 0, None, 64),
    (1, 1024, 8, 2, 0, [129, 383, 512], 64),
]


@pytest.mark.parametrize("B,S,Hq,Hkv,P,lengths,Dh", RESCALE_CASES)
def test_peaked_inputs_reach_the_rescale_branch(B, S, Hq, Hkv, P, lengths, Dh):
    """CPU: the planted scores make the forwards take the lazy rescale on a large share of rows, leave another share with
    P > 1 and no rescale, split warps between the two, underflow whole later tiles, and lift lse to ~ +300."""
    qkv, _ = _peaked_inputs(B, S, Hq, Hkv, Dh, P, lengths, seed=S + Dh)
    resc, pover, mixed, under, max_lse = _rescale_stats(qkv, B, S, Hq, Hkv, Dh, P, lengths)
    print(f"\nrescale rows {resc:.2f}  P>1 without rescale {pover:.2f}  mixed warp-steps {mixed}  underflow rows {under}"
          f"  max lse {max_lse:.1f}")
    assert resc >= 0.15 and pover >= 0.15   # short documents have few later tiles: 0.18 and 0.26 at [129, 383, 512]
    assert mixed >= 20
    assert under >= TILE
    assert max_lse > 250


@gpu
@pytest.mark.parametrize("B,S,Hq,Hkv,P,lengths,Dh", RESCALE_CASES)
def test_rescale_branch_vs_fp64(B, S, Hq, Hkv, P, lengths, Dh):
    """o and lse at the standard bars; the gradients at max(1e-2, 1.5 x the error of the fp64 formulas with delta taken
    from the bf16-rounded output), because a peaked softmax makes dP - delta cancel and the kernel reads delta from its
    bf16 o."""
    qkv, dout = _peaked_inputs(B, S, Hq, Hkv, Dh, P, lengths, seed=S + Dh)
    g, gd = qkv.cuda(), dout.cuda()
    out = _run_kernels(g, gd, B, S, Hq, Hkv, Dh, P, lengths)
    ref = _reference(g, gd, B, S, Hq, Hkv, Dh, P, lengths)
    emul = _reference(g, gd, B, S, Hq, Hkv, Dh, P, lengths, delta_from_bf16_o=True)
    errs = _errors(out, ref, B, S, Hq, Hkv, Dh)
    emul_err = {}
    for name, i in (("dq", 2), ("dk", 3), ("dv", 4)):
        emul_err[name] = emul_err[name + "_det"] = _slice_err(emul[i], ref[i], Hkv)[0]
    _print_table(f"rescale inputs B={B} S={S} Hq={Hq} Hkv={Hkv} P={P} docs={lengths} Dh={Dh}", errs, emul_err)
    assert ref[1].max().item() > 250   # the +300 offset heads reached the kernels
    bad = {}
    for name, (e, where) in errs.items():
        lim = 1e-3 if name == "lse" else max(TOL, 1.5 * emul_err[name]) if name in emul_err else TOL
        if e > lim:
            bad[name] = (e, where, lim)
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ D: edge shapes
# (B, S, Hq, Hkv, prefix, head_dim, document lengths, scale)
EDGE_CASES = [
    (3, 1, 4, 1, 0, 128, None, None),
    (3, 17, 4, 1, 5, 128, None, None),
    (3, 64, 4, 2, 0, 128, None, None),
    (3, 127, 4, 2, 100, 128, None, None),
    (2, 300, 8, 1, 0, 128, None, None),                       # GQA 8
    (1, 640, 16, 2, 128, 128, None, None),                    # GQA 8 with two kv heads
    (2, 200, 1, 1, 50, 128, None, None),                      # one query head, one kv head
    (4, 300, 4, 2, [0, 300, 800, 77], 128, None, None),       # per-sequence prefix: 0, S, above S
    (1, 300, 8, 2, 0, 64, [100, 28, 172], None),              # head_dim 64, packed documents
    (3, 256, 8, 2, [0, 256, 1000], 64, None, None),           # head_dim 64, per-sequence prefix
    (2, 384, 8, 2, 100, 128, None, 0.3),                      # non-default softmax scale
    (1, 640, 4, 1, 0, 128, [100, 28, 512], 0.3),              # ... with packed documents
    (2, 768, 4, 1, 0, 128, [128, 1, 126, 1, 128, 1, 383], None),   # 1-token documents at 128, 255 and 384
]


@gpu
@pytest.mark.parametrize("B,S,Hq,Hkv,P,Dh,lengths,scale", EDGE_CASES)
def test_edge_shapes_vs_fp64(B, S, Hq, Hkv, P, Dh, lengths, scale):
    g, gd = _inputs(B, S, Hq, Hkv, Dh, seed=3 * S + Hq)
    out = _run_kernels(g, gd, B, S, Hq, Hkv, Dh, P, lengths, scale)
    ref = _reference(g, gd, B, S, Hq, Hkv, Dh, P, lengths, scale)
    errs = _errors(out, ref, B, S, Hq, Hkv, Dh)
    _print_table(f"edge B={B} S={S} Hq={Hq} Hkv={Hkv} P={P} Dh={Dh} docs={lengths} scale={scale}", errs)
    bad = {n: e for n, e in errs.items() if e[0] > (1e-3 if n == "lse" else TOL)}
    assert not bad, bad
    assert torch.equal(out["dk"], out["dk_det"]) and torch.equal(out["dv"], out["dv_det"])


@gpu
@pytest.mark.parametrize("Dh", [128, 64])
def test_prefix_above_sequence_length_is_clamped(Dh):
    """A prefix longer than the sequence means "all of it": P = S + 500 gives exactly what P = S gives, as a scalar and
    as an entry of a per-sequence vector, in the forward and in both backwards."""
    B, S, Hq, Hkv = 2, 300, 4, 2
    g, gd = _inputs(B, S, Hq, Hkv, Dh, seed=Dh)
    for over, exact in ((S + 500, S), ([S + 500, 40], [S, 40])):
        a = _run_kernels(g, gd, B, S, Hq, Hkv, Dh, over)
        e = _run_kernels(g, gd, B, S, Hq, Hkv, Dh, exact)
        for name in ("o", "lse", "dk", "dv", "dq_det", "dk_det", "dv_det"):
            assert torch.equal(a[name], e[name]), (name, over)
