"""The fused-producer MSDA kernels at the inputs where they can go wrong: sampling locations on and next to
bilinear cell edges and map borders, points off the map and non-finite offsets, extreme and degenerate logits,
decoder-style queries (Lq != S) through the fused backward, seeded random shapes, and the full-size pyramids.

The fused kernels compute the module's producers (ops/modules/ms_deform_attn.py:105-112) themselves: the softmax
of each (query, head)'s L*P logits and the location `ref + offset / (W, H)`, three times over -- phase1_records()
(msda_common.cuh) for the forward and the per-row backward, and pass A of the merging backward
(msda_bwd_sorted.cu).  Two contracts follow and are pinned here:
  * the location is bit-identical to the fp32 tensor expression (div_by_size() is an exact division);
  * the merging backward recomputes the same bits as the forward.
A location one ulp off next to a cell edge moves the point into another bilinear cell, where the location
gradient is different: the gradients then no longer belong to the function the forward computed.

Every location reference is computed on the CPU, so its division is IEEE by construction."""
import numpy as np
import pytest
import torch

from test_deterministic_gpu import _records_per_image, deterministic_mode
from test_fused_gpu import make_case, reference_composition
from test_parity_gpu import check_against

DEV = "cuda:0"
gpu = pytest.mark.gpu
STEPS = 3                     # offsets 0..3 ulps to either side of the one that targets an edge


# ---------------------------------------------------------------- the edge generator (CPU)
def fma_coord(loc, size):
    """fp32 fmaf(loc, size, -0.5) -- the kernels' pixel coordinate (msda_common.cuh: decompose) -- emulated in fp64:
    the product of an fp32 location and a level size below 2^24 is exact in fp64, and the subtraction of 0.5 is
    checked to be exact (two-sum residual 0), so the one rounding is the final cast to fp32."""
    p = np.asarray(loc, np.float64) * float(size)
    d = p - 0.5
    b = d - p
    residual = (p - (d - b)) + (-0.5 - b)
    assert not residual[np.isfinite(residual)].any(), "loc * size - 0.5 is not exact in fp64"
    return d.astype(np.float32)


def _ulp_steps(x, steps=STEPS):
    """[K] fp32 -> [K, 2 * steps + 1]: x moved by -steps..steps ulps (np.nextafter)."""
    cols = []
    for j in range(-steps, steps + 1):
        y = x.copy()
        for _ in range(abs(j)):
            y = np.nextafter(y, np.float32(np.inf if j > 0 else -np.inf))
        cols.append(y)
    return np.stack(cols, 1)


MAX_EDGES = 4098


def edge_ks(size):
    """The edges k of a level of `size` pixels the generator targets: every integer in [-1, size] (k = -1: the
    lower validity edge, k = size: the upper one, every integer between: a floor edge), or above 4096 pixels the
    64 edges at either end and a seeded sample of the interior, MAX_EDGES in all."""
    if size + 2 <= MAX_EDGES:
        return np.arange(-1, size + 1)
    inner = np.random.default_rng(size).choice(np.arange(64, size - 64), MAX_EDGES - 130, replace=False)
    return np.concatenate((np.arange(-1, 64), np.sort(inner), np.arange(size - 64, size + 1)))


def edge_locations(size, k):
    """The fp32 location closest to each edge k that puts fma_coord(loc, size) exactly on k, or RN((k + 0.5) / size)
    where no fp32 location does -> (loc [len(k)] fp32, reachable [len(k)] bool).  An edge can be out of reach:
    c = 0 needs loc * size == 0.5 exactly, i.e. a power-of-two size."""
    t = ((k + 0.5) / size).astype(np.float32)
    cand = np.stack([t, np.nextafter(t, np.float32(-2)), np.nextafter(t, np.float32(2))], 1)
    hit = fma_coord(cand, size).astype(np.float64) == k[:, None]
    pick = np.where(hit.any(1), hit.argmax(1), 0)
    return cand[np.arange(len(k)), pick], hit.any(1)


def edge_offsets(size):
    """Offsets (in pixels, as the sampling_offsets Linear produces them) and reference coordinates that put the
    fp32 location `ref + off / size` on every edge c = k of edge_ks(size) and on both sides of it, for three kinds
    of reference coordinate:
      ref = 0           the location is the quotient itself: any error of the division shows;
      ref = a pixel centre (i + 0.5) / size, what the encoder's reference points are;
      ref = the edge's own location (edge_locations), with offsets of 0 and +-1..3 ulps of 0.
    For the first two, off = (loc* - ref) * size is solved in fp64 for loc* = (k + 0.5) / size, rounded to fp32 and
    stepped by +-0..3 ulps.  -> (k [E], ref [E], off [E]) fp32, E = 3 * len(edge_ks(size)) * (2 * STEPS + 1)."""
    k = edge_ks(size)
    kinds = [np.zeros(len(k), np.float32),
             ((np.arange(len(k)) % size + 0.5) / size).astype(np.float32),
             edge_locations(size, k)[0]]
    ks, refs, offs = [], [], []
    for i, ref in enumerate(kinds):
        if i < 2:
            off0 = (((k + 0.5) / size - ref.astype(np.float64)) * size).astype(np.float32)
        else:
            off0 = np.zeros(len(k), np.float32)
        o = _ulp_steps(off0)
        ks.append(np.repeat(k, o.shape[1]))
        refs.append(np.repeat(ref, o.shape[1]))
        offs.append(o.reshape(-1))
    return np.concatenate(ks), np.concatenate(refs), np.concatenate(offs)


def location(ref, off, size):
    """The module's fp32 location ref + off / size (IEEE division and add, numpy fp32 on the CPU)."""
    return (np.asarray(ref, np.float32) + np.asarray(off, np.float32) / np.float32(size)).astype(np.float32)


def sweep_levels():
    """(H, W) of the level-size sweep: every W in 1..1024 with H in {1, 2, 3} and the same transposed; a seeded
    sample of 1025..5000; sizes past 5000 (5001, 8191, 8192, 16383, 65535); the pyramid widths 39 / 78 / 156 /
    1248 and the powers of two up to 2^14.  Thin levels keep `value` small, and at most MAX_EDGES edges per
    axis keep the number of points of a call below 1.4 million."""
    rng = np.random.default_rng(5000)
    sizes = list(range(1, 1025)) + sorted(int(s) for s in rng.choice(np.arange(1025, 5001), 48, replace=False))
    sizes += [5001, 8191, 8192, 16383, 65535, 1248, 2048, 4096, 16384]
    levels = {(h, w) for w in sizes for h in (1, 2, 3)}
    levels |= {(w, h) for h, w in levels}
    return sorted(levels, key=lambda hw: (max(hw), hw))


def test_edge_generator_hits_every_edge_from_both_sides():
    """CPU: for every size of the sweep, the generated fp32 locations put fmaf(loc, size, -0.5) below and above
    every edge of edge_ks(size), and exactly on it wherever some fp32 location can (every edge of a power-of-two
    size; for the other sizes all but c = 0 and a few percent of the rest, which no fp32 location reaches)."""
    sizes = sorted({max(hw) for hw in sweep_levels()} | {1, 2, 3})
    edges = unreachable = 0
    for size in sizes:
        ks = edge_ks(size)
        k, ref, off = edge_offsets(size)
        c = fma_coord(location(ref, off, size), size).astype(np.float64)
        e = np.searchsorted(ks, k)                           # edge index of every generated offset
        on = np.zeros(len(ks), bool)
        below, above = on.copy(), on.copy()
        np.logical_or.at(on, e, c == k)
        np.logical_or.at(below, e, c < k)
        np.logical_or.at(above, e, c > k)
        reachable = edge_locations(size, ks)[1]
        edges += len(ks)
        unreachable += int((~reachable).sum())
        assert below.all() and above.all(), (size, ks[~(below & above)])
        assert on[reachable].all(), (size, ks[reachable & ~on])
        if size & (size - 1) == 0:
            assert reachable.all(), size
        else:
            assert not reachable[1], size          # c = 0: loc * size == 0.5 has no fp32 solution
    assert unreachable <= 0.08 * edges, (unreachable, edges)
    print(f"\n{len(sizes)} sizes, {edges} edges, all hit from both sides; {edges - unreachable} hit exactly, "
          f"{unreachable} out of reach of any fp32 location")


# ---------------------------------------------------------------- helpers (GPU)
def _dev(c):
    return {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in c.items()}


def _unfused_loc_weights(c):
    """The module's own fp32 producers on the CPU: location ref + off / (W, H) and torch's softmax of the logits."""
    N, Lq, M, L, P, _ = c["off"].shape
    wh = c["shapes"].flip(-1).float()
    loc = c["ref"][:, :, None, :, None, :] + c["off"] / wh[None, None, None, :, None, :]
    w = torch.softmax(c["logits"], -1).view(N, Lq, M, L, P)
    return loc.expand(N, Lq, M, L, P, 2).contiguous(), w.contiguous()


def _fused_fwd_bwd(pkg, c, variant):
    """Fused forward + backward on the GPU -> (out, grad_value, grad_offsets, grad_logits, backward launches).
    variant: the "bwd_variant" option (0: the default entry, 20: merging kernel forced, 2: per-row kernel forced)
    or "det" (torch.use_deterministic_algorithms(True))."""
    d = _dev(c)
    a = (d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"])
    out = pkg.ms_deform_attn_fused_forward(*a)
    n0 = pkg.launch_count()
    if variant == "det":
        with deterministic_mode():
            g = pkg.ms_deform_attn_fused_backward(*a, d["grad_out"])
    else:
        pkg.set_option("bwd_variant", variant)
        try:
            g = pkg.ms_deform_attn_fused_backward(*a, d["grad_out"])
        finally:
            pkg.set_option("bwd_variant", 0)
    torch.cuda.synchronize()
    return (out, *g, pkg.launch_count() - n0)


def _no_nan(*ts):
    return all(not torch.isnan(t).any().item() for t in ts)


def _check_composition(pkg, oracle, c, variant, tag, ref=None):
    """Fused forward and the three gradients against reference_composition at FWD_ABS_TOL / GRAD_REL_TOL."""
    out, gv, goff, glog, launches = _fused_fwd_bwd(pkg, c, variant)
    assert _no_nan(out, gv, goff, glog), tag
    ref = ref if ref is not None else reference_composition(oracle, c)
    check_against(out, gv, goff, glog, *ref, tag=f"{tag} bwd_variant={variant}")
    return out, gv, goff, glog, launches


# ---------------------------------------------------------------- 1. cell edges and map borders
def _sweep_groups():
    """The sweep's levels in groups of 16 (L = 16, P = 1: L*P = 16), sorted by size so that a group's levels need
    similar numbers of points; the last group is filled up with the smallest levels."""
    levels = sweep_levels()
    groups = [levels[i:i + 16] for i in range(0, len(levels), 16)]
    groups[-1] += levels[:16 - len(groups[-1])]
    return groups


def _edge_case(pkg, levels, seed):
    """One call's inputs: level l's points are its x edges (edge_offsets(W)) paired with its y edges (edge_offsets(H)),
    each list repeated cyclically to Lq = the longest list of the group; one head, one point per level, one image;
    all logits equal (softmax exactly 1/16 in the kernel and in torch)."""
    L = len(levels)
    per_level = [(edge_offsets(w), edge_offsets(h)) for h, w in levels]
    Lq = max(max(len(x[2]), len(y[2])) for x, y in per_level)
    ref = np.empty((1, Lq, L, 2), np.float32)
    off = np.empty((1, Lq, 1, L, 1, 2), np.float32)
    for l, ((_, rx, ox), (_, ry, oy)) in enumerate(per_level):
        ref[0, :, l, 0], off[0, :, 0, l, 0, 0] = np.resize(rx, Lq), np.resize(ox, Lq)
        ref[0, :, l, 1], off[0, :, 0, l, 0, 1] = np.resize(ry, Lq), np.resize(oy, Lq)
    gen = torch.Generator().manual_seed(seed)
    S = sum(h * w for h, w in levels)
    shapes, lsi = pkg.synthetic.level_tensors(levels)
    return dict(value=torch.randn(1, S, 1, 32, generator=gen), ref=torch.from_numpy(ref), off=torch.from_numpy(off),
                logits=torch.full((1, Lq, 1, L), 0.75), grad_out=torch.randn(1, Lq, 32, generator=gen),
                shapes=shapes, lsi=lsi, levels=levels)


@gpu
def test_edge_locations_are_bit_exact_in_forward_and_per_row_backward(pkg):
    """Check A and B over the whole size sweep (6 477 levels in 405 calls of 16 levels; every edge of
    edge_ks() of every level from both sides and, where reachable, exactly).
      A: ms_deform_attn_fused_forward == ms_deform_attn_forward fed with the CPU's ref + off / (W, H) and torch's
         softmax, BIT FOR BIT.  The logits are all equal, so both weights are exactly 1/16, and both run the same
         kernel template and configuration (launch_fwd_cfg<16, 16, 16, 2, 8> with FUSED on and off): only a
         location that differs can change a bit.
      B: with torch.use_deterministic_algorithms(True), the fused backward's grad_value == the plain backward's,
         BIT FOR BIT (the same records, gathered in the same order), and its grad_sampling_offsets == the plain
         grad_sampling_loc / (W, H) divided on the CPU, BIT FOR BIT."""
    for i, levels in enumerate(_sweep_groups()):
        c = _edge_case(pkg, levels, seed=i)
        loc, w = _unfused_loc_weights(c)
        assert torch.equal(w, torch.full_like(w, 1 / 16))
        d = _dev(dict(c, loc=loc, w=w))
        fused = pkg.ms_deform_attn_fused_forward(d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"])
        plain = pkg.ms_deform_attn_forward(d["value"], d["shapes"], d["lsi"], d["loc"], d["w"], 128)
        bad = (fused != plain).any(-1)[0]
        assert not bad.any().item(), f"{levels}: forward differs at queries {bad.nonzero()[:8, 0].tolist()}"
        with deterministic_mode():
            gf = pkg.ms_deform_attn_fused_backward(d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"],
                                                   d["grad_out"])
            gp = pkg.ms_deform_attn_backward(d["value"], d["shapes"], d["lsi"], d["loc"], d["w"], d["grad_out"], 128)
        assert torch.equal(gf[0], gp[0]), f"{levels}: grad_value differs"
        wh = c["shapes"].flip(-1).float()
        assert torch.equal(gf[1].cpu(), gp[1].cpu() / wh[None, None, None, :, None, :]), f"{levels}: grad_offsets"


def _edge_case_square(pkg, levels, heads, points, seed):
    """Lq == S inputs whose points sit on and next to cell edges: point i of level l targets entry i (cyclically) of
    edge_offsets(W_l) in x and edge_offsets(H_l) in y, re-solved for the query's own reference coordinate (image 0:
    the pixel-centre reference points of the encoder; image 1: reference points 0, so that the location is the
    quotient itself).  Varied logits."""
    c = make_case(pkg, levels, 2, heads, points, True, seed)
    N, S, M, L, P, _ = c["off"].shape
    ref = torch.cat((c["ref"], torch.zeros_like(c["ref"])))                  # [2, S, L, 2]
    off = np.empty((N, S, M, L, P, 2), np.float32)
    for l, (h, w) in enumerate(levels):
        for axis, size in ((0, w), (1, h)):
            k, _, o = edge_offsets(size)
            pick = (np.arange(S * M * P) * 7919 + 13 * l + axis) % len(k)       # spread the edges over queries
            kk = k[pick].reshape(S, M, P)
            for n in range(N):
                r = ref[n, :, l, axis].numpy().astype(np.float64)[:, None, None]
                base = (((kk + 0.5) / size - r) * size).astype(np.float32)
                step = (pick % (2 * STEPS + 1) - STEPS).reshape(S, M, P)         # the generator's ulp steps
                for j in range(1, STEPS + 1):
                    base = np.where(step >= j, np.nextafter(base, np.float32(np.inf)), base)
                    base = np.where(step <= -j, np.nextafter(base, np.float32(-np.inf)), base)
                off[n, :, :, l, :, axis] = base
    return dict(c, ref=ref.contiguous(), off=torch.from_numpy(off))


@gpu
@pytest.mark.parametrize("levels,heads,points", [
    ([(16, 32), (8, 16), (4, 8), (2, 4)], 4, 4),         # L*P = 16, powers of two
    ([(12, 39), (24, 78)], 2, 4),                        # KITTI-like widths, L*P = 8
    ([(9, 13), (17, 5), (1, 1), (3, 2)], 2, 4),          # odd sizes and a 1x1 level, L*P = 16
    ([(33, 65)], 3, 4),                                  # one level, L*P = 4
    ([(7, 11), (13, 3), (5, 31)], 2, 4),                 # L*P = 12
])
def test_edge_locations_merging_and_per_row_backward_match_the_composition(pkg, oracle, levels, heads, points):
    """Check C: at Lq == S (where the merging kernel runs), points on and next to cell edges, varied logits: the
    default backward (bwd_variant 0), the merging kernel forced (20) and the per-row kernel forced (2) each give
    the forward and grad_value / grad_sampling_offsets / grad_attn_logits of reference_composition within
    FWD_ABS_TOL / GRAD_REL_TOL.  A location the merging kernel's pass A recomputes into another cell is an O(1)
    error of grad_sampling_offsets there."""
    c = _edge_case_square(pkg, levels, heads, points, seed=len(levels) * 10 + heads)
    ref = reference_composition(oracle, c)
    for variant in (0, 20, 2):
        _check_composition(pkg, oracle, c, variant, str(levels), ref=ref)


# ---------------------------------------------------------------- 2. points off the map, non-finite offsets
BAD_LOCATIONS = [(-5.0, 0.5), (0.5, 3.0), (float("nan"), 0.5), (0.5, float("inf")), (-0.01, -0.01), (1.01, 0.99)]
BAD_OFFSETS = [(float("-inf"), 0.5), (1e20, 0.25), (-3e20, 0.5), (0.5, 2e20)]     # 1e20: __fdiv_rn in div_by_size


def _off_map_case(pkg):
    """A third of the points moved to BAD_LOCATIONS (as offsets from their query's reference point) or given the
    BAD_OFFSETS (infinite, or ~1e20 pixels).  -> (case, stand-in case for the oracle, bad mask [N, S, M, L, P])."""
    levels = [(16, 32), (8, 16)]
    c = make_case(pkg, levels, 2, 4, 4, False, seed=7)
    N, S, M, L, P, _ = c["off"].shape
    wh = c["shapes"].flip(-1).double()                                     # (W, H) per level
    gen = torch.Generator().manual_seed(1)
    pick = torch.rand(N, S, M, L, P, generator=gen) < 1 / 3
    which = torch.randint(0, len(BAD_LOCATIONS) + len(BAD_OFFSETS), (N, S, M, L, P), generator=gen)
    ref = c["ref"][:, :, None, :, None, :].double().expand(N, S, M, L, P, 2)
    bad_loc = torch.tensor(BAD_LOCATIONS, dtype=torch.float64)[which.clamp(max=len(BAD_LOCATIONS) - 1)]
    as_off = ((bad_loc - ref) * wh[None, None, None, :, None, :]).float()  # nan / inf stay nan / inf
    direct = torch.tensor(BAD_OFFSETS, dtype=torch.float32)[(which - len(BAD_LOCATIONS)).clamp(min=0)]
    bad = torch.where((which < len(BAD_LOCATIONS))[..., None], as_off, direct)
    off = torch.where(pick[..., None], bad, c["off"])
    # the oracle gets a finite point far off the map in place of the non-finite and 1e20 ones
    far = pick & ((which >= len(BAD_LOCATIONS)) | ~torch.isfinite(bad).all(-1))
    standin = torch.where(far[..., None], torch.full_like(off, 1000.0), off)
    return dict(c, off=off), dict(c, off=standin), far


@gpu
@pytest.mark.parametrize("variant", [0, 20, 2, "det"])
def test_points_off_the_map_and_non_finite_offsets(pkg, oracle, variant):
    """Offsets that put a third of the points at x or y = -5, in (-1, 0), just past the border, NaN, +-inf, or
    ~1e20 pixels away: the fused forward and the three gradients -- default backward, merging kernel, per-row
    kernel, deterministic path -- match reference_composition (the oracle given a finite far-away stand-in for
    the non-finite / 1e20 points) within FWD_ABS_TOL / GRAD_REL_TOL, and contain no NaN.  As in the plain op, the
    invalid points contribute nothing and get zero offset gradients, while the softmax gradient still counts
    their weight (grad_logit_i = -a_i * sum_j a_j g_j there, not 0)."""
    c, standin, far = _off_map_case(pkg)
    ref = reference_composition(oracle, standin)
    _, _, goff, glog, _ = _check_composition(pkg, oracle, c, variant, "off the map", ref=ref)
    assert not goff.cpu()[far].any()
    glog = glog.cpu().view(far.shape)
    assert glog[far].abs().max().item() > 0        # the weights of the skipped points still enter the softmax


# ---------------------------------------------------------------- 3. extreme and degenerate logits
def _extreme_logits(shape, gen):
    """Rows (one per (image, query, head)) of six kinds: uniform in +-80; all near +100 (exp overflows in fp32 unless
    the row maximum is subtracted); all near -100 (every exp underflows to 0 unless it is); one dominant logit
    (+80 among -80: one-hot weights); all equal; and some entries -inf (at least one finite per row)."""
    N, Lq, M, LP = shape
    kind = torch.randint(0, 6, (N, Lq, M, 1), generator=gen).expand(shape)
    u = (torch.rand(shape, generator=gen) * 2 - 1) * 80
    near = torch.randn(shape, generator=gen)
    hot = torch.randint(0, LP, (N, Lq, M, 1), generator=gen)
    one_hot = torch.where(torch.arange(LP) == hot, 80.0, -80.0)
    masked = torch.where(torch.rand(shape, generator=gen) < 0.4, float("-inf"), u)
    masked = torch.where(torch.arange(LP) == hot, u, masked)
    rows = [u, 100 + near, -100 + near, one_hot, torch.full(shape, 3.25), masked]
    out = rows[0].clone()
    for i, r in enumerate(rows):
        out = torch.where(kind == i, r, out)
    return out.contiguous()


@gpu
@pytest.mark.parametrize("levels,points", [
    ([(9, 13)], 4),                                      # L*P = 4
    ([(12, 20), (6, 10)], 4),                            # L*P = 8
    ([(8, 16), (16, 32), (32, 64)], 4),                  # L*P = 12
    ([(7, 9), (5, 3), (4, 4), (2, 2)], 4),               # L*P = 16
])
@pytest.mark.parametrize("variant", [0, 20, 2, "det"])
def test_extreme_and_degenerate_logits(pkg, oracle, levels, points, variant):
    """Logits up to +-80, rows near +100 and near -100, one-hot rows, rows of equal logits and rows with -inf
    entries: the fused forward and gradients (default backward, merging kernel, per-row kernel, deterministic
    path) match reference_composition -- torch's fp64 softmax: weight 0 and logit gradient 0 for a -inf entry,
    the rest normalised -- within FWD_ABS_TOL / GRAD_REL_TOL."""
    c = make_case(pkg, levels, 2, 4, points, True, seed=31)
    c["logits"] = _extreme_logits(tuple(c["logits"].shape), torch.Generator().manual_seed(len(levels)))
    _, _, _, glog, _ = _check_composition(pkg, oracle, c, variant, f"logits {levels}")
    ninf = torch.isneginf(c["logits"])
    assert ninf.any() and not glog.cpu()[ninf].any()


# ---------------------------------------------------------------- 4. decoder-style queries through the fused backward
def _decoder_case(pkg, levels, batch, heads, points, lq, shared_ref, seed):
    """Lq queries that are not the value pixels: reference points anywhere in the map (one set shared by the batch,
    batch stride 0, or one per image), offsets, logits and grad_output as make_case draws them."""
    c = make_case(pkg, levels, batch, heads, points, True, seed)
    gen = torch.Generator().manual_seed(seed + 1)
    L = len(levels)
    ref = torch.rand(1 if shared_ref else batch, lq, L, 2, generator=gen)
    rows = torch.randint(0, c["off"].shape[1], (lq,), generator=gen)
    return dict(c, ref=ref, off=c["off"][:, rows].contiguous(), logits=c["logits"][:, rows].contiguous(),
                grad_out=torch.randn(batch, lq, c["grad_out"].shape[-1], generator=gen))


LEVELS_DEC = [(8, 16), (16, 32), (32, 64)]
S_DEC = sum(h * w for h, w in LEVELS_DEC)


@gpu
@pytest.mark.parametrize("lq", [1, 301, S_DEC - 1])
@pytest.mark.parametrize("shared_ref", [True, False])
def test_decoder_queries_through_the_fused_backward(pkg, oracle, monkeypatch, lq, shared_ref):
    """Lq != S, reference points shared by the batch (ref_batch_stride 0) or per image: the fused forward and the
    three gradients of the default entry (the per-row kernel alone: one backward launch) and of the deterministic
    path with the batch processed in chunks of two images (ops.DETERMINISTIC_RECORD_LIMIT = two images' records
    + 1, which slices the per-image reference points ref[a:b]) match reference_composition within FWD_ABS_TOL /
    GRAD_REL_TOL; the chunked deterministic gradients equal the unchunked ones bit for bit."""
    c = _decoder_case(pkg, LEVELS_DEC, 5, 8, 4, lq, shared_ref, seed=lq)
    ref = reference_composition(oracle, c)
    *_, launches = _check_composition(pkg, oracle, c, 0, f"Lq={lq}", ref=ref)
    assert launches == 1
    whole = _fused_fwd_bwd(pkg, c, "det")
    monkeypatch.setattr(pkg.ops, "DETERMINISTIC_RECORD_LIMIT", 2 * _records_per_image(c["off"]) + 1)
    chunked = _check_composition(pkg, oracle, c, "det", f"Lq={lq} chunked", ref=ref)
    assert all(torch.equal(a, b) for a, b in zip(whole[1:4], chunked[1:4]))


# ---------------------------------------------------------------- 5. seeded random shapes
def test_random_shape_draws_cover_the_space():
    """CPU: the draws of test_fused_random_shapes_match_the_composition cover every L*P, Lq == S and Lq != S,
    shared and per-image reference points (batch > 1) and both offset spreads."""
    cases = _random_cases()
    assert {c["L"] * c["P"] for c in cases} == {4, 8, 12, 16}
    assert {c["lq"] is None for c in cases} == {True, False}
    assert {(c["shared"], c["batch"] > 1) for c in cases} >= {(True, True), (False, True)}
    assert {c["spread"] for c in cases} == {1.0, 5.0}


def _random_cases(count=12):
    rng = np.random.default_rng(808)
    points_for = {1: [4, 8, 12, 16], 2: [2, 4, 6, 8], 3: [4], 4: [1, 2, 3, 4]}
    cases = []
    for i in range(count):
        L = int(rng.integers(1, 5))
        cases.append(dict(L=L, P=int(rng.choice(points_for[L])),
                          levels=[(int(rng.integers(1, 41)), int(rng.integers(1, 41))) for _ in range(L)],
                          heads=int(rng.integers(1, 9)), batch=int(rng.integers(1, 4)),
                          lq=None if rng.random() < 0.5 else int(rng.integers(1, 400)),
                          shared=bool(rng.random() < 0.5), spread=float(rng.choice([1.0, 5.0])), seed=2000 + i))
    return cases


@gpu
def test_fused_random_shapes_match_the_composition(pkg, oracle):
    """The fused counterpart of test_random_shapes_match_oracle: 12 seeded shapes (L 1..4 with L*P in {4, 8, 12,
    16}, 1..8 heads, level sizes 1..40, batch 1..3, Lq == S or not, shared or per-image reference points, offsets
    spread x1 or x5 so that many points fall off the map) through whichever kernels the dispatcher picks: forward
    and the three gradients against reference_composition within FWD_ABS_TOL / GRAD_REL_TOL."""
    for i, r in enumerate(_random_cases()):
        if r["lq"] is None:
            c = make_case(pkg, r["levels"], r["batch"], r["heads"], r["P"], r["shared"], r["seed"])
        else:
            c = _decoder_case(pkg, r["levels"], r["batch"], r["heads"], r["P"], r["lq"], r["shared"], r["seed"])
        c["off"] = (c["off"] * r["spread"]).contiguous()
        _check_composition(pkg, oracle, c, 0, f"case {i}: {r}")


# ---------------------------------------------------------------- 6. full size
def _probe_says_local(off):
    """probe_points_stay_local<FUSED = true> (msda_common.cuh) on the host: the same 512 pseudo-random (image, query,
    head, point) samples; True when >= 75 % of their offsets are within 8 px in both axes (the merging kernel runs)."""
    N, Lq, M, L, P, _ = off.shape
    flat = off.reshape(N, Lq, M, L * P, 2)
    M32 = 0xffffffff
    inside = 0
    for i in range(512):
        h = (i * 2654435761 + 12345) & M32
        h ^= h >> 15
        h = (h * 2246822519) & M32
        h ^= h >> 13
        n = h % N
        h = (h * 1664525 + 1013904223) & M32
        q = (h >> 4) % Lq
        h = (h * 1664525 + 1013904223) & M32
        m, sp = (h >> 8) % M, (h >> 16) % (L * P)
        inside += bool((flat[n, q, m, sp].abs() <= 8).all())
    return 4 * inside >= 3 * 512


@gpu
@pytest.mark.parametrize("levels,batch", [
    ([(16, 32), (32, 64), (64, 128)], 8),                # configs[1]: the 512x1024 crop pyramid, batch 8
    ([(32, 64), (64, 128), (128, 256)], 2),              # the 1024x2048 pyramid, batch 2
])
def test_full_size_default_backward_matches_the_composition(pkg, oracle, levels, batch):
    """The fused forward and the default fused backward at full size, with model-like offsets: the location probe
    (replayed on the host) sends the backward to the merging kernel, over its persistent loop with many items per
    CTA and the double-buffered windows; forward and the three gradients against reference_composition within
    FWD_ABS_TOL / GRAD_REL_TOL."""
    c = make_case(pkg, levels, batch, 8, 4, True, seed=41)
    assert _probe_says_local(c["off"])
    *_, launches = _check_composition(pkg, oracle, c, 0, f"full size {levels} x{batch}")
    assert launches == 2                                # merging kernel + the per-row kernel it gates off
