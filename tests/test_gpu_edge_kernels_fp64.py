"""The edge-side kernels of the training step, one entry point at a time, against fp64 on one GPU.

The node side has its own file (``test_gpu_node_kernels_fp64.py``).  This one holds the fused edge scorer (training
form ``edge_scorer_train.cu``, inference form ``edge_scorer_tc.cu``), the chunked scorer's hand-off to the nodes,
the sorted-segment aggregation family and ``gcn_norm`` of ``gcn.cu``, and the cosine / dot pair decoders.  Each case
runs at the shapes where a schedule changes: tiles per CTA of the persistent scorer (the dW2 accumulator is drained
every ``kG3Flush = 4`` tiles), partial last tiles, the aggregation's 32-row chunks and UNROLL groups, every
lanes-per-row variant and the wide kernel, rows past 2^31 bytes.

Two kinds of check.

* Exact grid, bit-exact.  Inputs are small dyadic numbers (a few significant bits), chosen so that every product and
  every partial sum a kernel can form is an fp32 number: then neither the summation order nor the tensor core's
  truncating accumulation changes the result, and it must equal the fp64 reference bit for bit.  This is what
  catches schedule faults: a lost tile, an accumulator drained twice or never, the wrong parity buffer, a row closed
  early.  Every such case asserts its own precondition from the fp64 reference: each output is a multiple of its
  grid step, and ``sum |term| / step < 2^22`` for every output (``EXACT_UNITS``).
* Random values against condition-aware bars: ``|got - ref| <= rel * sum |term|`` per element, with ``sum |term|``
  carried through the layers (the error a pre-activation brings in is propagated like its value); where there is a
  plain-fp32 yardstick its error is reported beside ours.

``-s`` prints one table per case before any bar is checked.  Bars and figures: ``profiles/r09_edge_kernels_fp64.log``
(one B200) and DESIGN.md section 2.
"""
import ctypes as C
import zlib
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as tnf

from tests.helpers import Table, bits, check, lib, nan_fill, plain_fp32, ptr, ratio, scale_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NUM_SMS = 148
BM = 128                                       # edges per scorer tile
D = 64                                         # scorer width
EXACT_UNITS = 2.0 ** 22                        # exact-grid precondition: sum |term| / step below this, per output
# Bars (measured on one B200 in profiles/r09_edge_kernels_fp64.log; the figures are in DESIGN.md section 2)
SC_REL = 4e-7                                  # scorer, random values: |got - ref| <= SC_REL * sum |term| (measured
                                               # at most 0.29 of it, i.e. 1.1e-7 sum |term|)
LOSS_REL = 1e-7                                # loss sums, of sum |term| (fp32 per-thread sums across tiles): 2.3e-9
PROB_ULP = 3.0                                 # sigmoid of the kernel's own logit, in fp32 ulps: 2.23 measured
AGG_REL = 1e-6                                 # aggregation, random values: per element, of sum |val x|: 0.55 of it
                                               # (the plain-fp32 index_add_ 0.50)
ELU_ULP = 1.0                                  # aggregation ELU (expm1f) against fp64 ELU of the exact pre-activation:
                                               # 0.88 ulp measured
DIS_ULP = 2.0                                  # gcn_norm: dis against 1 / sqrt(sum w) in fp64: 1.70 ulp weighted, 0.79
                                               # unweighted (deg rounded to fp32 as PyG does, then 1.0f / sqrtf)
PAIR_REL = 5e-7                                # pair decoders: per element, of the propagated sum |term|: 0.26 of it
# the C3-size scorer case keeps test_gpu_c3_fp64.py's bars: scale-relative, dW2 at 5e-5 (1e7 cancelling products),
# each at most 4x the plain-fp32 evaluation's error.  The floor of that ratio rule is bar / 3 here, not bar / 5: db2
# is a per-thread fp32 running sum over 528 tiles, measured 2.2-2.5e-6 where torch's pairwise fp32 sum gives 5e-7.
C3_LOGIT, C3_GRAD, C3_DW2, C3_FP32, C3_FLOOR = 2e-6, 1e-5, 5e-5, 4.0, 3.0


def ops():
    from pangnn_b200 import ops as o
    return o


def gen(*seed):
    return torch.Generator(device=DEV).manual_seed(zlib.crc32(repr(seed).encode()))


def dyadic(shape, lo, hi, exp, g, density=1.0):
    """fp32 integers in [lo, hi] times 2^exp, each zero with probability 1 - density."""
    v = torch.randint(lo, hi + 1, shape, generator=g, device=DEV).float()
    if density < 1.0:
        v *= torch.rand(shape, generator=g, device=DEV) < density
    return v * 2.0 ** exp


def on_grid(t, step):
    q = t.double() / step
    return bool(torch.equal(q, torch.round(q)))


def exact_pre(name, ref, mag, step):
    """Precondition of a bit-exact case: ``ref`` on its grid and sum |term| / step < EXACT_UNITS.  -> units."""
    units = float(mag.max()) / step if mag.numel() else 0.0
    assert on_grid(ref, step), f"{name}: the fp64 reference is not a multiple of its grid step {step:g}"
    assert units < EXACT_UNITS, f"{name}: sum |term| / step = {units:.3g} >= 2^22; the grid is too fine for exactness"
    return units


def same(got, ref):
    """fp32 ``got`` equal in value to the fp64 ``ref`` (+0.0 == -0.0)."""
    return bool(torch.equal(got.double(), ref.double()))


def ulp32(x):
    """fp32 ulp at |x| (fp64 tensor), for normal numbers."""
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(x), (e - 24).to(torch.int32))


# ================================================================================================
# A. the fused edge scorer
# ================================================================================================
TRAIN_E = {"E1": 1, "E127": 127, "E128": 128, "E129": 129, "E147t69": 147 * BM + 69}
for _t in range(1, 10):
    TRAIN_E[f"T{_t}"] = NUM_SMS * BM * _t - 59                 # every CTA T tiles, the last one holds 69 edges
    TRAIN_E[f"T{_t}p1"] = NUM_SMS * BM * _t + 1                # CTA 0 T + 1 tiles, the last one holds one edge
FWD_CAP = 2 * NUM_SMS
FWD_E = {"E1": 1, "E129": 129, "E295t1": 295 * BM + 1}
for _t in (1, 2, 3):
    FWD_E[f"T{_t}"] = FWD_CAP * BM * _t - 59
    FWD_E[f"T{_t}p1"] = FWD_CAP * BM * _t + 1


def scorer_graph(E, N, order, g):
    """int32 (src, dst) of E edges on N nodes with duplicate edges and self-loops, in canonical (src, dst) order or
    shuffled."""
    src = torch.randint(0, N, (E,), generator=g, device=DEV)
    dst = torch.randint(0, N, (E,), generator=g, device=DEV)
    k = E // 16
    src[:k], dst[:k] = src[k:2 * k], dst[k:2 * k]             # duplicates
    dst[2 * k:3 * k] = src[2 * k:3 * k]                       # src == dst
    key = torch.argsort(src * N + dst) if order == "canonical" else torch.randperm(E, generator=g, device=DEV)
    return src[key].int().contiguous(), dst[key].int().contiguous()


def grid_params(g, skip=True, w3_scale=1.0):
    """Scorer parameters on the exact grid (see ``EXACT_STEPS``)."""
    w3 = (torch.randint(1, 3, (D,), generator=g, device=DEV).float() * 0.5 *
          (torch.randint(0, 2, (D,), generator=g, device=DEV).float() * 2 - 1)) * w3_scale
    return SimpleNamespace(
        w1c=dyadic((D,), -2, 2, -2, g) if skip else None, b1=dyadic((D,), -2, 2, -2, g),
        w2=dyadic((D, D), -2, 2, -2, g, density=0.125).contiguous(), b2=dyadic((D,), -8, 8, -5, g),
        w3=w3.view(1, D).contiguous(), b3=dyadic((1,), -16, 16, -6, g))


def random_params(g, skip=True):
    r = lambda *s, sc=1.0: torch.randn(*s, generator=g, device=DEV) * sc
    return SimpleNamespace(w1c=r(D, sc=0.3) if skip else None, b1=r(D, sc=0.2), w2=r(D, D, sc=D ** -0.5),
                           b2=r(D, sc=0.2), w3=r(1, D, sc=D ** -0.5), b3=r(1, sc=0.2))


# grid steps: pq, b1 2^-2; w1c 2^-2 x skip 2^-1 -> a1 2^-3; W2 2^-2 -> a2 2^-5, b2 2^-5; w3 2^-1 -> z 2^-6;
# W2' = w3 W2 2^-3 -> g 2^-3; dz = dlogits (2^-1) * scale (0.5) 2^-2
E_DZ = -2
EXACT_STEPS = {"a1": 2.0 ** -3, "pre2": 2.0 ** -5, "logits": 2.0 ** -6, "g": 2.0 ** -3, "da1": 2.0 ** (E_DZ - 3),
               "dW2": 2.0 ** (E_DZ - 4), "db2": 2.0 ** (E_DZ - 1), "dw3": 2.0 ** (E_DZ - 5), "db3": 2.0 ** E_DZ,
               "db1": 2.0 ** (E_DZ - 3), "dw1c": 2.0 ** (E_DZ - 4)}
GRAD_NAMES = ("dW2", "db2", "dw3", "db3", "db1", "dw1c")


def scorer_ref(pq, src, dst, sk, P, dz=None, y=None, pw=1.0, scale=1.0, dt=torch.float64, mags="prop"):
    """The scorer from its definition in ``dt`` on the same fp32 inputs: logits, loss sum, da1 and the six small
    gradients, with the upstream gradient ``dz`` given or from BCE-with-logits(pos_weight) * scale (``y < 0``: no
    label, no loss term, dz = 0).  ``mags``: sum |term| of every output, either "plain" (the terms' own values: the
    exact-grid precondition) or "prop", carried through the layers for the random-value bars (a1's sum |term| in
    place of |r1|, and so on; for the fused loss also the error a logit error brings into dz)."""
    c = lambda t: t.to(dt)
    s, d = src.long(), dst.long()
    W2, w3, b2 = c(P.w2), c(P.w3).reshape(-1), c(P.b2)
    a1 = c(pq[s, :D]) + c(pq[d, D:]) + c(P.b1)
    if sk is not None:
        a1 += c(sk)[:, None] * c(P.w1c)
    m1 = (a1 > 0).to(dt)
    r1 = a1 * m1
    pre2 = r1 @ W2.t() + b2
    m2 = (pre2 > 0).to(dt)
    r2 = pre2 * m2
    z = r2 @ w3 + c(P.b3)
    out = {"a1": a1, "pre2": pre2, "logits": z, "m1": m1, "m2": m2}
    lab = None
    if dz is None:
        yy = c(y)
        lab = (yy >= 0).to(dt)
        sg = torch.sigmoid(z)
        dz = lab * ((pw * yy + 1 - yy) * sg - pw * yy) * scale
        term = (1 - yy) * z + (1 + (pw - 1) * yy) * (torch.log1p(torch.exp(-z.abs())) + (-z).clamp_min(0))
        out["loss"] = (lab * term).sum().reshape(1)
    else:
        dz = c(dz)
    W2p = w3[:, None] * W2
    g = m2 @ W2p
    da1 = dz[:, None] * g * m1
    pm = dz[:, None] * m2
    out.update(dz=dz, g=g, da1=da1, dW2=w3[:, None] * (pm.t() @ r1), db2=w3 * pm.sum(0),
               dw3=(dz[:, None] * r2).sum(0).view(1, D), db3=dz.sum().reshape(1), db1=da1.sum(0),
               dw1c=(da1 * c(sk)[:, None]).sum(0) if sk is not None else torch.zeros(D, dtype=dt, device=DEV))
    if not mags:
        return out
    prop = mags == "prop"
    A1 = c(pq[s, :D]).abs() + c(pq[d, D:]).abs() + c(P.b1).abs()
    if sk is not None:
        A1 += (c(sk)[:, None] * c(P.w1c)).abs()
    P1 = A1 * m1 if prop else r1
    A2 = P1 @ W2.abs().t() + b2.abs()
    P2 = A2 * m2 if prop else r2
    Z = P2 @ w3.abs() + c(P.b3).abs()
    dzm = dz.abs()
    if lab is not None and prop:
        dzm = dzm + lab * scale * ((pw * yy + 1 - yy) * (sg + 0.25 * Z) + pw * yy)
    if lab is not None:
        out["loss mag"] = (lab * (term.abs() + (1 + (pw - 1) * yy) * Z)).sum().reshape(1)
    G = m2 @ W2p.abs()
    DA1 = dzm[:, None] * G * m1 if prop else da1.abs()
    pmm = dzm[:, None] * m2
    out["mag"] = {"a1": A1, "pre2": A2, "logits": Z, "g": G, "da1": DA1,
                  "dW2": w3.abs()[:, None] * (pmm.t() @ P1), "db2": w3.abs() * pmm.sum(0),
                  "dw3": (dzm[:, None] * P2).sum(0).view(1, D), "db3": dzm.sum().reshape(1), "db1": DA1.sum(0),
                  "dw1c": (DA1 * c(sk).abs()[:, None]).sum(0) if sk is not None else torch.zeros(D, dtype=dt,
                                                                                                  device=DEV)}
    return out


def call_bwd(pq, src, dst, sk, P, E, *, dlogits=None, y=None, pw=1.0, scale=1.0, da1=None, grads=None,
             logits=None, loss=None):
    o, lb = ops(), lib()
    ws = o._ws(lb.pangnn_edge_score_workspace_bytes(E), DEV)
    check(lb.pangnn_edge_score_bwd(ptr(pq), ptr(src), ptr(dst), ptr(sk), ptr(P.w1c), ptr(P.b1), ptr(P.w2),
                                   ptr(P.b2), ptr(P.w3), ptr(P.b3), E, ptr(dlogits), ptr(y), float(pw), float(scale),
                                   ptr(da1), ptr(grads), ptr(logits), ptr(loss), ptr(ws), ws.numel(), o._stream()),
          "edge_score_bwd")


def call_predict(pq, src, dst, sk, P, E, th, logits=None, prob=None, pred=None):
    o = ops()
    check(lib().pangnn_edge_score_predict(ptr(pq), ptr(src), ptr(dst), ptr(sk), ptr(P.w1c), ptr(P.b1), ptr(P.w2),
                                          ptr(P.b2), ptr(P.w3), ptr(P.b3), E, float(th), ptr(logits), ptr(prob),
                                          ptr(pred), o._stream()), "edge_score_predict")


def call_fwd(pq, src, dst, sk, P, E, logits=None, y=None, pw=1.0, loss=None):
    o, lb = ops(), lib()
    ws = o._ws(lb.pangnn_edge_score_workspace_bytes(E), DEV)
    check(lb.pangnn_edge_score_fwd(ptr(pq), ptr(src), ptr(dst), ptr(sk), ptr(P.w1c), ptr(P.b1), ptr(P.w2),
                                   ptr(P.b2), ptr(P.w3), ptr(P.b3), E, ptr(y), float(pw), ptr(logits), ptr(loss),
                                   ptr(ws), ws.numel(), o._stream()), "edge_score_fwd")


def grads_of(buf):
    return ops().scorer_grads(buf)._asdict()


def tiles_note(E, cap):
    tiles = -(-E // BM)
    grid = min(tiles, cap)
    hi = -(-tiles // grid)
    return f"{tiles} tiles, {grid} CTAs, {hi} tiles on CTA 0, D3 holds {(hi - 1) % 4 + 1} at the end"


def scorer_inputs_exact(E, order, g, skip=True, N=None):
    N = N or max(E // 3, 50)
    src, dst = scorer_graph(E, N, order, g)
    pq = dyadic((N, 2 * D), -2, 2, -2, g)
    sk = dyadic((E,), 0, 2, -1, g) if skip else None
    return pq, src, dst, sk, grid_params(g, skip)


def signed_dyadic(shape, exp, g, density):
    """+-1 or +-2 times 2^exp, zero with probability 1 - density."""
    v = torch.randint(1, 3, shape, generator=g, device=DEV).float() * \
        (torch.randint(0, 2, shape, generator=g, device=DEV).float() * 2 - 1)
    return v * (torch.rand(shape, generator=g, device=DEV) < density) * 2.0 ** exp


def check_train_exact(t, E, pq, src, dst, sk, P, g):
    """External-dlogits form on the exact grid: logits, da1 and the six gradients bit-exact; sentinel rows past E
    untouched; grads fully written."""
    dl = signed_dyadic((E,), -1, g, density=1.0 if E < 1000 else 0.25)
    scale = 0.5
    da1, logits, grads = nan_fill(E + BM, D), nan_fill(E + BM), nan_fill(ops().NGRADS)
    fill_da1, fill_z = bits(da1).clone(), bits(logits).clone()
    call_bwd(pq, src, dst, sk, P, E, dlogits=dl, scale=scale, da1=da1, grads=grads, logits=logits)
    ref = scorer_ref(pq, src, dst, sk, P, dz=dl * scale, mags="plain")
    got = {"logits": logits[:E], "da1": da1[:E], **grads_of(grads)}
    for name in ("a1", "pre2", "g"):
        t.add(f"precondition {name}", exact_pre(name, ref[name], ref["mag"][name], EXACT_STEPS[name]), "-")
    for name in ("logits", "da1") + GRAD_NAMES:
        units = exact_pre(name, ref[name], ref["mag"][name], EXACT_STEPS[name])
        ok = same(got[name], ref[name])
        nbad = int((got[name].double() != ref[name]).sum())
        t.add(name, units, nbad, ok=ok, why=f"{nbad} elements differ from fp64 (max |d| "
              f"{float((got[name].double() - ref[name]).abs().max()):.3e})")
    tail = torch.equal(bits(da1)[E:], fill_da1[E:]) and torch.equal(bits(logits)[E:], fill_z[E:])
    t.add("rows past E untouched", "-", "-", ok=tail, why="a store past row E - 1")


@pytest.mark.parametrize("order", ["canonical", "shuffled"])
@pytest.mark.parametrize("eid", list(TRAIN_E))
def test_scorer_train_exact_grid(eid, order):
    """``pangnn_edge_score_bwd`` with external dlogits on the exact grid, at 1..9 tiles per CTA with a partial last
    tile of 69 edges or of one edge (CTA 0 one tile more), and below one full wave."""
    E = TRAIN_E[eid]
    g = gen("train_exact", eid, order)
    pq, src, dst, sk, P = scorer_inputs_exact(E, order, g, skip=True)
    t = Table(f"scorer train, exact grid, {eid}: E = {E}, {order}; {tiles_note(E, NUM_SMS)}",
              ["units", "differ"])
    check_train_exact(t, E, pq, src, dst, sk, P, g)
    t.check()


def test_scorer_train_exact_grid_rows_past_2_31_bytes():
    """Endpoints above row 4.19e6 of pq (N = 4.5e6, 512-byte rows): the gathers' 64-bit offsets, in the training
    and both inference kernels."""
    g = gen("train_far")
    N, lo, E = 4_500_000, 4_194_400, NUM_SMS * BM * 2 + 1
    pq = torch.zeros(N, 2 * D, device=DEV)
    pq[lo:] = dyadic((N - lo, 2 * D), -2, 2, -2, g)
    src = torch.randint(lo, N, (E,), generator=g, device=DEV, dtype=torch.int32)
    dst = torch.randint(lo, N, (E,), generator=g, device=DEV, dtype=torch.int32)
    sk = dyadic((E,), 0, 2, -1, g)
    P = grid_params(g)
    t = Table(f"scorer, exact grid, rows past 2^31 bytes: N = {N}, E = {E}", ["units", "differ"])
    check_train_exact(t, E, pq, src, dst, sk, P, g)
    ref = scorer_ref(pq, src, dst, sk, P, dz=torch.zeros(E, device=DEV), mags=None)
    for name, fn in (("predict", lambda z: call_predict(pq, src, dst, sk, P, E, 0.5, logits=z)),
                     ("fwd", lambda z: call_fwd(pq, src, dst, sk, P, E, logits=z))):
        z = nan_fill(E)
        fn(z)
        t.add(f"logits ({name})", "-", int((z.double() != ref["logits"]).sum()), ok=same(z, ref["logits"]),
              why=f"{name} logits differ")
    t.check()


def random_train_inputs(E, order, g, skip):
    N = max(E // 3, 50)
    src, dst = scorer_graph(E, N, order, g)
    pq = torch.randn(N, 2 * D, generator=g, device=DEV) * 0.5
    sk = torch.rand(E, generator=g, device=DEV) * 80 + 1 if skip else None
    return pq, src, dst, sk, random_params(g, skip)


def away_from_kinks(ref):
    """Edges whose pre-activations are all farther than 1e-4 of their sum |term| from 0 (a mask flip there is a
    legitimate fp32 difference; those edges are given no label or no upstream gradient)."""
    m = ref["mag"]
    return (ref["a1"].abs() > 1e-4 * m["a1"]).all(1) & (ref["pre2"].abs() > 1e-4 * m["pre2"]).all(1)


@pytest.mark.parametrize("order", ["canonical", "shuffled"])
@pytest.mark.parametrize("eid", list(TRAIN_E))
def test_scorer_train_fused_loss_random(eid, order):
    """The fused BCE form on random values: labelled and unlabelled (y = -1) edges in every tile, a non-zero preset
    ``loss_sum`` that must come back plus the sum, unlabelled rows of da1 exactly zero (+0.0 or -0.0), sentinel rows
    past E."""
    E = TRAIN_E[eid]
    g = gen("train_fused", eid, order)
    skip = order == "canonical"
    pq, src, dst, sk, P = random_train_inputs(E, order, g, skip)
    pw = 2.7
    y0 = (torch.rand(E, generator=g, device=DEV) < 0.3).float()
    pre = scorer_ref(pq, src, dst, sk, P, y=y0, pw=pw)
    unl = (torch.rand(E, generator=g, device=DEV) < 0.25) | ~away_from_kinks(pre)
    y = torch.where(unl, -1.0, y0)
    n_lab = max(int((~unl).sum()), 1)
    scale = 1.0 / n_lab
    ref = scorer_ref(pq, src, dst, sk, P, y=y, pw=pw, scale=scale)
    with plain_fp32():
        r32 = scorer_ref(pq, src, dst, sk, P, y=y, pw=pw, scale=scale, dt=torch.float32, mags=None)
    da1, logits, grads = nan_fill(E + BM, D), nan_fill(E + BM), nan_fill(ops().NGRADS)
    fill_da1, fill_z = bits(da1).clone(), bits(logits).clone()
    preset = 12345.678
    loss = torch.full((1,), preset, dtype=torch.float64, device=DEV)
    call_bwd(pq, src, dst, sk, P, E, y=y, pw=pw, scale=scale, da1=da1, grads=grads, logits=logits, loss=loss)
    got = {"logits": logits[:E], "da1": da1[:E], **grads_of(grads)}
    t = Table(f"scorer train, fused loss, random, {eid}: E = {E}, {order}, skip {skip}, {int(unl.sum())} unlabelled;"
              f" {tiles_note(E, NUM_SMS)}", ["err/bar", "scale err", "fp32 scale"])
    for name in ("logits", "da1") + GRAD_NAMES:
        ref_v, mag = ref[name], ref["mag"][name]
        r = ratio((got[name].double() - ref_v).abs(), SC_REL * mag)
        t.add(name, r, scale_err(got[name], ref_v), scale_err(r32[name], ref_v), ok=r <= 1.0,
              why=f"{name} error {r:.2f} x bar")
    dl = float(loss) - preset
    r = abs(dl - float(ref["loss"])) / (LOSS_REL * float(ref["loss mag"]) + 2.0 ** -40 * abs(preset))
    t.add("loss_sum - preset", r, abs(dl - float(ref["loss"])) / abs(float(ref["loss"])), "-", ok=r <= 1.0,
          why=f"loss sum error {r:.2f} x bar")
    z_unl = da1[:E][unl]
    # exactly zero; the sign is that of 0 * g, as in torch's autograd of a zero upstream gradient (-0.0 where g < 0)
    t.add("unlabelled da1: non-zero, -0.0", int((z_unl != 0).sum()), int((bits(z_unl) == -2 ** 31).sum()), "-",
          ok=bool((z_unl == 0).all()), why="an unlabelled row of da1 is not zero")
    tail = torch.equal(bits(da1)[E:], fill_da1[E:]) and torch.equal(bits(logits)[E:], fill_z[E:])
    t.add("rows past E untouched", "-", "-", "-", ok=tail, why="a store past row E - 1")
    t.check()


def test_scorer_empty_edge_list():
    """E = 0: ``bwd`` zeroes grads and writes nothing else; ``fwd`` and ``predict`` write nothing; a preset
    loss_sum is left as it is."""
    g = gen("empty")
    P = grid_params(g)
    pq = dyadic((10, 2 * D), -2, 2, -2, g)
    src = dst = torch.zeros(0, dtype=torch.int32, device=DEV)
    da1, logits, grads, prob = nan_fill(BM, D), nan_fill(BM), nan_fill(ops().NGRADS), nan_fill(BM)
    pred = nan_fill(BM).view(torch.int32)
    fills = [bits(b).clone() for b in (da1, logits, prob, pred)]
    loss = torch.full((1,), 3.25, dtype=torch.float64, device=DEV)
    y = torch.zeros(BM, device=DEV)
    call_bwd(pq, src, dst, None, P, 0, y=y, da1=da1, grads=grads, logits=logits, loss=loss)
    call_fwd(pq, src, dst, None, P, 0, logits=logits, y=y, loss=loss)
    call_predict(pq, src, dst, None, P, 0, 0.5, logits=logits, prob=prob, pred=pred)
    torch.cuda.synchronize()
    assert bool((bits(grads) == 0).all()), "grads not zeroed (+0.0) at E = 0"
    for b, f in zip((da1, logits, prob, pred), fills):
        assert torch.equal(bits(b), f), "a buffer was written at E = 0"
    assert float(loss) == 3.25


# ------------------------------------------------------------------------------------------------
# scorer at the benchmark's size, T = 0 mod 4 (a full D3 chain left at the CTA epilogue)
# ------------------------------------------------------------------------------------------------
def test_scorer_train_random_at_c3_size_full_chain():
    """E = 148 * 128 * 528 - 59 (1.0e7 edges, 528 tiles per CTA: D3 holds a full chain of 4 at the epilogue), both
    forms, against fp64 and the plain-fp32 evaluation of the same formulas with test_gpu_c3_fp64.py's bars: logits
    2e-6, loss 2e-6, gradients 1e-5 but dW2 5e-5, each at most 4x the fp32 evaluation's error (floor bar / 5)."""
    from oracle.params import make_state_dict
    E, N = NUM_SMS * BM * 528 - 59, 1_000_000
    g = gen("c3_full_chain")
    src, dst = scorer_graph(E, N, "canonical", g)
    sd = {k: v.to(DEV) for k, v in make_state_dict(skip_connections=True).items()}
    P = SimpleNamespace(w1c=sd["mlp.0.weight"][:, 2 * D].contiguous(), b1=sd["mlp.0.bias"], w2=sd["mlp.2.weight"],
                        b2=sd["mlp.2.bias"], w3=sd["mlp.4.weight"], b3=sd["mlp.4.bias"])
    pq = torch.randn(N, 2 * D, generator=g, device=DEV)
    sk = torch.rand(E, generator=g, device=DEV) * 80 + 1
    y = (torch.rand(E, generator=g, device=DEV) < 0.1).float()
    pw, scale = 9.0, 1.0 / E
    z0 = nan_fill(E)
    call_fwd(pq, src, dst, sk, P, E, logits=z0)
    dz_ext = ((pw * y + 1 - y) * torch.sigmoid(z0) - pw * y) * scale * (torch.rand(E, generator=g, device=DEV) + 0.5)
    del z0
    t = Table(f"scorer train at E = {E} (N = {N}); {tiles_note(E, NUM_SMS)}", ["scale err", "fp32 scale", "bar"])
    da1, grads = torch.empty(E, D, device=DEV), torch.empty(ops().NGRADS, device=DEV)
    for form in ("fused loss", "external dlogits"):
        kw = dict(y=y, pw=pw, scale=scale) if form == "fused loss" else dict(dz=dz_ext)
        ref = scorer_ref(pq, src, dst, sk, P, mags=None, **kw)
        ref.pop("g")
        with plain_fp32():
            r32 = scorer_ref(pq, src, dst, sk, P, dt=torch.float32, mags=None, **kw)
        # da1 only: edges whose pre-activations are all farther than 1e-5 from a ReLU kink (test_gpu_c3_fp64.py)
        ok_e = (ref["a1"].abs().min(1).values > 1e-5) & (ref["pre2"].abs().min(1).values > 1e-5)
        got = {}
        if form == "fused loss":
            logits, loss = torch.empty(E, device=DEV), torch.zeros(1, dtype=torch.float64, device=DEV)
            call_bwd(pq, src, dst, sk, P, E, y=y, pw=pw, scale=scale, da1=da1, grads=grads, logits=logits, loss=loss)
            got.update(logits=logits, loss=loss)
        else:
            call_bwd(pq, src, dst, sk, P, E, dlogits=dz_ext, da1=da1, grads=grads)
        got.update(grads_of(grads))
        bars = {"logits": C3_LOGIT, "loss": C3_LOGIT, "dW2": C3_DW2}
        for name, v in got.items():
            bar = bars.get(name, C3_GRAD)
            e, e32 = scale_err(v, ref[name]), scale_err(r32[name], ref[name])
            t.add(f"{name} ({form})", e, e32, bar, ok=e <= bar and e <= max(C3_FP32 * e32, bar / C3_FLOOR),
                  why=f"{name}: {e:.3e} (fp32 {e32:.3e}, bar {bar:.0e})")
        e, e32 = scale_err(da1[ok_e], ref["da1"][ok_e]), scale_err(r32["da1"][ok_e], ref["da1"][ok_e])
        t.add(f"da1 off kinks ({form})", e, e32, C3_GRAD,
              ok=e <= C3_GRAD and e <= max(C3_FP32 * e32, C3_GRAD / C3_FLOOR),
              why=f"da1: {e:.3e} (fp32 {e32:.3e})")
        del ref, r32, ok_e
        torch.cuda.empty_cache()
    t.check()


# ------------------------------------------------------------------------------------------------
# inference form: fwd / predict
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("eid", list(FWD_E))
def test_scorer_predict_exact_grid(eid):
    """``predict``: logits bit-exact on the exact grid; probabilities within PROB_ULP of the fp64 sigmoid of the
    kernel's own logits; ``pred == (prob >= th)`` at th in {0, 0.37, 0.5, 1}, at prob[k] and the floats either side;
    every non-empty subset of the three outputs writes exactly those; ``fwd`` adds its loss to a preset loss_sum."""
    E = FWD_E[eid]
    g = gen("predict", eid)
    pq, src, dst, sk, P = scorer_inputs_exact(E, "shuffled", g, skip=eid != "E129")
    # wider logits than the training grid (w3 x 8): probabilities near 0 and 1 as well
    P.w3 = P.w3 * 8
    ref = scorer_ref(pq, src, dst, sk, P, dz=torch.zeros(E, device=DEV), mags="plain")
    t = Table(f"scorer predict, exact grid, {eid}: E = {E}; {tiles_note(E, FWD_CAP)}", ["value", "ok"])
    exact_pre("logits", ref["logits"], ref["mag"]["logits"], EXACT_STEPS["logits"])
    z, p, pr = nan_fill(E + BM), nan_fill(E + BM), nan_fill(E + BM).view(torch.int32)
    fills = [bits(b).clone() for b in (z, p, pr)]
    call_predict(pq, src, dst, sk, P, E, 0.5, logits=z, prob=p, pred=pr)
    t.add("logits bit-exact", int((z[:E].double() != ref["logits"]).sum()), same(z[:E], ref["logits"]),
          ok=same(z[:E], ref["logits"]), why="logits differ from fp64")
    s64 = torch.sigmoid(z[:E].double())
    ulps = float(((p[:E].double() - s64).abs() / ulp32(s64)).max())
    t.add("prob: max ulps", ulps, ulps <= PROB_ULP, ok=ulps <= PROB_ULP, why=f"prob {ulps:.2f} ulp from fp64")
    t.add("prob range [min, max]", f"{float(p[:E].min()):.2e}", f"{float(p[:E].max()):.7f}")
    full = [z[:E].clone(), p[:E].clone(), pr[:E].clone()]
    tails = all(torch.equal(bits(b)[E:], f[E:]) for b, f in zip((z, p, pr), fills))
    t.add("rows past E untouched", "-", tails, ok=tails, why="a store past row E - 1")
    # thresholds
    prob = full[1]
    ks = torch.linspace(0, E - 1, 5, device=DEV).long()
    ths = [0.0, 0.37, 0.5, 1.0]
    for k in ks.tolist():
        v = prob[k:k + 1]
        ths += [float(v), float(torch.nextafter(v, torch.zeros_like(v))), float(torch.nextafter(v, v + 1))]
    bad = []
    for th in ths:
        q = nan_fill(E).view(torch.int32)
        call_predict(pq, src, dst, sk, P, E, th, pred=q)
        if not torch.equal(q, (prob >= torch.tensor(th, dtype=torch.float32, device=DEV)).to(torch.int32)):
            bad.append(th)
    t.add(f"pred == (prob >= th), {len(ths)} th", len(bad), not bad, ok=not bad, why=f"thresholds {bad[:4]}")
    # NULL outputs
    for mask in range(1, 8):
        outs = [nan_fill(E + BM) if mask & 1 else None, nan_fill(E + BM) if mask & 2 else None,
                nan_fill(E + BM).view(torch.int32) if mask & 4 else None]
        fl = [None if b is None else bits(b).clone() for b in outs]
        call_predict(pq, src, dst, sk, P, E, 0.5, *outs)
        ok = all(b is None or (torch.equal(bits(b)[:E], bits(f)) and torch.equal(bits(b)[E:], f0[E:]))
                 for b, f, f0 in zip(outs, full, fl))
        t.add(f"outputs {'l' if mask & 1 else '-'}{'p' if mask & 2 else '-'}{'d' if mask & 4 else '-'}", "-", ok,
              ok=ok, why="an output subset writes other than its own outputs")
    # fwd: logits as predict's, loss added to a preset loss_sum
    y = (torch.rand(E, generator=g, device=DEV) < 0.4).float()
    zf = nan_fill(E)
    loss = torch.full((1,), -7.5, dtype=torch.float64, device=DEV)
    call_fwd(pq, src, dst, sk, P, E, logits=zf, y=y, pw=3.0, loss=loss)
    zz = ref["logits"]
    term = (1 - y.double()) * zz + (1 + 2.0 * y.double()) * (torch.log1p(torch.exp(-zz.abs())) + (-zz).clamp_min(0))
    r = abs(float(loss) + 7.5 - float(term.sum())) / (LOSS_REL * float(term.abs().sum()))
    t.add("fwd: logits as predict", "-", torch.equal(bits(zf), bits(full[0])), ok=torch.equal(bits(zf), bits(full[0])),
          why="fwd logits differ from predict's")
    t.add("fwd: loss_sum - preset err/bar", r, r <= 1.0, ok=r <= 1.0, why=f"fwd loss {r:.2f} x bar")
    t.check()


# ------------------------------------------------------------------------------------------------
# scorer -> nodes: the chunked form of EdgeScoreBCEPQFn
# ------------------------------------------------------------------------------------------------
def test_chunked_scorer_dpq_bit_exact(monkeypatch):
    """``EdgeScoreBCEPQFn`` in its chunked form (runs of at most 10 000 edges, one source of 15 000 edges in a run of
    its own) gives a dpq bit-identical to the single launch and to fp64, in both halves.  The fused loss gives exact
    dz only where sigmoid(z) rounds to 0 or 1: logits on the grid are mostly |z| >= 100 (w3 x 1024), and edges
    with a smaller |z| or with sigmoid(z) = 0 and y = 0 get no label."""
    o = ops()
    g = gen("chunked")
    N = 6000
    deg = torch.randint(0, 25, (N,), generator=g, device=DEV)
    deg[17] = 15_000
    src = torch.repeat_interleave(torch.arange(N, device=DEV), deg)
    E = src.numel()
    dst = torch.randint(0, N, (E,), generator=g, device=DEV)
    key = torch.argsort(src * N + dst)
    ei = torch.stack((src[key], dst[key])).contiguous()
    pq = dyadic((N, 2 * D), -2, 2, -2, g)
    sk = dyadic((E,), 0, 2, -1, g)
    W3S = 1024.0
    P = grid_params(g, w3_scale=W3S)
    pw, scale = 2.0, 1.0 / 8
    y0 = (torch.rand(E, generator=g, device=DEV) < 0.5).float()
    ei32 = (ei[0].int(), ei[1].int())
    z64 = scorer_ref(pq, ei32[0], ei32[1], sk, P, dz=torch.zeros(E, device=DEV), mags=None)["logits"]
    P.b3 = torch.round(P.b3 - z64.median()).float().view(1)          # centre the logits: both signs of dz
    z64 = scorer_ref(pq, ei32[0], ei32[1], sk, P, dz=torch.zeros(E, device=DEV), mags=None)["logits"]
    y = torch.where((z64.abs() < 100) | ((z64 < 0) & (y0 == 0)), -1.0, y0)
    ref = scorer_ref(pq, ei32[0], ei32[1], sk, P, y=y, pw=pw, scale=scale, mags="plain")
    exact_pre("logits", ref["logits"], ref["mag"]["logits"], EXACT_STEPS["logits"])
    dz_units = ref["dz"] / scale
    assert on_grid(dz_units, 1.0) and int((ref["dz"] > 0).sum()) > 100 and int((ref["dz"] < 0).sum()) > 100
    rows_s, rows_d = ei[0], ei[1]
    dpq64 = torch.cat((torch.zeros(N, D, dtype=torch.float64, device=DEV).index_add_(0, rows_s, ref["da1"]),
                       torch.zeros(N, D, dtype=torch.float64, device=DEV).index_add_(0, rows_d, ref["da1"])), 1)
    mag = torch.cat((torch.zeros(N, D, dtype=torch.float64, device=DEV).index_add_(0, rows_s, ref["mag"]["da1"]),
                     torch.zeros(N, D, dtype=torch.float64, device=DEV).index_add_(0, rows_d, ref["mag"]["da1"])), 1)
    t = Table(f"chunked scorer -> dpq, exact grid: N = {N}, E = {E}", ["value", "ok"])
    # da1 = dz g: dz in {scale, -pw scale}, g on the step of w3 W2 (0.5 W3S * 0.25)
    t.add("precondition dpq units", exact_pre("dpq", dpq64, mag, 0.5 * W3S * 0.25 * scale), "-")
    got = {}
    for form, n in (("single", 1 << 26), ("chunked", 10_000)):
        monkeypatch.setitem(o.SCORER_CHUNK_EDGES, "n", n)
        gs = o.GraphStruct(ei, N)
        p = pq.clone().requires_grad_(True)
        loss, logits = o.EdgeScoreBCEPQFn.apply(p, P.w1c, P.b1, P.w2, P.b2, P.w3, P.b3, gs, sk, y, pw, scale)
        loss.backward()
        got[form] = p.grad
        if form == "chunked":
            runs = o.scored_chunks(gs, n).runs
            t.add("runs (longest)", len(runs), max(c1 - c0 for *_, c0, c1 in runs))
            assert len(runs) >= 5 and max(c1 - c0 for *_, c0, c1 in runs) > n
        t.add(f"{form}: logits bit-exact", "-", same(logits, ref["logits"]), ok=same(logits, ref["logits"]),
              why=f"{form} logits differ")
        for half, sl in (("P (by source)", slice(0, D)), ("Q (by destination)", slice(D, 2 * D))):
            nbad = int((p.grad[:, sl].double() != dpq64[:, sl]).sum())
            t.add(f"{form}: dpq {half}", nbad, nbad == 0, ok=nbad == 0, why=f"{form} {half}: {nbad} differ from fp64")
    eq = torch.equal(bits(got["single"]), bits(got["chunked"]))
    t.add("chunked == single, bit for bit", "-", eq, ok=eq, why="chunked dpq differs from the single launch")
    t.check()


# ================================================================================================
# B. gcn_aggregate
# ================================================================================================
AGG_F = [4, 8, 12, 16, 20, 28, 32, 36, 60, 64, 68, 124, 128, 132, 256, 260, 512]
AGG_GRAPHS = ["n1", "n31", "n32", "n33", "mixed1000", "n100003"]
N_SRC = 3000


def agg_degrees(name, g):
    if name == "mixed1000":
        deg = torch.randint(0, 10, (1000,), generator=g, device=DEV)
        deg[[0, 31, 32, 63, 96, 127, 128, 991, 999]] = 0          # empty rows at chunk starts and ends
        deg[160:192] = 0                                          # a whole empty 32-row chunk
        deg[200:209] = torch.arange(1, 10, device=DEV)
        deg[210:216] = torch.tensor([31, 32, 33, 63, 64, 65], device=DEV)
        deg[224:256] = 33                                         # a chunk whose rows straddle every batch
        deg[500] = 100_000                                        # hub
        return deg
    n = int(name[1:])
    if n == 1:
        return torch.tensor([65], device=DEV)
    return torch.randint(0, 10, (n,), generator=g, device=DEV) * (torch.rand(n, generator=g, device=DEV) > 0.2)


def csr_of(deg, g, n_src):
    rowptr = torch.zeros(deg.numel() + 1, dtype=torch.int64, device=DEV)
    rowptr[1:] = deg.cumsum(0)
    E = int(rowptr[-1])
    col = torch.randint(0, n_src, (E,), generator=g, device=DEV, dtype=torch.int32)
    rows = torch.repeat_interleave(torch.arange(deg.numel(), device=DEV), deg)
    return rowptr, col, rows


def call_agg(rowptr, col, val, x, num_rows, bias, act, out):
    o = ops()
    check(lib().pangnn_gcn_aggregate(ptr(rowptr), ptr(col), ptr(val), ptr(x), x.stride(0), num_rows, x.size(1),
                                     ptr(bias), act, ptr(out), out.stride(0), o._stream()), "gcn_aggregate")


def agg_ref(rows, col, val, x, num_rows, bias):
    """fp64 pre-activation and its sum |term|."""
    xv = x.double()[col.long()]
    v = val.double()[:, None] if val is not None else 1.0
    pre = torch.zeros(num_rows, x.size(1), dtype=torch.float64, device=DEV).index_add_(0, rows, v * xv)
    mag = torch.zeros_like(pre).index_add_(0, rows, (v * xv).abs())
    if bias is not None:
        pre += bias.double()
        mag += bias.double().abs()
    return pre, mag


def elu64(x):
    return torch.where(x > 0, x, torch.expm1(x))


def out_slice(num_rows, F, half):
    """A column slice (left or right half) of a NaN-payload buffer two slices wide."""
    buf = nan_fill(num_rows, 2 * F)
    return buf, buf[:, half * F:(half + 1) * F]


@pytest.mark.parametrize("F", AGG_F)
@pytest.mark.parametrize("graph", AGG_GRAPHS)
def test_gcn_aggregate_exact_grid(graph, F):
    """val given and NULL, bias given and not, strided and contiguous x, output into either half of a wider buffer
    whose other columns must stay bit-identical: act = NONE bit-exact; ELU within ELU_ULP of the fp64 ELU of the
    exact pre-activation."""
    o = ops()
    g = gen("agg_exact", graph, F)
    deg = agg_degrees(graph, g)
    N = deg.numel()
    rowptr, col, rows = csr_of(deg, g, N_SRC)
    xw = dyadic((N_SRC, F + 8), -8, 8, -3, g)
    val = dyadic((col.numel(),), 1, 4, -2, g)
    bias = dyadic((F,), -8, 8, -3, g)
    t = Table(f"gcn_aggregate, exact grid, {graph}: N = {N}, E = {col.numel()}, F = {F}",
              ["units", "differ/ulps", "other cols"])
    k = 0
    for vv in (val, None):
        for bb in (bias, None):
            x = xw[:, 4:4 + F] if k % 2 else xw[:, :F].contiguous()
            pre, mag = agg_ref(rows, col, vv, x, N, bb)
            units = exact_pre("aggregate", pre, mag, 2.0 ** (-5 if vv is not None else -3))
            for act in (o.ACT_NONE, o.ACT_ELU):
                half = (k + act) % 2
                buf, out = out_slice(N, F, half)
                fill = bits(buf).clone()
                call_agg(rowptr, col, vv, x, N, bb, act, out)
                other = torch.equal(bits(buf)[:, (1 - half) * F:(2 - half) * F], fill[:, (1 - half) * F:(2 - half) * F])
                case = (f"val {'y' if vv is not None else 'n'} bias {'y' if bb is not None else 'n'} "
                        f"x {'strided' if k % 2 else 'dense'} {'elu' if act else 'none'} -> {'LR'[half]}")
                if act == o.ACT_NONE:
                    nbad = int((out.double() != pre).sum())
                    t.add(case, units, nbad, other, ok=nbad == 0 and other,
                          why=f"{nbad} elements differ" if nbad else "other columns written")
                else:
                    ref = elu64(pre)
                    u = float(((out.double() - ref).abs() / ulp32(ref)).max()) if N else 0.0
                    t.add(case, units, u, other, ok=u <= ELU_ULP and other,
                          why=f"ELU {u:.2f} ulp" if other else "other columns written")
            k += 1
    t.check()


@pytest.mark.parametrize("F", [32, 64, 128])
def test_gcn_aggregate_identity_rebased_slice(F):
    """The identity variant (col = NULL: entry i of the CSR is row i of x) called as the chunked scorer calls it: a
    ``rowptr`` slice that starts at row r0 > 0 (offsets still absolute) and x's base shifted back by rowptr[r0] rows;
    bit-exact row sums, with and without bias."""
    g = gen("agg_ident", F)
    deg = agg_degrees("mixed1000", g)
    rowptr, _, rows = csr_of(deg, g, 1)
    E = int(rowptr[-1])
    x_all = dyadic((E, F), -8, 8, -3, g)
    bias = dyadic((F,), -8, 8, -3, g)
    t = Table(f"gcn_aggregate identity, rebased slice, F = {F}, E = {E}", ["rows", "differ"])
    for r0, r1 in ((37, 995), (1, 1000), (500, 501), (161, 300)):
        c0, c1 = int(rowptr[r0]), int(rowptr[r1])
        x_run = x_all[c0:c1].clone()                               # its own allocation, as the chunk's da1 is
        for bb in (None, bias):
            out = nan_fill(r1 - r0, F)
            check(lib().pangnn_gcn_aggregate(ptr(rowptr[r0:]), None, None, C.c_void_p(x_run.data_ptr() - c0 * F * 4),
                                             F, r1 - r0, F, ptr(bb), ops().ACT_NONE, ptr(out), F, ops()._stream()),
                  "gcn_aggregate(identity)")
            sel = (rows >= r0) & (rows < r1)
            ref = torch.zeros(r1 - r0, F, dtype=torch.float64, device=DEV).index_add_(
                0, rows[sel] - r0, x_all[sel].double())
            mag = torch.zeros_like(ref).index_add_(0, rows[sel] - r0, x_all[sel].double().abs())
            if bb is not None:
                ref, mag = ref + bb.double(), mag + bb.double().abs()
            exact_pre("identity", ref, mag, 2.0 ** -3)
            nbad = int((out.double() != ref).sum())
            t.add(f"rows [{r0}, {r1}), bias {'y' if bb is not None else 'n'}", r1 - r0, nbad, ok=nbad == 0,
                  why=f"{nbad} elements differ")
    t.check()


@pytest.mark.parametrize("F", AGG_F)
def test_gcn_aggregate_random_vs_index_add(F):
    """Random values (mixed signs) on the mixed graph with its hub: per element within AGG_REL * sum |val x| of
    ``index_add_`` in fp64; the plain-fp32 ``index_add_`` is the yardstick."""
    g = gen("agg_random", F)
    deg = agg_degrees("mixed1000", g)
    N = deg.numel()
    rowptr, col, rows = csr_of(deg, g, N_SRC)
    x = torch.randn(N_SRC, F, generator=g, device=DEV)
    val = torch.rand(col.numel(), generator=g, device=DEV) * 0.5 + 0.01
    bias = torch.randn(F, generator=g, device=DEV) * 0.1
    pre, mag = agg_ref(rows, col, val, x, N, bias)
    out = torch.empty(N, F, device=DEV)
    call_agg(rowptr, col, val, x, N, bias, ops().ACT_NONE, out)
    y32 = torch.zeros(N, F, device=DEV).index_add_(0, rows, val[:, None] * x[col.long()]) + bias
    r, r32 = ratio((out.double() - pre).abs(), AGG_REL * mag), ratio((y32.double() - pre).abs(), AGG_REL * mag)
    t = Table(f"gcn_aggregate, random, mixed1000 + hub, F = {F}", ["err/bar", "fp32 err/bar"])
    t.add("val + bias", r, r32, ok=r <= 1.0, why=f"error {r:.2f} x bar")
    t.check()


def test_gcn_aggregate_rows_past_2_31_bytes():
    """F = 128, x of 5e6 rows (512 bytes each): every gathered row lies past 2^31 bytes; bit-exact."""
    g = gen("agg_far")
    Nx, lo, F = 5_000_000, 4_200_000, 128
    x = torch.zeros(Nx, F, device=DEV)
    x[lo:] = dyadic((Nx - lo, F), -8, 8, -3, g)
    deg = torch.randint(0, 20, (1000,), generator=g, device=DEV)
    rowptr = torch.zeros(1001, dtype=torch.int64, device=DEV)
    rowptr[1:] = deg.cumsum(0)
    col = torch.randint(lo, Nx, (int(rowptr[-1]),), generator=g, device=DEV, dtype=torch.int32)
    rows = torch.repeat_interleave(torch.arange(1000, device=DEV), deg)
    val = dyadic((col.numel(),), 1, 4, -2, g)
    pre, mag = agg_ref(rows, col, val, x, 1000, None)
    exact_pre("aggregate far", pre, mag, 2.0 ** -5)
    out = nan_fill(1000, F)
    call_agg(rowptr, col, val, x, 1000, None, ops().ACT_NONE, out)
    assert same(out, pre), f"{int((out.double() != pre).sum())} elements differ"


# ================================================================================================
# C. gcn_norm / gcn_norm_apply
# ================================================================================================
@pytest.mark.parametrize("weighted", [True, False])
def test_gcn_norm_matches_fp64(weighted):
    """dis within DIS_ULP of 1 / sqrt(sum w) in fp64 and 0 at in-degree 0; val bit-identical to fp32 torch
    ``(dis[src] * w) * dis[dst]`` from the kernel's own dis, in the by-destination (gcn_norm) and by-source
    (gcn_norm_apply) orientation.  A hub with 1e5 in-edges at w = 81, 500 nodes with no in-edge."""
    o = ops()
    g = gen("gcn_norm", weighted)
    N, E = 20_000, 200_000
    src = torch.randint(0, N, (E,), generator=g, device=DEV)
    dst = torch.randint(0, N - 500, (E,), generator=g, device=DEV)
    w = torch.rand(E, generator=g, device=DEV) * 80 + 1
    src[:100_000], dst[:100_000], w[:100_000] = torch.randint(0, N, (100_000,), generator=g, device=DEV), 7, 81.0
    key = torch.argsort(src * N + dst)
    src, dst, w = src[key], dst[key], w[key]
    ei = torch.stack((src, dst)).contiguous()
    wt = w if weighted else None
    csr_d = o.csr_build(ei, N, by_dst=True)
    csr_s = o.csr_build(ei, N, by_dst=False)
    dis, val_d = torch.full((N,), float("nan"), device=DEV), nan_fill(E)
    check(lib().pangnn_gcn_norm(ptr(csr_d.rowptr), ptr(csr_d.col), ptr(csr_d.perm), ptr(wt), N, ptr(dis), ptr(val_d),
                                o._stream()), "gcn_norm")
    val_s = nan_fill(E)
    check(lib().pangnn_gcn_norm_apply(ptr(csr_s.rowptr), ptr(csr_s.col), ptr(csr_s.perm), ptr(wt), ptr(dis), N, 0,
                                      ptr(val_s), o._stream()), "gcn_norm_apply")
    w1 = w if weighted else torch.ones_like(w)
    deg = torch.zeros(N, dtype=torch.float64, device=DEV).index_add_(0, dst, w1.double())
    ref = torch.where(deg > 0, deg.rsqrt(), 0.0)
    nz = deg > 0
    ulps = float(((dis[nz].double() - ref[nz]).abs() / ulp32(ref[nz])).max())
    t = Table(f"gcn_norm, {'weighted' if weighted else 'unweighted'}: N = {N}, E = {E}, hub in-degree "
              f"{int((dst == 7).sum())}", ["value", "ok"])
    t.add("dis: max ulps", ulps, ulps <= DIS_ULP, ok=ulps <= DIS_ULP, why=f"dis {ulps:.2f} ulp")
    zero = bool((dis[~nz] == 0).all())
    t.add(f"dis = 0 at in-degree 0 ({int((~nz).sum())})", "-", zero, ok=zero, why="dis not 0 at in-degree 0")
    for name, csr, val in (("by destination", csr_d, val_d), ("by source", csr_s, val_s)):
        p = csr.perm.long()
        want = (dis[src[p]] * w1[p]) * dis[dst[p]]
        eq = torch.equal(bits(val), bits(want))
        t.add(f"val {name}", int((bits(val) != bits(want)).sum()), eq, ok=eq, why=f"val {name} not bit-identical")
    t.check()


# ================================================================================================
# D. pair decoders (cosine, dot)
# ================================================================================================
@pytest.mark.parametrize("F", [64, 30])
@pytest.mark.parametrize("mode", ["cosine", "dot"])
def test_edge_pair_score_matches_fp64_autograd(mode, F):
    """``edge_pair_score`` forward and backward against fp64 autograd of torch's definitions
    (``F.cosine_similarity(eps=1e-8)``, row-wise dot), with all-zero rows and rows whose norm is below the 1e-8
    clamp.  F = 64 takes the kernels, F = 30 the library backward of an odd width."""
    o = ops()
    g = gen("pair", mode, F)
    N, E = 5000, 60_000
    h = torch.randn(N, F, generator=g, device=DEV)
    h[::97] = 0.0                                                 # all-zero rows
    h[5::89] *= 3e-10                                             # norms ~1e-9 < 1e-8
    src = torch.randint(0, N, (E,), generator=g, device=DEV)
    dst = torch.randint(0, N, (E,), generator=g, device=DEV)
    key = torch.argsort(src * N + dst)
    ei = torch.stack((src[key], dst[key])).contiguous()
    s, d = ei[0], ei[1]
    dz = torch.randn(E, generator=g, device=DEV)
    gs = o.GraphStruct(ei, N)
    hh = h.clone().requires_grad_(True)
    out = o.edge_pair_score(hh, gs, 0 if mode == "cosine" else 1)
    out.backward(dz)
    h64 = h.double().requires_grad_(True)
    a, b = h64[s], h64[d]
    ref = tnf.cosine_similarity(a, b, dim=1, eps=1e-8) if mode == "cosine" else (a * b).sum(1)
    ref.backward(dz.double())
    # sums of |term|: forward |a||b| / (na nb); backward per edge |dz| (|h_other| / (na nb) + |c| |h_self| / na^2)
    with torch.no_grad():
        ha, hb = h.double()[s], h.double()[d]
        if mode == "cosine":
            ra, rb = ha.norm(dim=1, keepdim=True), hb.norm(dim=1, keepdim=True)
            na, nb = ra.clamp_min(1e-8), rb.clamp_min(1e-8)
            fmag = ((ha.abs() * hb.abs()).sum(1, keepdim=True) / (na * nb)).squeeze(1)
            c = ref.detach().abs()[:, None]
            ga = dz.double().abs()[:, None] * (hb.abs() / (na * nb) + c * ha.abs() / (na * ra.clamp_min(1e-300)))
            gb = dz.double().abs()[:, None] * (ha.abs() / (na * nb) + c * hb.abs() / (nb * rb.clamp_min(1e-300)))
        else:
            fmag = (ha.abs() * hb.abs()).sum(1)
            ga, gb = dz.double().abs()[:, None] * hb.abs(), dz.double().abs()[:, None] * ha.abs()
        gmag = torch.zeros(N, F, dtype=torch.float64, device=DEV).index_add_(0, s, ga).index_add_(0, d, gb)
    t = Table(f"edge_pair_score {mode}, F = {F}: N = {N}, E = {E}, {len(range(0, N, 97))} zero rows, "
              f"{len(range(5, N, 89))} rows of norm < 1e-8", ["err/bar", "scale err"])
    r = ratio((out.detach().double() - ref.detach()).abs(), PAIR_REL * fmag + 1e-30)
    t.add("forward", r, scale_err(out.detach(), ref.detach()), ok=r <= 1.0, why=f"forward {r:.2f} x bar")
    small = torch.zeros(N, dtype=torch.bool, device=DEV)
    small[5::89] = True
    for name, sel in (("dh, all rows", slice(None)), ("dh, rows of norm < 1e-8", small)):
        err = (hh.grad[sel].double() - h64.grad[sel]).abs()
        r = ratio(err, PAIR_REL * gmag[sel])
        t.add(name, r, scale_err(hh.grad[sel], h64.grad[sel]), ok=r <= 1.0, why=f"{name}: {r:.2f} x bar")
    t.check()
