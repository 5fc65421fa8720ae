"""The tensor-core conv (tpconv_umma_kernel) against a float64 replay of its own packed weight image (tests/_umma_image.py),
elementwise, at the schedule, aggregation, option and layout edges where a persistent, split, two-warpgroup kernel goes
wrong.

Inputs of GEMM1 (emb, the first ns columns of p1 / p2, W1, b1) lie on a dyadic grid (activations k/16 with |k| <= 64,
weights m/64 with |m| <= 128): every GEMM1 sum is then a multiple of 2^-10 below 2^11, exact in fp32 in any order, so the
kernel and the replay round the same hidden values to bf16.  What is left between them is fp32 accumulation (GEMM2 in
TMEM, the epilogue's FMAs, the atomics), which the gate bounds relative to the same replay on absolute values:
    |got - ref| <= TAU * ref_abs     elementwise (ref_abs = 0 -> got must be exactly 0)
A dropped or doubled edge, a partial sum added twice or a wrong tile / column is orders of magnitude above that.  Every sum
buffer carries GUARD sentinel rows on both sides that must come back bitwise unchanged.  The fixed-point entry points run
the same cases (gate + n_partials * 2^-33, status word 0, a repeat bitwise equal); the fp32 CUDA-core kernel runs the same
edge sets, with a per-edge weight, against float64 conv math; and the bf16x3 kernel is held to the oracle itself on
random (non-grid) inputs."""
import ctypes as C

import numpy as np
import pytest
import torch

import _common as T
import _umma_image as U
from diffdock_pocket_b200 import _lib, tp as tpmod
from diffdock_pocket_b200._lib import ptr
from diffdock_pocket_b200.score_model import TensorProductConvLayer
from oracle import e3nn_mini as E
from oracle.score_model_ref import TensorProductConvLayer as RefConv

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda:0')
# Worst |got - ref| / ref_abs seen on one NVIDIA B200 (1000 W power limit): 1.7e-7 in mode 0, 2.9e-7 in mode 1 (TAU = 1.5e-5),
# 1.5e-8 for the fp32 kernel (TAU_FP32 = 6.1e-5).  Kernel mutants that round the hidden activations toward zero, drop the
# in-degree from s0 or lose the last edge of a partial tile fail these tests (the first: 5.9e-4)
TAU = 2.0 ** -16             # tensor-core kernel, both modes
TAU_FP32 = 2.0 ** -14        # fp32 CUDA-core kernel (fp32 GEMMs: its error is not bounded by the bf16 replay's)
GUARD = 64
SENT32 = 0x7FA5A5A5          # NaN bit patterns: any write into a guard row shows
SENT64 = 0x7FA5A5A5_5A5A5A5A
SPLIT_MAX = 8
N_NODES = 70000              # node tables (x, p1, p2): gathered indices above 65535
E_SHAPE, E_UNSUPPORTED = -2, -3

# (ns, nv, layer, sh_lmax): the trunk irreps of the three instantiated widths, and one sh_lmax = 2 conv (L2 kernel, kind 5)
CONFIGS = {'60x10_l0': (60, 10, 0, 1), '60x10_l1': (60, 10, 1, 1), '60x10_l2': (60, 10, 2, 1), '60x10_l3': (60, 10, 3, 1),
           '24x6_l3': (24, 6, 3, 1), '16x4_l2': (16, 4, 2, 1), '16x4_l3': (16, 4, 3, 1), '16x4_l3_sh2': (16, 4, 3, 2)}
CASES = [(c, m) for c in CONFIGS for m in (0, 1)]
CASE_IDS = [f'{c}-mode{m}' for c, m in CASES]


def _irreps(ns, nv, layer):
    seq = [f'{ns}x0e', f'{ns}x0e + {nv}x1o', f'{ns}x0e + {nv}x1o + {nv}x1e', f'{ns}x0e + {nv}x1o + {nv}x1e + {ns}x0o']
    return seq[min(layer, 3)], seq[min(layer + 1, 3)]


def _sh_irreps(sh_lmax):
    return '1x0e+1x1o' if sh_lmax == 1 else '1x0e+1x1o+1x2e'


def _grid(shape, half, denom, g):
    return (torch.randint(-half, half + 1, shape, generator=g) / denom).float()


def _make_conv(ns, nv, layer, sh_lmax, seed):
    """A trunk conv whose first Linear lies on the weight grid (m / 64) and whose second is arbitrary."""
    in_ir, out_ir = _irreps(ns, nv, layer)
    torch.manual_seed(seed)
    conv = TensorProductConvLayer(in_ir, _sh_irreps(sh_lmax), out_ir, 3 * ns, residual=False, batch_norm=False, faster=sh_lmax == 1)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        conv.fc[0].weight.copy_(_grid(conv.fc[0].weight.shape, 128, 64, g))
        conv.fc[0].bias.copy_(_grid(conv.fc[0].bias.shape, 128, 64, g))
        conv.fc[3].weight.copy_(torch.randn(conv.fc[3].weight.shape, generator=g) * 0.1)
        conv.fc[3].bias.copy_(torch.randn(conv.fc[3].bias.shape, generator=g) * 0.1)
    return conv.to(DEV)


def _sm_count():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def split_k(live_tiles, cap_tiles, n_sms, n_tiles):
    """Host mirror of the kernel's work split: grid = min(tiles of the capacity, SMs); the last partial round of
    R = live_tiles mod grid edge tiles is split k = min(8, grid / R, n_tiles) ways along the weight tiles."""
    grid = min(cap_tiles, n_sms)
    r = live_tiles % grid
    return 1 if r == 0 else min(SPLIT_MAX, grid // r, n_tiles)


def split_parts(img, k):
    """The kernel's split[] boundaries: contiguous weight-tile ranges of about equal MMA cost (n_cols + 86 per tile), each
    with at least one tile."""
    cum = np.cumsum([0] + [td['n_cols'] + 86 for td in img.tiles])
    n, sp, t = img.n_tiles, [], 0
    for p in range(k + 1):
        target = int(cum[n]) * p // k
        while t < n and cum[t] < target:
            t += 1
        sp.append(n if p == k else t)
    for p in range(1, k):
        sp[p] = min(max(sp[p], sp[p - 1] + 1), n - (k - p))
    return sp


def schedule_views(n_sms, n_tiles):
    """(name, live edges, k) for every k in 1..8 (clipped to n_tiles): the partial round alone and behind a full round
    of n_sms tiles, with the last tile full and 37 edges short.  Capacity >= 2 * n_sms tiles keeps the grid at n_sms."""
    out = []
    for k in range(1, SPLIT_MAX + 1):
        rs = [r for r in range(1, n_sms) if min(SPLIT_MAX, n_sms // r) == k]
        if not rs:
            continue
        r = max(rs)
        for full in (0, 1):
            for short in (0, 37):
                tiles = r + full * n_sms
                live = tiles * 128 - short
                out.append((f'k{k}_R{r}_{"full" if full else "alone"}_short{short}', live, split_k(tiles, 2 * n_sms, n_sms, n_tiles)))
    return out


def _runs(lengths, n):
    return torch.repeat_interleave(torch.arange(len(lengths)), torch.as_tensor(lengths))[:n].to(torch.int32)


def agg_orders(cap, g):
    """Aggregation node per edge ([cap] int32) for the aggregation orders of the epilogue's pre-reduction."""
    warps = cap // 32 + 1
    o = {'random': torch.randint(0, 5000, (cap,), generator=g, dtype=torch.int32),
         'runs1': torch.arange(cap, dtype=torch.int32),
         'runs2': _runs([2] * (16 * warps), cap),                                 # 16 heads per warp
         'runs2_1': _runs(([2] * 15 + [1, 1]) * warps, cap),                      # 17 heads per warp: no pre-reduction
         'one_node': torch.full((cap,), 7, dtype=torch.int32),
         'ragged': _runs(torch.randint(1, 300, (cap // 100 + 10,), generator=g).tolist(), cap),
         'over_65535': torch.randint(0, N_NODES, (cap,), generator=g, dtype=torch.int32)}
    for run in (31, 32, 33, 127, 128, 129):
        o[f'run{run}'] = _runs([run] * (cap // run + 1), cap)
    return o


class Pool:
    """One configuration's conv, packed image, decoded replay and a pool of 2 * n_sms * 128 edges on the input grid, with
    the per-edge replay (value and absolute scale) computed once; every case is a view of it."""

    def __init__(self, name, mode):
        ns, nv, layer, sh_lmax = CONFIGS[name]
        self.name, self.mode, self.ns = name, mode, ns
        self.conv = _make_conv(ns, nv, layer, sh_lmax, seed=10 + 7 * list(CONFIGS).index(name))
        self.pk = self.conv.packed(DEV, ns, ns)
        self.image = self.pk.umma_image(self.conv, mode, DEV)
        self.img = U.Image(self.image.cpu().numpy().tobytes())
        self.rp = U.Replay(self.img, DEV)
        self.f_in, self.f_out, self.sh_dim = self.pk.spec.f_in, self.pk.spec.f_out, self.pk.spec.sh_dim
        _check_w1_grid(self.img, self.conv)
        self.n_sms = _sm_count()
        self.cap = 2 * self.n_sms * 128
        g = torch.Generator().manual_seed(1000 + len(name) + mode)
        cap, n = self.cap, N_NODES
        self.emb = _grid((cap, ns), 64, 16, g).to(DEV)
        p1, p2 = _grid((n, ns), 64, 16, g), _grid((n, ns), 64, 16, g)
        self.x = torch.randn(n, self.f_in, generator=g).to(DEV)
        self.gather = torch.randint(0, n, (cap,), generator=g, dtype=torch.int32).to(DEV)
        self.i1 = torch.randint(0, n, (cap,), generator=g, dtype=torch.int32).to(DEV)
        self.i2 = torch.randint(0, n, (cap,), generator=g, dtype=torch.int32).to(DEV)
        self.sh = torch.randn(cap, self.sh_dim, generator=g).to(DEV)
        self.ew = torch.rand(cap, generator=g).to(DEV) + 0.5
        self.p1, self.p2 = p1.to(DEV), p2.to(DEV)
        # padded layouts with the same values: ld1 / ld2 not a multiple of 4 (scalar gather loads), ldx = f_in + 2; the
        # padding is NaN, so a read of it that reaches the arithmetic shows
        nan = float('nan')
        self.p1_pad = torch.full((n, ns + 1), nan, device=DEV); self.p1_pad[:, :ns] = self.p1
        self.p2_pad = torch.full((n, ns + 3), nan, device=DEV); self.p2_pad[:, :ns] = self.p2
        self.x_pad = torch.full((n, self.f_in + 2), nan, device=DEV); self.x_pad[:, :self.f_in] = self.x
        self.aggs = {k: v.to(DEV) for k, v in agg_orders(cap, g).items()}
        self.deg = torch.tensor([0, 1, 1, 2, 3, 5, 17, 0], dtype=torch.int32)[torch.randint(0, 8, (N_NODES,), generator=g)].to(DEV)
        self.scale = (torch.rand(self.f_out, generator=g) * 1.5 + 0.5).to(DEV)
        A = U.a_operand(self.img, self.emb, self.p1, self.i1, self.p2, self.i2)
        _check_gemm1_exact(self.rp, A)
        xg = self.x[self.gather.long()]
        self.out_e = U.replay_chunked(self.rp, A, xg, self.sh)
        self.abs_e = U.replay_chunked(self.rp, A, xg, self.sh, absolute=True)


def _check_w1_grid(img, conv):
    """The decoded W1 reproduces the grid weights exactly (bf16 hi, zero lo): the precondition of the exact GEMM1."""
    ns, ks = img.ns, img.ks
    w1, b1 = conv.fc[0].weight.detach().cpu().numpy(), conv.fc[0].bias.detach().cpu().numpy()
    hid = w1.shape[0]
    for s in range(3):
        assert np.array_equal(img.w1_hi[:hid, s * ks:s * ks + ns], w1[:, s * ns:(s + 1) * ns]), s
    assert np.array_equal(img.w1_hi[:hid, ns], b1) and not img.w1_lo.any()


def _check_gemm1_exact(rp, A):
    a = A.double()
    assert torch.equal(a, A.to(torch.bfloat16).double()), 'A operand is not on the bf16-exact grid'
    pre = a @ rp.w1_hi.T
    q = pre * 1024
    assert torch.equal(q, q.round()) and float(pre.abs().max()) < 2.0 ** 11, 'GEMM1 sums are not exact in fp32'


# ------------------------------------------------------------------------------------------ launches
def _guarded(n_out, f_out, fixed):
    buf = torch.zeros(n_out + 2 * GUARD, f_out, dtype=torch.int64 if fixed else torch.float32, device=DEV)
    bits = buf.view(torch.int64 if fixed else torch.int32)
    bits[:GUARD] = SENT64 if fixed else SENT32
    bits[-GUARD:] = SENT64 if fixed else SENT32
    return buf


def _guards_intact(buf, fixed):
    bits = buf.view(torch.int64 if fixed else torch.int32)
    s = SENT64 if fixed else SENT32
    return bool((bits[:GUARD] == s).all()) and bool((bits[-GUARD:] == s).all())


def _body_ptr(buf):
    return buf.data_ptr() + GUARD * buf.shape[1] * buf.element_size()


def _to_float(buf):
    out = torch.empty(buf.shape, dtype=torch.float32, device=DEV)
    _lib.check(_lib.lib().ddp_fixed_to_float(ptr(buf), buf.numel(), ptr(out), _lib.stream_ptr()), 'ddp_fixed_to_float')
    return out


def _edges(pool, v, keep=()):
    """ddp_tpconv_edges_t of view v over the pool's arrays; keep collects the tensors the struct points into."""
    padded = v.get('layout') == 'padded'
    p1, p2, x = (pool.p1_pad, pool.p2_pad, pool.x_pad) if padded else (pool.p1, pool.p2, pool.x)
    n_dev = torch.tensor([v['n_dev']], dtype=torch.int32, device=DEV)
    agg = pool.aggs[v['agg']]
    keep += (n_dev,)
    return _lib.TpEdges(emb=ptr(pool.emb), p1=ptr(p1), i1=ptr(pool.i1), ld1=p1.shape[1], p2=ptr(p2), i2=ptr(pool.i2), ld2=p2.shape[1],
                        x=ptr(x), gather=ptr(pool.gather), ldx=x.shape[1], sh=ptr(pool.sh), agg=ptr(agg),
                        ew=ptr(pool.ew) if v.get('ew') else None, n_edges_dev=ptr(n_dev), edge_cap=v['cap'],
                        out_scale=ptr(pool.scale) if v.get('scale') else None, agg_deg=ptr(pool.deg) if v.get('deg') else None), keep


def run_umma(pool, v, fixed):
    """-> (sum rows as float32 [n_out, f_out], guards intact, status word)."""
    L = _lib.lib()
    ed, keep = _edges(pool, v)
    buf = _guarded(v['n_out'], pool.f_out, fixed)
    st = _lib.stream_ptr()
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    if fixed:
        rc = L.ddp_tpconv_umma_fixed(C.byref(pool.pk.cdesc), ptr(pool.image), pool.mode, C.byref(ed), _body_ptr(buf), ptr(status), st)
    else:
        rc = L.ddp_tpconv_umma(C.byref(pool.pk.cdesc), ptr(pool.image), pool.mode, C.byref(ed), _body_ptr(buf), st)
    _lib.check(rc, 'ddp_tpconv_umma' + ('_fixed' if fixed else ''))
    torch.cuda.synchronize()
    ok = _guards_intact(buf, fixed)
    body = buf[GUARD:-GUARD]
    return (_to_float(body) if fixed else body.clone()), ok, int(status.item()), (body.clone() if fixed else None)


def run_fp32(pool, v, fixed):
    L = _lib.lib()
    ed, keep = _edges(pool, v)
    buf = _guarded(v['n_out'], pool.f_out, fixed)
    st = _lib.stream_ptr()
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    if fixed:
        rc = L.ddp_tpconv_fp32_fixed(C.byref(pool.pk.cdesc), C.byref(ed), _body_ptr(buf), ptr(status), st)
    else:
        rc = L.ddp_tpconv_fp32(C.byref(pool.pk.cdesc), C.byref(ed), _body_ptr(buf), st)
    _lib.check(rc, 'ddp_tpconv_fp32' + ('_fixed' if fixed else ''))
    torch.cuda.synchronize()
    ok = _guards_intact(buf, fixed)
    body = buf[GUARD:-GUARD]
    return (_to_float(body) if fixed else body.clone()), ok, int(status.item()), (body.clone() if fixed else None)


# ------------------------------------------------------------------------------------------ references and the gate
def reference(pool, v, out_e, abs_e):
    """Scatter of the per-edge replay for view v: (ref, ref_abs, live in-degree) float64 [n_out, f_out]."""
    live = max(0, min(v['n_dev'], v['cap']))
    agg = pool.aggs[v['agg']][:live].long()
    f = torch.ones(live, dtype=torch.float64, device=DEV)
    if v.get('deg'):
        f = (1.0 / pool.deg[agg].clamp(min=1).float()).double()      # fp32 1 / max(deg, 1), as the kernel forms it
    if v.get('ew'):
        f = f * pool.ew[:live].double()
    ref = torch.zeros(v['n_out'], pool.f_out, dtype=torch.float64, device=DEV).index_add_(0, agg, out_e[:live] * f[:, None])
    ref_abs = torch.zeros_like(ref).index_add_(0, agg, abs_e[:live] * f.abs()[:, None])
    if v.get('scale'):
        ref, ref_abs = ref * pool.scale.double(), ref_abs * pool.scale.double().abs()
    cnt = torch.zeros(v['n_out'], dtype=torch.float64, device=DEV).index_add_(0, agg, torch.ones(live, dtype=torch.float64, device=DEV))
    return ref, ref_abs, cnt


def gate(got, ref, ref_abs, tau, slack=None):
    """-> (passes, worst |got - ref| / ref_abs, description of the worst element)."""
    err = (got.double() - ref).abs()
    bound = tau * ref_abs + (0 if slack is None else slack)
    ok = bool((err <= bound).all()) and bool(torch.isfinite(got).all())
    inf = torch.full_like(err, torch.inf)
    ratio = torch.where(ref_abs > 0, err / ref_abs.clamp(min=1e-300), torch.where(err > 0, inf, torch.zeros_like(err)))
    ratio = torch.where(torch.isfinite(got), ratio, inf)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    where = ''
    if ratio.numel() and worst > 0:
        i = int(ratio.argmax())
        r, c = divmod(i, ratio.shape[1])
        where = f'node {r} col {c}: got {float(got[r, c]):.6g} ref {float(ref[r, c]):.6g} ref_abs {float(ref_abs[r, c]):.3g}'
    return ok, worst, where


def check_views(pool, views, runner=None, out_e=None, abs_e=None, tau=TAU):
    """Run every view in the atomic and the fixed-point mode; -> list of failure lines and {mode: worst ratio}."""
    runner = run_umma if runner is None else runner
    out_e = pool.out_e if out_e is None else out_e
    abs_e = pool.abs_e if abs_e is None else abs_e
    fails, worst = [], {'float': 0.0, 'fixed': 0.0}
    for v in views:
        ref, ref_abs, cnt = reference(pool, v, out_e, abs_e)
        got, guards, status, _ = runner(pool, v, False)
        ok, r, where = gate(got, ref, ref_abs, tau)
        worst['float'] = max(worst['float'], r)
        if not (ok and guards):
            fails.append(f"{v['name']}: worst |got-ref|/ref_abs = {r:.3g} (tau {tau:.3g}), guards intact {guards}; {where}")
        # fixed point: each partial sum carries <= 2^-33 of rounding; an edge's contribution to a node arrives in at most
        # 2 (epilogue warpgroups) x 8 (split parts) partials
        got, guards, status, raw = runner(pool, v, True)
        ok, r, where = gate(got, ref, ref_abs, tau, slack=(16 * cnt[:, None] + 1) * 2.0 ** -33)
        worst['fixed'] = max(worst['fixed'], r)
        again = runner(pool, v, True)[3]
        same = torch.equal(raw, again)
        if not (ok and guards and status == 0 and same):
            fails.append(f"{v['name']} [fixed]: worst ratio {r:.3g}, guards intact {guards}, status {status}, repeat bitwise equal {same}; {where}")
    return fails, worst


_POOLS = {}


def _pool(name, mode):
    key = (name, mode)
    if key not in _POOLS:               # built once, shared by every test of the configuration (~0.3 GB each)
        _POOLS[key] = Pool(name, mode)
    return _POOLS[key]


def _view(name, live, cap, agg='random', n_dev=None, **kw):
    n_out = {'random': 5000, 'over_65535': N_NODES}.get(agg)
    return dict(name=name, n_dev=live if n_dev is None else n_dev, cap=cap, agg=agg, n_out=n_out, **kw)


def _finish_views(pool, views):
    for v in views:
        if v['n_out'] is None:
            live = max(0, min(v['n_dev'], v['cap']))
            top = int(pool.aggs[v['agg']][:max(live, 1)].max())
            v['n_out'] = top + 3                           # nodes no edge aggregates into must come back exactly 0
    return views


def _report(record_property, pool, worst, fails):
    for k, r in worst.items():
        record_property(f'worst_ratio_{k}', f'{r:.4g}')
    assert not fails, f'{pool.name} mode {pool.mode}: {len(fails)} failing view(s)\n' + '\n'.join(fails[:20])


# ------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize('name,mode', CASES, ids=CASE_IDS)
def test_split_schedule(name, mode, record_property):
    """Every split factor k = 1..8 (clipped to the image's tile count) of the last partial round, alone and behind a full
    round, last tile full and 37 edges short; plus live == capacity."""
    pool = _pool(name, mode)
    sv = schedule_views(pool.n_sms, pool.img.n_tiles)
    reached = {k for _, _, k in sv}
    assert reached == set(range(1, min(SPLIT_MAX, pool.img.n_tiles) + 1)), (reached, pool.img.n_tiles)
    for _, _, k in sv:
        sp = split_parts(pool.img, k)
        assert all(a < b for a, b in zip(sp, sp[1:])) and sp[0] == 0 and sp[-1] == pool.img.n_tiles, (k, sp)
    views = [_view(n, live, pool.cap) for n, live, _ in sv] + [_view('live_eq_cap', pool.cap, pool.cap)]
    fails, worst = check_views(pool, _finish_views(pool, views))
    _report(record_property, pool, worst, fails)


def _schedules(pool):
    """Two schedules for the non-schedule cases: split k = 3 behind a full round with a 37-edge short last tile, and the
    whole capacity (no split)."""
    r3 = max(r for r in range(1, pool.n_sms) if min(SPLIT_MAX, pool.n_sms // r) == 3)
    return [('k3', (pool.n_sms + r3) * 128 - 37), ('full', pool.cap)]


@pytest.mark.parametrize('name,mode', CASES, ids=CASE_IDS)
def test_aggregation_orders(name, mode, record_property):
    """Random aggregation; sorted runs of 1 and 2 (16 heads per warp) and a 2 / 1 mix (17 heads: no pre-reduction); runs
    of 31, 32, 33, 127, 128, 129 and random lengths up to 300 that cross warp, tile and split-item boundaries; every edge
    into one node; aggregation nodes above 65535."""
    pool = _pool(name, mode)
    views = [_view(f'{agg}_{sn}', live, pool.cap, agg=agg) for agg in pool.aggs for sn, live in _schedules(pool)]
    fails, worst = check_views(pool, _finish_views(pool, views))
    _report(record_property, pool, worst, fails)


@pytest.mark.parametrize('name,mode', CASES, ids=CASE_IDS)
def test_options_layouts_and_live_counts(name, mode, record_property):
    """agg_deg (with degree-0 and degree-1 nodes) and out_scale alone and together; ldx = f_in + 2 with ld1 / ld2 not a
    multiple of 4; live = 0 with capacity; a live count above the capacity (clamped)."""
    pool = _pool(name, mode)
    (_, live), _ = _schedules(pool)
    views = []
    for agg in ('random', 'run33'):
        for deg, scale in ((False, False), (True, False), (False, True), (True, True)):
            views.append(_view(f'{agg}_deg{int(deg)}_scale{int(scale)}', live, pool.cap, agg=agg, deg=deg, scale=scale))
            views.append(_view(f'{agg}_deg{int(deg)}_scale{int(scale)}_padded', live, pool.cap, agg=agg, deg=deg, scale=scale,
                               layout='padded'))
    views.append(_view('live0', 0, pool.cap))
    views.append(_view('live0_run33', 0, pool.cap, agg='run33'))
    views.append(_view('n_dev_above_cap', pool.cap, 5000 - 37))
    views.append(_view('n_dev_above_cap_run129', pool.cap, 3 * 128, agg='run129', deg=True))
    fails, worst = check_views(pool, _finish_views(pool, views))
    _report(record_property, pool, worst, fails)


# ------------------------------------------------------------------------------------------ fp32 CUDA-core kernel
def conv_math(pool, absolute=False, chunk=4096):
    """Per-edge fp32-kernel conv in float64 from the spec's row groups (the definition in include/ddp_b200.h), without the
    bf16 roundings: relu(W1 [emb | p1 | p2] + b1) -> W2 h + b2 -> sum_ij C[i][j][k] x sh."""
    pk, spec = pool.pk, pool.pk.spec
    f = (lambda t: t.abs()) if absolute else (lambda t: t)
    W1, b1 = f(pk.w1_host.double().to(DEV)), f(pk.b1_host.double().to(DEV))
    W2, b2 = f(pk.w2_host.double().to(DEV)), f(pk.b2_host.double().to(DEV))
    ctab = torch.tensor(spec.ctab, dtype=torch.float64, device=DEV)
    outs = []
    for c0 in range(0, pool.cap, chunk):
        sl = slice(c0, c0 + chunk)
        A = torch.cat([pool.emb[sl], pool.p1[pool.i1[sl].long()], pool.p2[pool.i2[sl].long()]], 1).double()
        h = f(A) @ W1.T + b1
        h = h if absolute else torch.relu(h)
        w = h @ W2.T + b2
        x, sh = f(pool.x[pool.gather[sl].long()].double()), f(pool.sh[sl].double())
        n = x.shape[0]
        out = torch.zeros(n, spec.f_out, dtype=torch.float64, device=DEV)
        for g in spec.groups:
            d1, d2, do, mi, mo = g['d1'], g['d2'], g['d_out'], g['mul_in'], g['mul_out']
            Cg = f(ctab[g['c_off']:g['c_off'] + d1 * d2 * do].reshape(d1, d2, do))
            xs = x[:, g['x_off']:g['x_off'] + mi * d1].reshape(n, mi, d1)
            basis = torch.einsum('ijk,eui,ej->euk', Cg, xs, sh[:, g['sh_off']:g['sh_off'] + d2])
            wg = w[:, g['w_off']:g['w_off'] + mi * mo].reshape(n, mi, mo)
            out[:, g['out_off']:g['out_off'] + mo * do] += torch.einsum('euo,euk->eok', wg, basis).reshape(n, mo * do)
        outs.append(out)
    return torch.cat(outs)


@pytest.mark.parametrize('name', ['60x10_l3', '24x6_l3', '16x4_l2', '16x4_l3_sh2'])
def test_fp32_kernel_same_edge_sets(name, record_property):
    """ddp_tpconv_fp32 / _fixed (the only conv that takes a per-edge weight) through the same edge sets and options,
    against float64 conv math with the same elementwise gate form."""
    pool = _pool(name, 0)
    out_e, abs_e = conv_math(pool), conv_math(pool, absolute=True)
    (_, live), _ = _schedules(pool)
    views = [_view('random_ew', live, pool.cap, ew=True), _view('run129_ew_deg_scale', live, pool.cap, agg='run129', ew=True, deg=True, scale=True),
             _view('one_node_padded', pool.cap, pool.cap, agg='one_node', layout='padded'), _view('over_65535', live, pool.cap, agg='over_65535', ew=True),
             _view('small_cap', pool.cap, 1000 - 5, agg='run33', ew=True), _view('live0', 0, pool.cap)]
    fails, worst = check_views(pool, _finish_views(pool, views), runner=run_fp32, out_e=out_e, abs_e=abs_e, tau=TAU_FP32)
    _report(record_property, pool, worst, fails)


# ------------------------------------------------------------------------------------------ grouped launch
def _group_call(convs, imgs, mode, eds, sums, fixed, status=None):
    L = _lib.lib()
    k = len(eds)
    a = lambda xs: (C.c_void_p * k)(*xs)
    cv = a([C.addressof(c) for c in convs])
    im = a([ptr(i) for i in imgs])
    ed = a([C.addressof(e) for e in eds])
    sm = a(sums)
    if fixed:
        return L.ddp_tpconv_umma_group_fixed(cv, im, mode, ed, sm, k, ptr(status), _lib.stream_ptr())
    return L.ddp_tpconv_umma_group(cv, im, mode, ed, sm, k, _lib.stream_ptr())


@pytest.mark.parametrize('mode', [0, 1])
def test_grouped_launch_nine_jobs(mode, record_property):
    """Nine jobs with different weights and live counts 0, 1, 127, 128, 129, ... (one with edge_cap = 0, one large enough that
    the launch's last round splits): every job against its own replay, guard rows intact, in the atomic and the
    fixed-point mode."""
    ns, nv, layer, sh_lmax = CONFIGS['24x6_l3']
    n_sms = _sm_count()
    big = n_sms + 20 - 45                                   # live tiles of the large job: the launch has n_sms + 20 in all
    lives = [0, 1, 127, 128, 129, 1000, 4000, big * 128 - 37, 0]
    caps = [256, 128, 128, 256, 384, 1024, 4096, (n_sms + 10) * 128, 0]
    g = torch.Generator().manual_seed(77)
    jobs = []
    for j, (live, cap) in enumerate(zip(lives, caps)):
        conv = _make_conv(ns, nv, layer, sh_lmax, seed=300 + j)
        pk = conv.packed(DEV, ns, ns)
        image = pk.umma_image(conv, mode, DEV)
        img = U.Image(image.cpu().numpy().tobytes())
        c = max(cap, 1)
        n = 3000
        t = dict(emb=_grid((c, ns), 64, 16, g), p1=_grid((n, ns), 64, 16, g), p2=_grid((n, ns), 64, 16, g),
                 x=torch.randn(n, pk.spec.f_in, generator=g), gather=torch.randint(0, n, (c,), generator=g, dtype=torch.int32),
                 i1=torch.randint(0, n, (c,), generator=g, dtype=torch.int32), i2=torch.randint(0, n, (c,), generator=g, dtype=torch.int32),
                 sh=torch.randn(c, 4, generator=g), agg=torch.sort(torch.randint(0, 2000, (c,), generator=g, dtype=torch.int32)).values,
                 n_dev=torch.tensor([live], dtype=torch.int32))
        t = {k: v.to(DEV) for k, v in t.items()}
        ed = _lib.TpEdges(emb=ptr(t['emb']), p1=ptr(t['p1']), i1=ptr(t['i1']), ld1=ns, p2=ptr(t['p2']), i2=ptr(t['i2']), ld2=ns,
                          x=ptr(t['x']), gather=ptr(t['gather']), ldx=pk.spec.f_in, sh=ptr(t['sh']), agg=ptr(t['agg']), ew=None,
                          n_edges_dev=ptr(t['n_dev']), edge_cap=cap)
        rp = U.Replay(img, DEV)
        A = U.a_operand(img, t['emb'][:live], t['p1'], t['i1'][:live], t['p2'], t['i2'][:live])
        xg, sh = t['x'][t['gather'][:live].long()], t['sh'][:live]
        out_e, abs_e = U.replay_chunked(rp, A, xg, sh), U.replay_chunked(rp, A, xg, sh, absolute=True)
        agg = t['agg'][:live].long()
        ref = torch.zeros(2000, pk.spec.f_out, dtype=torch.float64, device=DEV).index_add_(0, agg, out_e)
        ref_abs = torch.zeros_like(ref).index_add_(0, agg, abs_e)
        cnt = torch.zeros(2000, dtype=torch.float64, device=DEV).index_add_(0, agg, torch.ones(live, dtype=torch.float64, device=DEV))
        jobs.append(dict(pk=pk, image=image, ed=ed, t=t, ref=ref, ref_abs=ref_abs, cnt=cnt))
    n_tiles = U.Image(jobs[0]['image'].cpu().numpy().tobytes()).n_tiles
    k = split_k(sum((l + 127) // 128 for l in lives), sum((c + 127) // 128 for c in caps), n_sms, n_tiles)
    assert k > 1, 'the grouped launch should end in a split round'
    fails, worst = [], {}
    for fixed in (False, True):
        bufs = [_guarded(2000, j['pk'].spec.f_out, fixed) for j in jobs]
        status = torch.zeros(1, dtype=torch.int32, device=DEV)
        rc = _group_call([j['pk'].cdesc for j in jobs], [j['image'] for j in jobs], mode, [j['ed'] for j in jobs],
                         [_body_ptr(b) for b in bufs], fixed, status)
        _lib.check(rc, 'ddp_tpconv_umma_group' + ('_fixed' if fixed else ''))
        torch.cuda.synchronize()
        assert int(status.item()) == 0
        w = 0.0
        for j, (job, b) in enumerate(zip(jobs, bufs)):
            body = b[GUARD:-GUARD]
            got = _to_float(body) if fixed else body
            ok, r, where = gate(got, job['ref'], job['ref_abs'], TAU, slack=(16 * job['cnt'][:, None] + 1) * 2.0 ** -33 if fixed else None)
            w = max(w, r)
            guards = _guards_intact(b, fixed)
            if not (ok and guards):
                fails.append(f'job {j} (live {lives[j]}, cap {caps[j]}) {"fixed" if fixed else "float"}: worst ratio {r:.3g}, guards {guards}; {where}')
        worst['fixed' if fixed else 'float'] = w
    for k, r in worst.items():
        record_property(f'worst_ratio_{k}', f'{r:.4g}')
    assert not fails, '\n'.join(fails)


def test_grouped_launch_argument_errors():
    """10 jobs -> DDP_E_SHAPE; a per-edge weight or an odd ldx -> DDP_E_UNSUPPORTED (the kernel has neither)."""
    ns, nv, layer, sh_lmax = CONFIGS['16x4_l3']
    conv = _make_conv(ns, nv, layer, sh_lmax, seed=5)
    pk = conv.packed(DEV, ns, ns)
    image = pk.umma_image(conv, 0, DEV)
    cap, n = 256, 100
    emb, p = torch.zeros(cap, ns, device=DEV), torch.zeros(n, ns, device=DEV)
    x = torch.zeros(n, pk.spec.f_in + 1, device=DEV)
    idx = torch.zeros(cap, dtype=torch.int32, device=DEV)
    sh, ew = torch.zeros(cap, 4, device=DEV), torch.ones(cap, device=DEV)
    n_dev = torch.tensor([cap], dtype=torch.int32, device=DEV)
    s = torch.zeros(n, pk.spec.f_out, device=DEV)

    def ed(ew_=None, ldx=pk.spec.f_in):
        return _lib.TpEdges(emb=ptr(emb), p1=ptr(p), i1=ptr(idx), ld1=ns, p2=ptr(p), i2=ptr(idx), ld2=ns, x=ptr(x), gather=ptr(idx),
                            ldx=ldx, sh=ptr(sh), agg=ptr(idx), ew=ew_, n_edges_dev=ptr(n_dev), edge_cap=cap)
    good = ed()
    assert _group_call([pk.cdesc] * 10, [image] * 10, 0, [good] * 10, [ptr(s)] * 10, False) == E_SHAPE
    assert _group_call([pk.cdesc] * 10, [image] * 10, 0, [good] * 10, [ptr(s)] * 10, True, torch.zeros(1, dtype=torch.int32, device=DEV)) == E_SHAPE
    assert _group_call([pk.cdesc], [image], 0, [ed(ew_=ptr(ew))], [ptr(s)], False) == E_UNSUPPORTED
    assert _group_call([pk.cdesc], [image], 0, [ed(ldx=pk.spec.f_in + 1)], [ptr(s)], False) == E_UNSUPPORTED
    torch.cuda.synchronize()
    assert float(s.abs().max()) == 0


# ------------------------------------------------------------------------------------------ independent check vs the oracle
@pytest.mark.parametrize('name', list(CONFIGS))
def test_bf16x3_matches_oracle_on_random_inputs(name):
    """Random, non-grid inputs: the bf16x3 kernel against the oracle conv in float64 (not the image), per channel."""
    ns, nv, layer, sh_lmax = CONFIGS[name]
    in_ir, out_ir = _irreps(ns, nv, layer)
    sh_ir = _sh_irreps(sh_lmax)
    torch.manual_seed(21)
    conv = TensorProductConvLayer(in_ir, sh_ir, out_ir, 3 * ns, residual=False, batch_norm=False, faster=sh_lmax == 1)
    ref = RefConv(in_ir, sh_ir, out_ir, 3 * ns, residual=False, batch_norm=False, faster=sh_lmax == 1)
    ref.load_state_dict(conv.state_dict())
    conv = conv.to(DEV)
    pk = conv.packed(DEV, ns, ns)
    image = pk.umma_image(conv, 1, DEV)
    g = torch.Generator().manual_seed(22)
    cap, n_e, n = 3000, 3000 - 37, 400                     # live < capacity: rows past n_e are allocated, not used
    x = torch.randn(n, pk.spec.f_in, generator=g)
    ea = torch.randn(cap, 3 * ns, generator=g)
    sh = E.spherical_harmonics(sh_ir, torch.randn(cap, 3, generator=g))
    agg, src = torch.randint(0, n, (cap,), generator=g), torch.randint(0, n, (cap,), generator=g)
    with torch.no_grad():
        per_edge = ref.double().tp(x.double()[src[:n_e]], sh[:n_e].double(), ref.fc(ea[:n_e].double()))
    want = torch.zeros(n + 2, pk.spec.f_out, dtype=torch.float64).index_add_(0, agg[:n_e], per_edge)
    d = lambda t, dt=torch.float32: t.to(device=DEV, dtype=dt).contiguous()
    parts = [d(ea[:, i * ns:(i + 1) * ns]) for i in range(3)]
    ident = d(torch.arange(cap), torch.int32)
    xd, shd, aggd, srcd = d(x), d(sh), d(agg, torch.int32), d(src, torch.int32)
    n_dev = torch.tensor([n_e], dtype=torch.int32, device=DEV)
    ed = _lib.TpEdges(emb=ptr(parts[0]), p1=ptr(parts[1]), i1=ptr(ident), ld1=ns, p2=ptr(parts[2]), i2=ptr(ident), ld2=ns, x=ptr(xd),
                      gather=ptr(srcd), ldx=pk.spec.f_in, sh=ptr(shd), agg=ptr(aggd), ew=None, n_edges_dev=ptr(n_dev), edge_cap=cap)
    got = torch.zeros(n + 2, pk.spec.f_out, device=DEV)
    _lib.check(_lib.lib().ddp_tpconv_umma(C.byref(pk.cdesc), ptr(image), 1, C.byref(ed), ptr(got), _lib.stream_ptr()), 'ddp_tpconv_umma')
    torch.cuda.synchronize()
    assert tpmod.umma_supported(pk.spec, ns)
    err = T.rel_err_cols(got, want)
    assert err < 1e-4, (name, err)
