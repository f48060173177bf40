"""The backward reductions bit for bit at the training shapes, through TrainEngine's own launch plans.

Every operand is a small integer that bf16 holds exactly, so every product is an exact integer, and while the sum of
|terms| of an output stays below 2^24 every partial sum in any order -- tensor-core accumulators, per-CTA partials,
atomics, the deterministic finalize -- is an exact fp32 integer.  A kernel's result is then the exact sum whatever its
split, order or schedule, and must equal a float64 reference with torch.equal: one dropped, duplicated or misplaced
8x8 pixel tile is an integer error.  A factor that is not a power of two is applied once to an exact sum
(wgrad_reduce_kernel's and det_finalize's ``scale * s``), so the expected value is fl32(fl32(scale) * S); the one
exception is the default (atomic) column sum with scale 0.2, which scales every CTA's partial before adding it, and is
held to a bound instead.

Operands (``_values``): activation-like operands are +-1; gradient-like operands are +-1 except 0 at the first pixel
of every 8x8 tile.  An interior tile's contribution to any weight-gradient element, bias sum or edge sum is then a sum
of 63 odd terms -- odd, never zero -- so the data cannot hide a dropped tile.  The host tests (no GPU needed) check
that premise where the kernels' schedules put their last tiles and their stage-ring wraps, and that every site stays
inside the 2^24 budget; the GPU tests check it again on the values they compare.

The role and destination tables, kernel choice and CTA split under test are the production ones: the engine's
_rdb_wgrad / _single_conv_wgrad / _edge_wgrad are called on its own buffers.  Both the default mode and the
deterministic mode (a DetPlan driven with begin / the calls / flush, as TrainEngine._backward does) are checked.
"""

import numpy as np
import pytest
import torch
import torch.nn.functional as F

U = 2.0 ** -24
EXACT = 2 ** 24     # integers below this are exact in fp32, and so is every partial sum of terms whose |sum| is below
SM_COUNT = 148      # B200: the host-side schedule model (the GPU tests read the device's own figures)
SMEM_OPTIN = 232448
M31 = 2 ** 31 - 1


def gamma(k: int) -> float:
    """Worst-case relative error of a float32 sum of depth k."""
    return k * U / (1 - k * U)


# ------------------------------------------------------------------------------------------- integer operand fields
def _mix(idx: torch.Tensor, seed: int) -> torch.Tensor:
    """A hash of int64 indices below 2^31 (every product stays below 2^63, so CPU and GPU agree)."""
    h = (idx * 48271 + seed * 7919 + 1) % M31
    h = (h * 48271) % M31
    h = h ^ (h >> 13)
    h = (h * 16807) % M31
    return h ^ (h >> 9)


def _values(kind: str, seed: int, dims, b, y, x, c) -> torch.Tensor:
    """Element (b, y, x, c) of a logical [B, H, W, C] integer field (0 outside the image); b, y, x, c broadcast.
    kind "x": +-1.  "dy": +-1, 0 at every (y % 8, x % 8) == (0, 0).  "v2": 0 or +-2.  "gate": the clamp gate of
    conv_last, one value per horizontal pixel pair from {-0.5, 0, 0.5, 1, 1.5}, inside [0, 1] on the pair that holds a
    tile's first pixel (so a tile's gated "dy" field keeps an odd number of +-1)."""
    B, H, W, C = dims
    inside = (y >= 0) & (y < H) & (x >= 0) & (x < W)
    yc, xc = y.clamp(0, H - 1), x.clamp(0, W - 1)
    if kind == "gate":
        h = _mix((b * H + yc) * W + xc // 2, seed)
        v = ((h >> 7) % 5).double() * 0.5 - 0.5
        first = (yc % 8 == 0) & ((xc // 2) % 4 == 0)
        v = torch.where(first, ((h >> 7) & 1).double(), v)
        return torch.where(inside, v, torch.zeros_like(v))
    h = _mix(((b * H + yc) * W + xc) * C + c, seed)
    s = 1 - 2 * ((h >> 7) & 1)
    if kind == "dy":
        s = s * ~((yc % 8 == 0) & (xc % 8 == 0))
    elif kind == "v2":
        s = 2 * s * ((h >> 8) & 1)
    return torch.where(inside, s, torch.zeros_like(s))


def _image(kind: str, seed: int, dims, b: int, device) -> torch.Tensor:
    """Image b of a field as an int64 [H, W, C] tensor."""
    _, H, W, C = dims
    ar = lambda n: torch.arange(n, device=device)  # noqa: E731
    return _values(kind, seed, dims, torch.tensor(b, device=device), ar(H)[:, None, None], ar(W)[None, :, None],
                   ar(C)[None, None, :])


def _fill(buf: torch.Tensor, kind: str, seed: int) -> None:
    """buf [B, H, W, C] (NHWC) := the field, image by image."""
    dims = tuple(buf.shape)
    for b in range(dims[0]):
        buf[b] = _image(kind, seed, dims, b, buf.device).to(buf.dtype)


def _fill_nchw(t: torch.Tensor, kind: str, seed: int) -> None:
    """fp32 [B, 1, H, W] := the field with C = 1."""
    B, _, H, W = t.shape
    for b in range(B):
        t[b, 0] = _image(kind, seed, (B, H, W, 1), b, t.device)[..., 0].to(t.dtype)


def _window(kind: str, seed: int, dims, b: int, y0: int, x0: int, ny: int, nx: int, c0: int = 0, nc: int = -1):
    """Rows [y0, y0 + ny) x columns [x0, x0 + nx) x channels [c0, c0 + nc) of image b (float64, CPU)."""
    nc = dims[3] - c0 if nc < 0 else nc
    v = _values(kind, seed, dims, torch.tensor(b), torch.arange(y0, y0 + ny)[:, None, None],
                torch.arange(x0, x0 + nx)[None, :, None], torch.arange(c0, c0 + nc)[None, None, :])
    return v.double()


# ------------------------------------------------------------------------------------------- schedules (host model)
def _wgrad_schedule(roles, b, h, w, sm_count=SM_COUNT, smem_optin=SMEM_OPTIN):
    """xmm_conv3x3_wgrad's CTA split and stage count for a role table (the launcher's rules, xmm_b200.cu)."""
    cost, max_stage = [], 0
    for r in roles:
        tap_count, n, mode = r[1], r[5], (r[6] if len(r) > 6 else 0)
        cost.append(tap_count * max(n / 2.0, 47.0) * (1.3 if mode == 1 else 1.0))
        rows8 = mode == 0 and r[0] // 3 == (r[0] + tap_count - 1) // 3
        y_boxes = (n + 63) // 64
        st = r[3] * 8192 + 7168 if mode == 1 else r[3] * (10240 if rows8 else 13312) + y_boxes * 8192
        max_stage = max(max_stage, st)
    total = sum(cost)
    cnt = [max(1, int(sm_count * c / total)) for c in cost]
    k = 0
    while sum(cnt) != sm_count:
        if sum(cnt) < sm_count:
            cnt[k] += 1
        elif cnt[k] > 1:
            cnt[k] -= 1
        k = (k + 1) % len(cnt)
    stages = min(6, (smem_optin - 2048) // max_stage)
    tiles_x, tiles_y = (w + 7) // 8, (h + 7) // 8
    return cnt, stages, tiles_x, tiles_y, tiles_x * tiles_y * b


def _wgrad_teeth_tiles(roles, b, h, w, **dev):
    """Per role: the last tile of its last CTA, and CTA 0's first tile after its stage ring wraps (where it exists),
    as (label, image, tile row, tile column)."""
    cnt, stages, tx, ty, num = _wgrad_schedule(roles, b, h, w, **dev)
    out = []
    for r, c in enumerate(cnt):
        last = min(c, num) - 1
        picks = [(f"role {r} last tile of CTA {last}", last + (num - 1 - last) // c * c)]
        if stages * c < num:
            picks.append((f"role {r} CTA 0 at the ring wrap (stage 0, second phase)", stages * c))
        for label, t in picks:
            img, rest = divmod(t, tx * ty)
            out.append((label, img, rest // tx, rest % tx))
    return out


def _edge_teeth_tiles(b, h, w):
    """Row-blocked reductions (edge_wgrad: a CTA per 8 rows of one image; colsum: grid-stride over pixels): the last
    8x8 tile of the last image, and one interior tile."""
    return [("last tile", b - 1, (h - 1) // 8, (w - 1) // 8), ("interior tile", b // 2, h // 16, w // 16)]


def _tile_delta(xwin: torch.Tensor, dy: torch.Tensor) -> torch.Tensor:
    """Contribution of one tile to D[tap][i][o] = sum_p x[p + off(tap)][i] dy[p][o]: xwin [ny + 2, nx + 2, CX] (the
    tile with its halo), dy [ny, nx, CY]."""
    ny, nx = dy.shape[:2]
    yy = dy.reshape(ny * nx, -1)
    return torch.stack([xwin[t // 3:t // 3 + ny, t % 3:t % 3 + nx].reshape(ny * nx, -1).t() @ yy for t in range(9)])


# ------------------------------------------------------------------------------------------- engine plumbing
def _gen(kind, nf, nb, device="cpu"):
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR

    torch.manual_seed(11)
    g = GeneratorRRDB_DN(1, 1, nf, nb) if kind == "dn" else GeneratorRRDB_SR(1, 1, nf, nb, num_upsample=1)
    return g.to(device)


def _capture(monkeypatch, kind, nf, b, h, w, call):
    """The wgrad / colsum launches one engine method makes, recorded instead of run (meta buffers, no GPU)."""
    from xmm_superres_denoise_b200 import ops
    from xmm_superres_denoise_b200.engine_train import TrainEngine

    eng = TrainEngine(_gen(kind, nf, 1), kind)
    meta = torch.device("meta")
    bufs = eng._train_buffers(b, h, w, meta, False)
    grads = eng._grad_views(meta)
    calls = []
    monkeypatch.setattr(ops, "conv3x3_wgrad", lambda x, dy, roles, dsts: calls.append(("wgrad", x, dy, roles, dsts)))
    monkeypatch.setattr(ops, "colsum", lambda inp, *a, **k: calls.append(("colsum", inp)))
    monkeypatch.setattr(ops, "colsum_multi", lambda inp, segs: calls.append(("colsum", inp)))
    call(eng, bufs, grads)
    return eng, calls


# Wgrad sites: (id, kind, F, batch, H, W, which) -- `which` picks the engine call.
WGRAD_SITES = [
    ("dense F=32 r=0 1x8x8", "dn", 32, 1, 8, 8, ("rdb", 0)),
    ("dense F=32 r=0 3x37x29", "dn", 32, 3, 37, 29, ("rdb", 0)),
    ("dense F=32 r=0 16x416x416", "dn", 32, 16, 416, 416, ("rdb", 0)),
    ("dense F=32 r=2 16x416x416", "dn", 32, 16, 416, 416, ("rdb", 2)),
    ("dense F=64 r=1 4x416x416", "dn", 64, 4, 416, 416, ("rdb", 1)),
    ("dense F=64 r=0 3x37x29", "dn", 64, 3, 37, 29, ("rdb", 0)),
    ("trunk F=32 16x416x416", "dn", 32, 16, 416, 416, ("trunk",)),
    ("trunk F=64 4x416x416", "dn", 64, 4, 416, 416, ("trunk",)),
    ("upsampling F=32 16x416x416", "sr", 32, 16, 416, 416, ("up",)),
    ("HRconv F=32 16x832x832", "sr", 32, 16, 416, 416, ("hr",)),
]


def _site_io(eng, bufs, which):
    """(x buffer, dy buffer, engine call) of a wgrad site."""
    g = eng.gen
    if which[0] == "rdb":
        r = which[1]
        return (eng._block_act(bufs, 0, r), bufs["ring"][r],
                lambda grads: eng._rdb_wgrad(0, r, bufs, grads))
    if which[0] == "trunk":
        x = bufs["act"][3 * eng.nb]
        return x, bufs["d_trunk"], lambda grads: eng._single_conv_wgrad(g.trunk_conv, x, bufs["d_trunk"], grads)
    if which[0] == "up":
        return (bufs["trunk"], bufs["d_up0"],
                lambda grads: eng._single_conv_wgrad(g.upsampling[0], bufs["trunk"], bufs["d_up0"], grads, perm=1))
    return bufs["up0"], bufs["d_hr"], lambda grads: eng._single_conv_wgrad(g.HRconv, bufs["up0"], bufs["d_hr"], grads)


def _site_params(eng, which):
    """[(weight, bias or None, k (dense-block layer) or 0, perm)] of a wgrad site."""
    g = eng.gen
    if which[0] == "rdb":
        rdb = eng._rdb(0, which[1])
        return [(getattr(rdb, f"conv{k}").weight, getattr(rdb, f"conv{k}").bias, k, 0) for k in range(1, 6)]
    conv = g.trunk_conv if which[0] == "trunk" else g.upsampling[0] if which[0] == "up" else g.HRconv
    return [(conv.weight, conv.bias, 0, int(which[0] == "up"))]


def _perm(n: int) -> torch.Tensor:
    """Packed column j = g * (n / 4) + c of the upsampling conv holds PixelShuffle channel 4c + g."""
    j = torch.arange(n)
    return 4 * (j % (n // 4)) + j // (n // 4)


def _want_weights(D, f, params, s5):
    """Expected dW of every parameter from exact sums D[tap][x channel][dy channel] (float64), as fp32: exact sums,
    conv5's through one rounding of fl32(s5) * S."""
    out = []
    for wt, _, k, perm in params:
        n, cin = wt.shape[0], wt.shape[1]
        cy0 = (k - 1) * f if k else 0
        S = D[:, :cin, cy0:cy0 + n].permute(2, 1, 0).reshape(n, cin, 3, 3)
        if perm:
            full = torch.empty_like(S)
            full[_perm(n).to(S.device)] = S
            S = full
        out.append(_scaled(S, s5 if k == 5 else 1.0))
    return out


def _scaled(S: torch.Tensor, scale: float) -> torch.Tensor:
    """fl32(fl32(scale) * S) for exact integer sums S (the float64 product is exact: 24 x 24 significant bits)."""
    return (S * float(np.float32(scale))).float()


def _want_biases(colsums, f, params, s5):
    """Expected bias gradients from exact column sums of the site's dy buffer (None where the site does not produce
    them: fused into the F = 32 data-gradient launches)."""
    out = []
    for wt, bias, k, perm in params:
        n = wt.shape[0]
        if bias is None or colsums is None:
            out.append(None)
            continue
        c0 = (k - 1) * f if k else 0
        S = colsums[c0:c0 + n]
        if perm:
            full = torch.empty_like(S)
            full[_perm(n).to(S.device)] = S
            S = full
        out.append(_scaled(S, s5 if k == 5 else 1.0))
    return out


# ------------------------------------------------------------------------------------------- host side (no GPU)
def _site(site_id):
    return next(s for s in WGRAD_SITES if s[0] == site_id)


@pytest.mark.parametrize("site_id", [s[0] for s in WGRAD_SITES])
def test_wgrad_site_budget_and_teeth(monkeypatch, site_id):
    """The engine's own role tables; the schedule's last tiles and ring wraps; every interior tile there moves >= 90 %
    of the checked sums; the site's sum of |x dy| stays below 2^24."""
    _, kind, f, b, h, w, which = _site(site_id)
    box = {}

    def call(eng, bufs, grads):
        x, dy, run = _site_io(eng, bufs, which)
        box.update(x=x, dy=dy, params=_site_params(eng, which))
        run(grads)

    eng, calls = _capture(monkeypatch, kind, f, b, h, w, call)
    x, dy = box["x"], box["dy"]
    wcalls = [c for c in calls if c[0] == "wgrad"]
    assert wcalls, site_id
    xb, yb = x.shape, dy.shape
    B, H, W = xb[:3]
    # budget: |x| <= 1 and |dy| <= 1, so every weight-gradient element and column sum adds at most B*H*W units
    assert B * H * W * 1 * 1 < EXACT, f"{site_id}: {B * H * W} pixels void the 2^24 exactness budget"
    s5 = 0.04 if which == ("rdb", 2) else 0.2
    checked = changed = 0
    for _, xc, dyc, roles, dsts in wcalls:
        assert xc is x and dyc is dy
        for label, img, ty, tx in _wgrad_teeth_tiles(roles, B, H, W):
            xwin = _window("x", 1, xb, img, 8 * ty - 1, 8 * tx - 1, 10, 10)
            ywin = _window("dy", 2, yb, img, 8 * ty, 8 * tx, 8, 8)
            D = _tile_delta(xwin, ywin)
            moved = [t != 0 for t in _want_weights(D, f, box["params"], 1.0)]
            c, m = sum(t.numel() for t in moved), sum(int(t.sum()) for t in moved)
            interior = 0 < ty and 8 * ty + 8 < H and 0 < tx and 8 * tx + 8 < W
            print(f"{site_id}: {label} (image {img}, tile {ty},{tx}): {m} of {c} checked sums move")
            if interior:
                assert m == c, f"{site_id}: {label} is an interior tile, its sums are odd -- {c - m} did not move"
            checked, changed = checked + c, changed + m
    assert changed >= 0.9 * checked, f"{site_id}: a dropped tile moves only {changed} of {checked} checked sums"
    if any(p[1] is not None for p in box["params"]) and (f == 64 or which[0] != "rdb"):
        assert [c for c in calls if c[0] == "colsum"], f"{site_id}: no bias pass recorded"


@pytest.mark.parametrize("kind,b,h,w", [("dn", 16, 416, 416), ("sr", 16, 832, 832)])
def test_edge_site_budget_and_teeth(kind, b, h, w):
    """conv_last (gated gout x features, and its bias sum) and conv_first (image x (d_fea + d_trunk)): every tile the
    schedule finishes on moves every sum; |s| (|v| + |v2|) <= 3 keeps the sums below 2^24."""
    f = 32
    dims_s, dims_v = (b, h, w, 1), (b, h, w, f)
    vmax = 3 if kind == "dn" else 1  # conv_first (DN shape): v + v2 in {+-1, +-3}
    assert b * h * w * vmax < EXACT
    moved = {}
    for label, img, ty, tx in _edge_teeth_tiles(b, h, w):
        s = _window("dy", 3, dims_s, img, 8 * ty, 8 * tx, 8, 8)
        gate = _window("gate", 4, dims_s, img, 8 * ty, 8 * tx, 8, 8)
        sg = s * ((gate >= 0) & (gate <= 1))
        v = _window("x", 5, dims_v, img, 8 * ty - 1, 8 * tx - 1, 10, 10)
        sums = {"conv_last": torch.cat([_tile_delta(v, sg).reshape(-1), sg.sum().reshape(1)]),
                "column sums": _window("dy", 2, dims_v, img, 8 * ty, 8 * tx, 8, 8).sum(dim=(0, 1))}
        if kind == "dn":
            sums["conv_first"] = _tile_delta(v + _window("v2", 6, dims_v, img, 8 * ty - 1, 8 * tx - 1, 10, 10), s)
        interior = 0 < ty and 8 * ty + 8 < h and 0 < tx and 8 * tx + 8 < w
        for site, t in sums.items():
            m, c = int((t != 0).sum()), t.numel()
            print(f"{site} {b}x{h}x{w}: {label} (image {img}, tile {ty},{tx}): {m} of {c} sums move")
            assert m == c or not interior, f"{site}: {label} is an interior tile, its sums are odd"
            a = moved.setdefault(site, [0, 0])
            a[0], a[1] = a[0] + m, a[1] + c
    for site, (m, c) in moved.items():
        assert m >= 0.9 * c, f"{site} {b}x{h}x{w}: a dropped tile moves only {m} of {c} sums"


def test_fields_agree_with_their_windows():
    """_window (host, the teeth) and _image (the GPU fill) are the same field, zero outside the image."""
    dims = (2, 11, 13, 24)
    for kind in ("x", "dy", "v2"):
        full = _image(kind, 9, dims, 1, "cpu").double()
        win = _window(kind, 9, dims, 1, -1, 4, 13, 10, 8, 16)
        assert torch.equal(win[1:12, :9], full[:, 4:13, 8:24])
        assert float(win[0].abs().sum()) == 0.0 and float(win[12].abs().sum()) == 0.0
    d = _image("dy", 9, dims, 0, "cpu")
    assert int((d == 0).sum()) == 2 * 2 * 24 and set(d.unique().tolist()) == {-1, 0, 1}


# ------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def dev():
    from xmm_superres_denoise_b200 import _lib

    _lib.check(_lib.load().xmm_check_device())
    return torch.device("cuda:0")


def _dev_sched(d):
    p = torch.cuda.get_device_properties(d)
    return dict(sm_count=p.multi_processor_count, smem_optin=getattr(p, "shared_memory_per_block_optin", SMEM_OPTIN))


_ENGINES = {}


def _engine(kind, nf, d):
    key = (kind, nf)
    if key not in _ENGINES:
        from xmm_superres_denoise_b200.engine_train import TrainEngine

        _ENGINES.clear()
        gen = _gen(kind, nf, 1, d)
        eng = TrainEngine(gen, kind)
        eng.arena.ensure(d)
        _ENGINES[key] = eng
    return _ENGINES[key]


def _modes(eng, d, bhw, run, setup=None, after=None):
    """[(mode, flat gradient views)]: the same engine calls in the default mode and in deterministic mode (setup():
    refill inputs the calls overwrite; after(mode): snapshot outputs the next mode overwrites)."""
    from xmm_superres_denoise_b200 import determinism

    out = []
    for mode in ("default", "deterministic"):
        if setup is not None:
            setup()
        grads = eng._grad_views(d, eng._det_scratch_floats() if mode == "deterministic" else 0)
        plan = None
        if mode == "deterministic":
            plan = determinism.DetPlan(d)
            plan.begin(eng._flat_ext)
            eng._det, eng._det_bhw = plan, bhw
        try:
            run(grads)
            if plan is not None:
                plan.flush()
        finally:
            eng._det = None
        torch.cuda.synchronize()
        if after is not None:
            after(mode)
        out.append((mode, grads))
    return out


def _gv(eng, grads, p):
    return grads[eng._pindex[id(p)]]


def _wgrad_sums(x: torch.Tensor, dy: torch.Tensor) -> torch.Tensor:
    """D[tap][i][o] = sum_p x[p + off(tap)][i] dy[p][o] in float64 (x, dy [B, H, W, C] on the GPU)."""
    B, H, W, cx = x.shape
    cy = dy.shape[3]
    D = torch.zeros(9, cx, cy, dtype=torch.float64, device=x.device)
    for b in range(B):
        xp = F.pad(x[b].double(), (0, 0, 1, 1, 1, 1))
        yy = dy[b].double().reshape(H * W, cy)
        for t in range(9):
            D[t] += xp[t // 3:t // 3 + H, t % 3:t % 3 + W].reshape(H * W, cx).t() @ yy
    return D


def _tile_from(x, dy, img, ty, tx):
    """The (x halo window, dy tile) of one 8x8 tile of GPU buffers, zero outside the image (float64)."""
    H, W = x.shape[1:3]
    xp = F.pad(x[img].double(), (0, 0, 1, 9, 1, 9))
    yp = F.pad(dy[img].double(), (0, 0, 0, 8, 0, 8))
    return xp[8 * ty:8 * ty + 10, 8 * tx:8 * tx + 10], yp[8 * ty:8 * ty + 8, 8 * tx:8 * tx + 8]


def _compare(tag, got, want) -> int:
    """Mismatches of a list of fp32 results against their expected fp32 values; prints the count and the first few."""
    n = bad = 0
    lines = []
    for k, (g, w) in enumerate(zip(got, want)):
        if w is None:
            continue
        g = g.float().reshape(w.shape)
        ne = g != w
        n, bad = n + w.numel(), bad + int(ne.sum())
        for idx in ne.nonzero()[:4].tolist():
            lines.append(f"  tensor {k} at {tuple(idx)}: got {float(g[tuple(idx)])!r}, want {float(w[tuple(idx)])!r}")
    print(f"{tag}: {n} elements compared, {bad} mismatches")
    if lines:
        print("\n".join(lines))
    return bad


def _teeth_on_gpu(tag, D, x, dy, tiles, want_fn, got_want):
    """The compared values with one tile's sums removed: >= 90 % of them must differ from what the kernels matched."""
    for label, img, ty, tx in tiles:
        xw, yw = _tile_from(x, dy, img, ty, tx)
        w2 = want_fn(D - _tile_delta(xw, yw))
        c = sum(w.numel() for w in got_want if w is not None)
        m = sum(int((a != b).sum()) for a, b in zip(w2, got_want) if b is not None)
        print(f"{tag}: without {label} (image {img}, tile {ty},{tx}) {m} of {c} compared values differ")
        assert m >= 0.9 * c, f"{tag}: the data hides {label}"


def _run_wgrad_site(d, site_id):
    _, kind, f, b, h, w, which = _site(site_id)
    eng = _engine(kind, f, d)
    bufs = eng._train_buffers(b, h, w, d, False)
    x, dy, run = _site_io(eng, bufs, which)
    params = _site_params(eng, which)
    _fill(x, "x", 1)
    _fill(dy, "dy", 2)
    roles = []
    from xmm_superres_denoise_b200 import ops

    real = ops.conv3x3_wgrad

    def spy(*a):
        roles.append(a[2])
        real(*a)

    ops.conv3x3_wgrad = spy
    try:
        results = _modes(eng, d, (b, h, w) if which[0] == "rdb" else tuple(dy.shape[:3]), run)
    finally:
        ops.conv3x3_wgrad = real
    s5 = 0.04 if which == ("rdb", 2) else 0.2
    D = _wgrad_sums(x, dy)
    assert float(D.abs().max()) < EXACT
    wantw = _want_weights(D, f, params, s5)
    colsums = dy.double().sum(dim=(0, 1, 2)) if (f == 64 or which[0] != "rdb") else None
    wantb = _want_biases(colsums, f, params, s5)
    bounded = {}
    if which[0] == "rdb" and f == 64:
        # default mode: colsum_multi scales each CTA's partial by 0.2 / 0.04 before its atomicAdd -- bounded
        from xmm_superres_denoise_b200 import _lib

        K = ops.det_slots(_lib.DET_COLSUM, b, h, w, 5 * f)
        mag = dy[..., 4 * f:].double().abs().sum(dim=(0, 1, 2))
        bounded[4] = (gamma(K + 1) * s5 * mag + U * wantb[4].double().abs(), K)
    total_bad = 0
    for mode, grads in results:
        gw = [_gv(eng, grads, p[0]) for p in params]
        gb = [_gv(eng, grads, p[1]) if p[1] is not None else None for p in params]
        wb = list(wantb)
        if mode == "default" and 4 in bounded:
            bound, K = bounded[4]
            err = (gb[4].double() - wantb[4].double()).abs()
            print(f"{site_id} [{mode}] conv5 bias (atomic, scale {s5}, K = {K}): max |err| / bound = "
                  f"{float((err / bound).max()):.3f}")
            assert bool((err <= bound).all()), f"{site_id}: conv5 bias outside its bound"
            wb[4] = None
        total_bad += _compare(f"{site_id} [{mode}] weight gradients", gw, wantw)
        total_bad += _compare(f"{site_id} [{mode}] bias gradients", gb, wb)
    if total_bad:
        return total_bad
    dsched = _dev_sched(d)
    for rt in roles[:len(roles) // 2]:
        _teeth_on_gpu(site_id, D, x, dy, _wgrad_teeth_tiles(rt, b, h, w, **dsched),
                      lambda Dz: _want_weights(Dz, f, params, s5), wantw)
    return total_bad


@pytest.mark.gpu
def test_one_tile_wgrad_premise(dev):
    """Runs first: one 8x8 tile, one CTA per role.  A mismatch here is not a schedule fault."""
    bad = _run_wgrad_site(dev, "dense F=32 r=0 1x8x8")
    assert bad == 0, ("tensor-core fp32 accumulation of integers below 2^24 was not exact (one 8x8 tile, one CTA per "
                      "role): the premise of every exact check in this file is broken, not a schedule")


@pytest.mark.gpu
@pytest.mark.parametrize("site_id", [s[0] for s in WGRAD_SITES[1:]])
def test_wgrad_site_exact(dev, site_id):
    assert _run_wgrad_site(dev, site_id) == 0, site_id


def _edge_sums(s: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """R[o][c][tap] = sum_p s[o][p] v[p + off(tap)][c] in float64: s [B, ns, H, W], v [B, H, W, C]."""
    B, ns, H, W = s.shape
    C = v.shape[3]
    R = torch.zeros(ns, C, 9, dtype=torch.float64, device=v.device)
    for b in range(B):
        vp = F.pad(v[b].double(), (0, 0, 1, 1, 1, 1))
        sb = s[b].double().reshape(ns, H * W)
        for t in range(9):
            R[:, :, t] += sb @ vp[t // 3:t // 3 + H, t % 3:t % 3 + W].reshape(H * W, C)
    return R


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dn", "sr"])
def test_conv_last_edge_wgrad_exact(dev, kind):
    """conv_last's weight and bias gradients (edge_wgrad with the clamp gate) at DN 416^2 / SR 832^2, batch 16."""
    f, b, h, w = 32, 16, 416, 416
    eng = _engine(kind, f, dev)
    bufs = eng._train_buffers(b, h, w, dev, False)
    g = eng.gen
    feat = bufs["trunk"] if kind == "dn" else bufs["hr"]
    H, W = feat.shape[1:3]
    gout = torch.empty(b, 1, H, W, device=dev)
    _fill_nchw(gout, "dy", 3)
    pre = bufs["pre"]
    _fill_nchw(pre, "gate", 4)
    _fill(feat, "x", 5)
    dw = g.conv_last.weight
    results = _modes(eng, dev, (b, h, w), lambda grads: eng._edge_wgrad(
        gout, feat, 0, f, _gv(eng, grads, dw).view(1, f, 9), ssum=_gv(eng, grads, g.conv_last.bias), gate=pre))
    sg = gout.double() * ((pre >= 0) & (pre <= 1))
    R = _edge_sums(sg, feat)
    S = sg.sum().reshape(1)
    assert float(R.abs().max()) < EXACT and float(sg.abs().sum()) < EXACT
    want = [R.float(), S.float()]
    bad = 0
    for mode, grads in results:
        bad += _compare(f"conv_last {kind} {b}x{H}x{W} [{mode}]", [_gv(eng, grads, dw).view(1, f, 9),
                                                                  _gv(eng, grads, g.conv_last.bias)], want)
    for label, img, ty, tx in _edge_teeth_tiles(b, H, W):
        vw, _ = _tile_from(feat, feat, img, ty, tx)
        sw = F.pad(sg[img, 0], (0, 8, 0, 8))[8 * ty:8 * ty + 8, 8 * tx:8 * tx + 8, None]
        R2 = R - _tile_delta(vw, sw).permute(2, 1, 0)
        m = int((R2.float() != want[0]).sum()) + int(float(S - sw.sum()) != float(S))
        print(f"conv_last {kind}: without {label} {m} of {R.numel() + 1} compared values differ")
        assert m >= 0.9 * (R.numel() + 1)
    assert bad == 0


@pytest.mark.gpu
def test_conv_first_edge_wgrad_and_bias_exact(dev):
    """conv_first's weight gradient through v + v2 (d_fea + d_trunk) and its bias as two column sums, as
    TrainEngine._backward launches them, DN 416^2 batch 16."""
    from xmm_superres_denoise_b200 import ops

    f, b, h, w = 32, 16, 416, 416
    eng = _engine("dn", f, dev)
    bufs = eng._train_buffers(b, h, w, dev, False)
    g = eng.gen
    x = torch.empty(b, 1, h, w, device=dev)
    _fill_nchw(x, "dy", 3)
    d_fea, d_trunk = bufs["d_fea"], bufs["d_trunk"]
    _fill(d_fea, "x", 5)
    _fill(d_trunk, "v2", 6)
    box = {}

    def run(grads):  # the conv_first block of TrainEngine._backward
        dbf = _gv(eng, grads, g.conv_first.bias)
        if eng._det is None:
            r = torch.zeros(1, f, 9, dtype=torch.float32, device=dev)
            ops.edge_wgrad(x, d_fea, 0, f, r, v2=d_trunk, v2_coff=0)
            ops.colsum(d_fea, 0, f, dbf)
            ops.colsum(d_trunk, 0, f, dbf, accumulate=True)
        else:
            r = eng._scratch(f * 9).view(1, f, 9)
            eng._det.edge_wgrad(x, d_fea, 0, f, r, v2=d_trunk, v2_coff=0)
            eng._det.colsum([d_fea, d_trunk], [(0, f, dbf, 1.0, False)])
        box[eng._det is None] = r

    results = _modes(eng, dev, (b, h, w), run)
    V = d_fea.double() + d_trunk.double()
    R = _edge_sums(x, V)
    S = V.sum(dim=(0, 1, 2))
    assert float((x.double().abs().sum())) * 3 < EXACT
    want = [R.float(), S.float()]
    bad = 0
    for mode, grads in results:
        bad += _compare(f"conv_first {b}x{h}x{w} [{mode}]", [box[mode == "default"], _gv(eng, grads, g.conv_first.bias)],
                        want)
    for label, img, ty, tx in _edge_teeth_tiles(b, h, w):
        vw, _ = _tile_from(V, V, img, ty, tx)
        sw = F.pad(x[img, 0].double(), (0, 8, 0, 8))[8 * ty:8 * ty + 8, 8 * tx:8 * tx + 8, None]
        m = int(((R - _tile_delta(vw, sw).permute(2, 1, 0)).float() != want[0]).sum())
        print(f"conv_first: without {label} {m} of {R.numel()} compared values differ")
        assert m >= 0.9 * R.numel()
    assert bad == 0


# ------------------------------------------------------------------------------------------- dense-block data gradients
# _rdb_backward of block (i, r) at the F = 32 training shape, nb = 2: r = 2 writes ring[1] (with RDB2's conv5 bias,
# 0.2), r = 1 ring[0] (RDB1's, 0.2), r = 0 of i = 1 ring[2] in place of its own r2 input (RDB3 of i = 0, 0.04), r = 0
# of i = 0 d_fea.  Exactness needs three arrangements, the factors not being powers of two:
#  * activations x1..x4 are positive, so LeakyReLU' (slope 0.2) multiplies by 1;
#  * conv5's weights are 5 m (r < 2) or 25 m (r = 2): the packed data-gradient weights bf16(fl32(s5) * w) are then m;
#  * RDB3's block-input gradient adds 0.2 * G[4] by one FMA, exact only where the result is a nonzero integer or the
#    accumulator is zero.  So G[4] = 5 u (u the +-1 "dy" field) and RDB3's weights on x0 are zero: the FMA adds
#    u (1 + 1.5e-8) to an exact 0 and rounds to u.  (Even x0 weights would keep acc + u odd, but every dY_j of RDB3 is
#    then +-5, and a column of the block-input gradient would sum ~10 per pixel, 2.7e7 in all: over the 2^24 budget of
#    RDB2's conv5 bias sum.  The x0 accumulation is covered by the r = 0 / 1 cases and the production-valued case.)
# Weights (m): every input column of a layer has one +-1 at a random (output channel, tap).  In RDB3, where dY5 is 5 u,
# only conv_{j+1} reads x_j (j >= 1), so that every dY_j is a shifted +-5 field and its column sums stay below 2^24.
DGRAD_CASES = [(1, 2), (1, 1), (1, 0), (0, 0)]


def _dense_int_weights(gen, f):
    """Integer dense-block weights (see above); returns {(i, r, k): m}, the effective (folded) weights."""
    g = torch.Generator().manual_seed(5)
    eff = {}
    with torch.no_grad():
        for i, rrdb in enumerate(gen.rrdb):
            for r, rdb in enumerate((rrdb.RDB1, rrdb.RDB2, rrdb.RDB3)):
                for k in range(1, 6):
                    conv = getattr(rdb, f"conv{k}")
                    n, cin = conv.weight.shape[:2]
                    m = torch.zeros(n, cin, 9)
                    o = torch.randint(0, n, (cin,), generator=g)
                    t = torch.randint(0, 9, (cin,), generator=g)
                    sign = (torch.randint(0, 2, (cin,), generator=g) * 2 - 1).float()
                    keep = torch.ones(cin)
                    if r == 2:
                        j = torch.arange(cin) // f
                        keep = ((j == k - 1) & (j > 0)).float()
                    m[o, torch.arange(cin), t] = sign * keep
                    m = m.view(n, cin, 3, 3)
                    conv.weight.copy_(m * (1.0 if k < 5 else 5.0 if r < 2 else 25.0))
                    eff[(i, r, k)] = m
    return eff


def _dgrad_sums(dy: torch.Tensor, ws) -> torch.Tensor:
    """sum_k sum_tap dY_k[p - off(tap)][o] W_k[o][i][tap] in float64: dy [B, H, W, K] (the concatenated slots the layer
    reads), ws the matching [f, n_i, 3, 3] weights in slot order."""
    B, H, W, K = dy.shape
    wcat = torch.cat([w.double() for w in ws], dim=0).to(dy.device)  # [K, n_i, 3, 3]
    out = torch.zeros(B, H, W, wcat.shape[1], dtype=torch.float64, device=dy.device)
    for b in range(B):
        yp = F.pad(dy[b].double(), (0, 0, 1, 1, 1, 1))
        for t in range(9):
            ky, kx = divmod(t, 3)
            out[b] += (yp[2 - ky:2 - ky + H, 2 - kx:2 - kx + W].reshape(H * W, K) @ wcat[:, :, ky, kx]).view(H, W, -1)
    return out


def test_conv5_fold_is_exact_for_the_chosen_weights():
    """bf16(fl32(0.2) * fl32(5 m)) = m and bf16(fl32(0.04) * fl32(25 m)) = m for every m in [-8, 8] (the packing's
    rounding of conv5's data-gradient weights)."""
    m = torch.arange(-8, 9).float()
    for s5, mult in ((0.2, 5.0), (0.04, 25.0)):
        packed = (torch.tensor(s5, dtype=torch.float32) * (m * mult)).to(torch.bfloat16).float()
        assert torch.equal(packed, m), (s5, packed - m)


@pytest.mark.gpu
@pytest.mark.parametrize("i,r", DGRAD_CASES)
def test_dense_block_data_gradients_exact(dev, i, r):
    """Every stored dY1..dY4 slot and the block-input gradient equal bf16 of the float64 layer computed from the slots
    the kernels read; the fused bias sums of conv1..conv4 are exact in both modes, the previous block's conv5 bias sum
    exact in deterministic mode and bounded in the default (atomic, scaled per warp) mode."""
    from xmm_superres_denoise_b200 import _lib, ops
    from xmm_superres_denoise_b200.engine_train import TrainEngine

    f, b, h, w = 32, 16, 416, 416
    _ENGINES.clear()
    gen = _gen("dn", f, 2, dev)
    eff = _dense_int_weights(gen, f)
    for (ii, rr, k), m in eff.items():  # the fold of conv5 lands on the effective weights (test_conv5_fold_...)
        if k == 5:
            s5 = 0.04 if rr == 2 else 0.2
            conv5 = (gen.rrdb[ii].RDB1, gen.rrdb[ii].RDB2, gen.rrdb[ii].RDB3)[rr].conv5.weight
            assert torch.equal((conv5.cpu() * torch.tensor(s5, dtype=torch.float32)).to(torch.bfloat16).float(), m)
    eng = TrainEngine(gen, "dn")
    eng.arena.ensure(dev)
    bufs = eng._train_buffers(b, h, w, dev, False)
    ring, A, G = bufs["ring"], bufs["act"][3 * i + r], bufs["ring"][r]
    A.fill_(1.0)
    A[..., :f] = -3.0  # x0 is no mask: its sign must not matter
    if r == 2:
        out, s1, s2, prev = ring[1][..., 4 * f:], 0.2, 0.0, (eng._rdb(i, 1).conv5, 0.2)
    elif r == 1:
        out, s1, s2, prev = ring[0][..., 4 * f:], 1.0, 0.0, (eng._rdb(i, 0).conv5, 0.2)
    else:
        out, s1, s2 = (ring[2][..., 4 * f:] if i > 0 else bufs["d_fea"]), 1.0, 1.0
        prev = (eng._rdb(i - 1, 2).conv5, 0.04) if i > 0 else None
    g4 = torch.empty(b, h, w, f, dtype=torch.bfloat16, device=dev)
    _fill(g4, "dy", 7)
    if r == 2:
        g4 *= 5
    r2 = torch.empty_like(g4)
    _fill(r2, "x", 8)

    def setup():
        G.fill_(77.0)  # slots the layers must overwrite
        G[..., 4 * f:] = g4
        out.fill_(-55.0)
        if r == 0:
            ring[2][..., 4 * f:] = r2

    snaps = {}

    def after(mode):
        snaps[mode] = (G.clone(), out.clone())

    results = _modes(eng, dev, (b, h, w), lambda grads: eng._rdb_backward(i, r, bufs, grads, bufs["d_fea"]),
                     setup, after)
    rdb = eng._rdb(i, r)
    bad = 0
    stored_ref = None
    for mode, grads in results:
        Gs, outs = snaps[mode]
        refs = {}
        for j in range(4, 0, -1):  # dY_j from the stored dY_{j+1..5}, mask 1
            refs[j] = _dgrad_sums(Gs[..., j * f:], [eff[(i, r, k)][:, j * f:(j + 1) * f] for k in range(j + 1, 6)])
        acc = _dgrad_sums(Gs, [eff[(i, r, k)][:, :f] for k in range(1, 6)])
        ref0 = acc + s1 * g4.double() + (s2 * r2.double() if s2 else 0.0)
        for j, ref in list(refs.items()) + [(0, ref0)]:
            assert float(ref.abs().sum(dim=(0, 1, 2)).max()) < EXACT, f"({i}, {r}) layer {j}: column sums over 2^24"
        got = [Gs[..., (j - 1) * f:j * f] for j in range(4, 0, -1)] + [outs]
        want = [refs[j].float().to(torch.bfloat16) for j in range(4, 0, -1)] + [ref0.float().to(torch.bfloat16)]
        n = sum(t.numel() for t in want)
        nb = sum(int((g != wv).sum()) for g, wv in zip(got, want))
        print(f"dense ({i}, {r}) [{mode}] dY4..dY1 + block-input gradient: {n} elements compared, {nb} mismatches")
        for j, g, wv in zip([4, 3, 2, 1, 0], got, want):
            ne = (g != wv).nonzero()[:3].tolist()
            for idx in ne:
                print(f"  layer {j} at (b, y, x, c) {tuple(idx)}: got {float(g[tuple(idx)])}, "
                      f"want {float(wv[tuple(idx)])}")
        bad += nb
        # bias sums: conv1..conv4 (scale 1) and the previous block's conv5 (s5)
        gb = [_gv(eng, grads, getattr(rdb, f"conv{j}").bias) for j in range(1, 5)]
        wb = [refs[j].sum(dim=(0, 1, 2)).float() for j in range(1, 5)]
        if prev is not None:
            S, sc = ref0.sum(dim=(0, 1, 2)), prev[1]
            gp = _gv(eng, grads, prev[0].bias)
            if mode == "default":
                K = ops.det_slots(_lib.DET_CONV3X3, b, h, w, 32)
                bound = gamma(K + 1) * sc * ref0.abs().sum(dim=(0, 1, 2)) + U * (sc * S).abs()
                ratio = float(((gp.double() - sc * S).abs() / bound).max())
                print(f"dense ({i}, {r}) [{mode}] conv5 bias of the previous block (atomic, scale {sc}, K = {K}): "
                      f"max |err| / bound = {ratio:.3f}")
                assert ratio <= 1.0
            else:
                gb.append(gp)
                wb.append(_scaled(S, sc))
        bad += _compare(f"dense ({i}, {r}) [{mode}] bias sums", gb, wb)
        if stored_ref is None:
            stored_ref = [refs[j] for j in range(1, 5)] + [ref0]
    assert bad == 0
    # teeth of the bias sums: one 8x8 tile of the integrand removed moves >= 90 % of them
    c = m = 0
    for label, img, ty, tx in _edge_teeth_tiles(b, h, w):
        for ref in stored_ref:
            t = ref[img, 8 * ty:8 * ty + 8, 8 * tx:8 * tx + 8].sum(dim=(0, 1))
            c, m = c + t.numel(), m + int((t != 0).sum())
    print(f"dense ({i}, {r}): a tile removed moves {m} of {c} bias sums")
    assert m >= 0.9 * c


def _dgrad_abs(dy: torch.Tensor, ws) -> torch.Tensor:
    """S of helpers.assert_bf16_elementwise for a data-gradient layer: sum |dY| |W| over each output's window."""
    return _dgrad_sums(dy.abs(), [w.abs() for w in ws])


@pytest.mark.gpu
@pytest.mark.parametrize("i,r", [(1, 2), (0, 0)])
def test_dense_block_data_gradients_production_values(dev, i, r):
    """_rdb_backward with the generator's own initial weights, activations of both signs (LeakyReLU' slope 0.2 in
    play), RDB3's s1 = 0.2 and the folded 0.04 / 0.2: every stored dY_j and the block-input gradient per element
    within ulp_bf16 + C_TC * S of float64 from the stored slots (images 0, 7 and 15 checked)."""
    from helpers import C_TC, assert_bf16_elementwise
    from xmm_superres_denoise_b200.engine_train import TrainEngine

    f, b, h, w = 32, 16, 416, 416
    _ENGINES.clear()
    gen = _gen("dn", f, 2, dev)
    eng = TrainEngine(gen, "dn")
    eng.arena.ensure(dev)
    bufs = eng._train_buffers(b, h, w, dev, False)
    ring, A, G = bufs["ring"], bufs["act"][3 * i + r], bufs["ring"][r]
    g = torch.Generator(device=dev).manual_seed(17)
    A.copy_(torch.randn(A.shape, generator=g, device=dev).to(torch.bfloat16))
    G.copy_((torch.randn(G.shape, generator=g, device=dev) * 0.1).to(torch.bfloat16))
    s5 = 0.04 if r == 2 else 0.2
    if r == 2:
        out, s1, s2 = ring[1][..., 4 * f:], 0.2, 0.0
    else:
        out, s1, s2 = (ring[2][..., 4 * f:] if i > 0 else bufs["d_fea"]), 1.0, 1.0
        ring[2][..., 4 * f:] = (torch.randn(b, h, w, f, generator=g, device=dev) * 0.1).to(torch.bfloat16)
    sel = [0, 7, 15]
    g4, r2 = G[sel][..., 4 * f:].double(), ring[2][sel][..., 4 * f:].double()
    grads = eng._grad_views(dev)
    eng._rdb_backward(i, r, bufs, grads, bufs["d_fea"])
    torch.cuda.synchronize()
    rdb = eng._rdb(i, r)
    fold = torch.tensor(s5, dtype=torch.float32, device=dev)  # the packing's fl32(s5) * w, then bf16
    wq = {k: (getattr(rdb, f"conv{k}").weight * (fold if k == 5 else 1.0)).to(torch.bfloat16).double()
          for k in range(1, 6)}
    Gs, As, outs = G[sel], A[sel], out[sel]
    nchw = lambda t: t.permute(0, 3, 1, 2)  # noqa: E731
    for j in range(4, 0, -1):
        ws = [wq[k][:, j * f:(j + 1) * f] for k in range(j + 1, 6)]
        mask = torch.where(As[..., j * f:(j + 1) * f].double() > 0, 1.0, 0.2)
        ref = mask * _dgrad_sums(Gs[..., j * f:], ws)
        S = mask * _dgrad_abs(Gs[..., j * f:], ws)
        rr = assert_bf16_elementwise(nchw(Gs[..., (j - 1) * f:j * f]), nchw(ref), nchw(S), C_TC,
                                     what=f"dense ({i}, {r}) dY{j}")
        print(f"dense ({i}, {r}) production values dY{j}: max |err|/bound = {rr:.3f}")
    ws = [wq[k][:, :f] for k in range(1, 6)]
    ref = _dgrad_sums(Gs, ws) + s1 * g4 + s2 * r2
    S = _dgrad_abs(Gs, ws)
    rr = assert_bf16_elementwise(nchw(outs), nchw(ref), nchw(S), C_TC, what=f"dense ({i}, {r}) block-input gradient")
    print(f"dense ({i}, {r}) production values block-input gradient: max |err|/bound = {rr:.3f}")


@pytest.mark.gpu
def test_sr_tail_data_gradients_per_element(dev):
    """SR-2x tail of the backward at batch 16, as TrainEngine._backward launches it: d.hr (HRconv's data gradient,
    LeakyReLU' slope 0.01 of the upsampling output, inverse pixel-shuffle store into d_up0), d.up0 (the upsampling conv's
    data gradient over the 128 un-shuffled channels) and d.trunk (into RDB3's G[4], with its fused bias sum), each per
    element from the buffer it read (images 0, 7 and 15 checked)."""
    from helpers import C_TC, assert_bf16_elementwise

    f, b, h, w = 32, 16, 416, 416
    eng = _engine("sr", f, dev)
    g = eng.gen
    bufs = eng._train_buffers(b, h, w, dev, False)
    gr = torch.Generator(device=dev).manual_seed(23)
    bufs["d_hr"].copy_((torch.randn(bufs["d_hr"].shape, generator=gr, device=dev) * 0.1).to(torch.bfloat16))
    bufs["up0"].copy_(torch.randn(bufs["up0"].shape, generator=gr, device=dev).to(torch.bfloat16))
    grads = eng._grad_views(dev)
    ring = bufs["ring"]
    eng._run(eng._conv("d.hr", bufs["d_hr"], 0, f, bufs["d_up0"], 0, mask=bufs["up0"], mask_coff=0, mask_slope=0.01,
                       pixel_shuffle=2))
    eng._run(eng._conv("d.up0", bufs["d_up0"], 0, 4 * f, bufs["d_trunk"], 0))
    eng._run(eng._conv("d.trunk", bufs["d_trunk"], 0, f, ring[2], 4 * f,
                       **eng._bias_sum(grads, eng._rdb(eng.nb - 1, 2).conv5, 0.04)))
    torch.cuda.synchronize()
    sel = [0, 7, 15]
    nchw = lambda t: t.permute(0, 3, 1, 2)  # noqa: E731
    bq = lambda conv: conv.weight.to(torch.bfloat16).double()  # noqa: E731

    def check(tag, got, ref, S):
        rr = assert_bf16_elementwise(nchw(got), nchw(ref), nchw(S), C_TC, what=tag)
        print(f"SR tail {tag}: max |err|/bound = {rr:.3f}")

    def unshuffle(t):  # [n, 2h, 2w, f] -> [n, h, w, 4f], channel (2 (y & 1) + (x & 1)) f + c
        n = t.shape[0]
        return t.reshape(n, h, 2, w, 2, f).permute(0, 1, 3, 2, 4, 5).reshape(n, h, w, 4 * f)

    d_hr = bufs["d_hr"][sel]
    mask = torch.where(bufs["up0"][sel].double() > 0, 1.0, 0.01)
    check("d.hr (inverse pixel shuffle)", bufs["d_up0"][sel], unshuffle(mask * _dgrad_sums(d_hr, [bq(g.HRconv)])),
          unshuffle(mask * _dgrad_abs(d_hr, [bq(g.HRconv)])))
    wup = [bq(g.upsampling[0])[_perm(4 * f).to(dev)]]  # packed column j holds PixelShuffle channel 4c + g
    d_up = bufs["d_up0"][sel]
    check("d.up0", bufs["d_trunk"][sel], _dgrad_sums(d_up, wup), _dgrad_abs(d_up, wup))
    d_tr = bufs["d_trunk"][sel]
    check("d.trunk", ring[2][sel][..., 4 * f:], _dgrad_sums(d_tr, [bq(g.trunk_conv)]),
          _dgrad_abs(d_tr, [bq(g.trunk_conv)]))
