"""Every tensor-core kernel variant and every tile-schedule path, bit-exactly (-m gpu, except the coverage guard).

Which of the 34 instantiations of gemm_tc_kernel a call runs, and how its tiles are scheduled (one round of whole
tiles, a K-split tail of 2-4 parts folded into C in order, a half-width tail, several rounds with a whole-tile
remainder, exact rounds), is decided by the size heuristics in capi.cu.  The parity tests only see what those pick
for their shapes.  Here every target forces its kernel with the tuning hooks, derives a shape from the device's SM
count that lands on one schedule path, and asserts both through last_kernel() and last_schedule(), so a changed
heuristic fails the test instead of quietly testing another kernel.

Small-integer data (entries in [-4, 4] with some exact zeros, k <= 4096) makes every floating-point kind exact:
every product and every partial sum is an integer below 2^24, so tf32 truncation loses nothing, the second and
third bf16 / fp16 planes of the split modes are zero, the F16X2 power-of-two scalings are exact and every fold is
an exact fp32 add.  The output must then equal the integer product bit for bit over the whole matrix, which
catches a fold in the wrong order, a tile stored twice or a stale read of C.  Integer data says nothing about
which plane product goes where, so a random-data check against the oracle within the per-mode bars stays beside it.
"""
import re
import zlib
from dataclasses import dataclass

import numpy as np
import pytest

import _libs
from test_gpu_parity import TOL_BF16, TOL_F16X2, TOL_TF32, TOL_X2, TOL_X3, rel

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

# schedule paths: one round of whole tiles, a K-split tail of 2 / 3 / 4 parts, a half-width tail, several rounds
# with a whole-tile remainder, an exact number of rounds
PATHS = ("one", "split2", "split3", "split4", "halfn", "whole", "exact")
# kind: (kernel-name prefix, input type, output type, k-block)
KINDS = {
    "tf32": ("tc_tf32", "f32", "f32", 32),
    "bf16": ("tc_bf16", "bf16", "f32", 64),
    "bf16o": ("tc_bf16_obf16", "bf16", "bf16", 64),
    "s8": ("tc_s8", "s8", "s32", 128),
    "s8rq": ("tc_s8_requant", "s8", "s8", 128),
    "x3": ("tc_bf16x3", "f32", "f32", 32),
    "x2": ("tc_bf16x2", "f32", "f32", 32),
    "f16x2": ("tc_f16x2", "f32", "f32", 32),
}
SPLIT_MODES = ("x3", "x2", "f16x2")
F32_MODES = ("tf32",) + SPLIT_MODES
# tile configurations: 1-CTA 128 x BN tiles, CTA pairs (256 x 256) with the default 8 epilogue warps ("pair") or
# with 4 ("pair4", b200_gemm_debug_set_epilogue bit 1; the split modes' pair kernels always drain with 8)
SUFFIX = {"128": "_128x128", "192": "_128x192", "256": "_128x256", "pair": "_2cta_256x256", "pair4": "_2cta_256x256"}


@dataclass(frozen=True)
class Target:
    kind: str
    cfg: str
    path: str

    @property
    def pair(self):
        return self.cfg.startswith("pair")

    @property
    def kernel(self):
        e8 = self.cfg == "pair" and self.kind not in SPLIT_MODES
        return KINDS[self.kind][0] + SUFFIX[self.cfg] + ("_e8" if e8 else "")

    @property
    def bn(self):
        return 256 if self.pair else int(self.cfg)

    @property
    def epilogue_warps(self):
        return 8 if self.kind in SPLIT_MODES or self.cfg == "pair" else 4

    @property
    def id(self):
        return f"{self.kernel}-{self.path}"


# Tile configurations of each kind: 128x256 is ignored for BF16X3 and 128x192 for int8 (192 is not a whole number of
# 128-byte int8 column blocks).
CFGS = {"tf32": ("128", "192", "256", "pair", "pair4"), "bf16": ("128", "192", "256", "pair", "pair4"),
        "bf16o": ("128", "192", "256", "pair", "pair4"), "s8": ("128", "256", "pair", "pair4"),
        "s8rq": ("128", "256", "pair", "pair4"), "x3": ("128", "192", "pair"), "x2": ("128", "192", "256", "pair"),
        "f16x2": ("128", "192", "256", "pair")}


def dispatchable(kind, cfg, path):
    """Paths the dispatcher can produce: only fp32 / int32 outputs fold a K-split tail into C, and a half-width tail
    needs BN/2 per CTA to be a whole number of 128-byte B column blocks (not so for 192-wide 16-bit tiles, nor for
    int8 tiles other than 1-CTA 128x256)."""
    ind, outd = KINDS[kind][1:3]
    if path.startswith("split"):
        return outd in ("f32", "s32")
    if path == "halfn":
        if ind == "s8":
            return cfg == "256"
        return cfg != "192" or kind == "tf32"
    return True


# Every kernel the dispatcher can produce on every schedule path it can run.
TARGETS = tuple(Target(kind, cfg, path) for kind in KINDS for cfg in CFGS[kind] for path in PATHS
                if dispatchable(kind, cfg, path))
# strict fp32 (CUDA-core FFMA) kernels: b200_gemm_debug_set_ffma_variant bit 1 = 128x256 fat-thread kernel,
# bit 0 = half tiles in the last partial round
FFMA_TARGETS = {0: "ffma_128x128x32_tma", 1: "ffma_128x128x32_tma", 2: "ffma_fat_128x256x32_tma",
                3: "ffma_fat_128x256x32_tma"}
# operands the TMA cannot address (16-byte misaligned base) go to the CUDA-core generic kernels
GENERIC_TARGETS = (("generic_f32_64x64", "strict"), ("generic_f32_64x64", "tf32"), ("generic_bf16_64x64", "f32"),
                   ("generic_bf16_64x64", "bf16"), ("generic_s8_64x64", "s32"), ("generic_s8_requant_64x64", "s8"))


# ---- CPU-only guard: a kernel the dispatcher can emit but no target reaches fails on any machine ----------------
def dispatcher_kernel_names():
    import glob
    import os
    src = "".join(open(f).read() for f in sorted(glob.glob(os.path.join(_libs.ROOT, _libs.PKG, "csrc", "*.cu*"))))
    macro = re.search(r"#define TC_PLAIN\(KIND, OUT, NAME\)(.*?)\n\n", src, re.S).group(1)
    suffixes = set(re.findall(r'NAME\s*"(_\w+)"', macro))
    plain = set(re.findall(r'TC_PLAIN\(\s*\w+\s*,\s*\w+\s*,\s*"(\w+)"\s*\)', src))
    names = {n + s for n in plain for s in suffixes}
    names |= set(re.findall(r'"((?:tc|ffma|generic)_\w+)"', src)) - plain
    return names, plain, suffixes


def test_every_dispatched_kernel_has_a_target():
    names, plain, suffixes = dispatcher_kernel_names()
    assert plain == {"tc_bf16", "tc_bf16_obf16"} and len(suffixes) == 5, (plain, suffixes)
    covered = {t.kernel for t in TARGETS} | set(FFMA_TARGETS.values()) | {n for n, _ in GENERIC_TARGETS}
    missing = sorted(names - covered - {"tc_mxf4_128x128"})       # the MXFP4 kernel has its own tests (test_mxf4.py)
    assert not missing, f"kernels without a target in tests/test_tc_variants.py: {missing}"
    assert not covered - names, f"targets naming kernels the dispatcher cannot emit: {sorted(covered - names)}"
    assert len([n for n in names if n.startswith("tc_") and n != "tc_mxf4_128x128"]) == 34
    assert len(set(TARGETS)) == len(TARGETS)


# ---- hooks ----------------------------------------------------------------------------------------------------
def reset_hooks(lib):
    lib.b200_gemm_debug_set_bn(0)
    lib.b200_gemm_debug_set_cta_group(0)
    lib.b200_gemm_debug_set_split_tail(1)
    lib.b200_gemm_debug_set_dynamic_sched(0)
    lib.b200_gemm_debug_set_epilogue(0)
    lib.b200_gemm_debug_set_pdl(1)
    lib.b200_gemm_debug_set_group_rows(0)
    lib.b200_gemm_debug_set_ffma_variant(-1)
    lib.b200_gemm_debug_set_split_chunk(-1, -1)


@pytest.fixture(autouse=True)
def _restore_hooks(gemm):
    """Every process-global hook goes back to its default whatever the test did, so a failing case cannot leak
    forced settings into the rest of the session."""
    try:
        yield
    finally:
        reset_hooks(gemm.lib)


def force(lib, t):
    lib.b200_gemm_debug_set_cta_group(2 if t.pair else 1)
    lib.b200_gemm_debug_set_bn(0 if t.pair else t.bn)
    lib.b200_gemm_debug_set_epilogue(2 if t.cfg == "pair4" else 0)


@pytest.fixture(scope="module")
def sms():
    assert torch.cuda.is_available()
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- shapes derived from the SM count -------------------------------------------------------------------------
@dataclass
class Shape:
    m: int
    n: int
    k: int
    tile_m: int
    tiles_m: int
    tiles_n: int
    units: int


def tile_range(path, units, cap):
    """Tile counts that put a launch of `units` CTAs (or pairs) on `path` (capi.cu launch_tc); `cap`: most tail
    tiles the K-split flag slots hold."""
    if path.startswith("split"):
        s = int(path[-1])
        lo, hi = (1, units // 4) if s == 4 else (units // (s + 1) + 1, units // s)
        return lo, min(hi, cap)
    return {"one": (units // 2 + 1, units - 1), "halfn": (units + 1, units + units // 2),
            "whole": (units + units // 2 + 1, 2 * units - 1), "exact": (units, units)}[path]


def factor(lo, hi, tile_m, bn, seed):
    """tiles_m x tiles_n with a product in [lo, hi]: the largest product with at least two tiles each way (one of the
    two most nearly square such grids, by seed), else the lowest product as it comes."""
    for T in range(hi, lo - 1, -1):
        fs = [(tm, T // tm) for tm in range(2, T // 2 + 1) if T % tm == 0 and T // tm >= 2]
        if fs:
            fs.sort(key=lambda f: abs(f[0] * tile_m - f[1] * bn))
            return fs[seed % min(2, len(fs))]
    return 1, lo


def shape_for(t, sms):
    seed = zlib.crc32(t.id.encode())
    cg = 2 if t.pair else 1
    tile_m, units = 128 * cg, sms // cg
    bk = KINDS[t.kind][3]
    cap = 1024 // (cg * t.epilogue_warps)
    tm, tn = factor(*tile_range(t.path, units, cap), tile_m, t.bn, seed)
    dm = (37, 141, 90, 5)[seed % 4] % tile_m if tm > 1 else (37, 90, 5)[seed % 3]
    dn = (21, t.bn // 2 + 3, 1, t.bn - 9)[(seed >> 4) % 4]
    if t.pair and tn == 1:
        dn = min(dn, 100)          # a CTA pair needs n > 128
    if t.path.startswith("split"):
        k = 8 * int(t.path[-1]) * bk - 7     # just enough k-blocks for the split (>= 8 per part)
    else:
        k = (19, 301, 77, 150)[(seed >> 8) % 4]
    return Shape(tm * tile_m - dm, tn * t.bn - dn, k, tile_m, tm, tn, units)


def check_schedule(gemm, t, sh, **over):
    s = gemm.last_schedule()
    assert s is not None, gemm.last_kernel()
    tiles = sh.tiles_m * sh.tiles_n
    rem = tiles % sh.units
    split = int(t.path[-1]) if t.path.startswith("split") else 1
    halfn = int(t.path == "halfn")
    full = tiles - rem if (split > 1 or halfn) else tiles
    items = full + (tiles - full) * (2 if halfn else split)
    want = dict(tile_m=sh.tile_m, bn=t.bn, cta_group=2 if t.pair else 1, epilogue_warps=t.epilogue_warps,
                tiles=tiles, grid_units=min(items, sh.units), full_tiles=full, split=split, halfn=halfn, dynamic=0)
    want.update(over)
    assert s == want, (gemm.last_kernel(), t.path, s)
    assert {"one": 0 < tiles < sh.units, "whole": tiles > sh.units and rem, "exact": rem == 0,
            "halfn": tiles > sh.units}.get(t.path, tiles < sh.units)


# ---- operands and calls -------------------------------------------------------------------------------------
TORCH_DT = {"f32": torch.float32, "bf16": torch.bfloat16, "s8": torch.int8, "s32": torch.int32}
SENTINEL = {"f32": 12345.0, "bf16": -7.0, "s8": 90, "s32": 0x5A5A5A5A}


def padded(rows, cols, dt, fill=None):
    """A rows x cols view of a buffer whose pitch is a multiple of 16 elements past cols (TMA-able, 16-byte vector
    stores), and the buffer: the columns past the view must come out untouched."""
    pitch = (cols + 15) // 16 * 16 + 16
    buf = torch.empty((rows, pitch), dtype=TORCH_DT[dt], device="cuda")
    if fill is not None:
        buf.fill_(fill)
    return buf[:, :cols], buf


def small_ints(rows, cols, dt, gen):
    """Entries in [-4, 4] (one in nine an exact zero) plus one all-zero row and one all-zero column."""
    v, buf = padded(rows, cols, dt)
    buf.copy_(torch.randint(-4, 5, buf.shape, generator=gen, device="cuda").to(buf.dtype))
    v[rows // 3].zero_()
    v[:, cols // 2].zero_()
    return v


def random_operands(oracle, t, sh, seed):
    """Random data in the kind's input type: uniform(-1, 1) (bf16: rounded) or full-range int8, as numpy + views."""
    ind = KINDS[t.kind][1]
    if ind == "s8":
        a, b = _libs.gen_s8(oracle, sh.m, sh.k, seed), _libs.gen_s8(oracle, sh.k, sh.n, seed + 1)
    else:
        a, b = _libs.gen_f32(oracle, sh.m, sh.k, seed), _libs.gen_f32(oracle, sh.k, sh.n, seed + 1)
        if ind == "bf16":
            a, b = _libs.round_bf16(oracle, a), _libs.round_bf16(oracle, b)
    A, _ = padded(sh.m, sh.k, ind)
    B, _ = padded(sh.k, sh.n, ind)
    A.copy_(torch.from_numpy(a).to(A.dtype))
    B.copy_(torch.from_numpy(b).to(B.dtype))
    return a, b, A, B


def requant_params(m, seed):
    """Power-of-two scales and half-integer biases: odd accumulators land on .5 ties (rounding mode matters)."""
    rng = np.random.default_rng(seed)
    scales = np.float32(2.0) ** -rng.integers(1, 7, m).astype(np.float32)
    bias = (rng.integers(-8, 9, m) * 0.5).astype(np.float32)
    return scales, bias


MODE = {"tf32": "F32_TF32", "x3": "F32_BF16X3", "x2": "F32_BF16X2", "f16x2": "F32_F16X2"}


def call(gemm, t, A, B, out, rq=None, packed=None, accumulate=False):
    if t.kind in MODE:
        if packed is not None:
            return gemm.gemm_f32_packed(A, packed, out=out, accumulate=accumulate)
        return gemm.gemm_f32(A, B, out=out, mode=getattr(gemm, MODE[t.kind]), accumulate=accumulate)
    assert not accumulate
    if t.kind in ("bf16", "bf16o"):
        return gemm.gemm_bf16(A, B, out=out)
    if t.kind == "s8":
        return gemm.gemm_s8s32(A, B, out=out)
    return gemm.gemm_s8s8_requant(A, B, rq[0], rq[1], out=out)


def check_rows(sh):
    """One row in every tile row (at a varying offset), at most 12 of them, plus the first and last rows of the last
    tile row: every tile column is seen in every row checked."""
    step = max(1, sh.tiles_m // 12)
    rows = {min(r * sh.tile_m + (r * 53) % sh.tile_m, sh.m - 1) for r in range(0, sh.tiles_m, step)}
    rows |= {0, (sh.tiles_m - 1) * sh.tile_m, sh.m - 1}
    return np.array(sorted(rows))


def padding_intact(buf, n, fill):
    return bool((buf[:, n:] == fill).all())


def pid(t):
    return t.id


# ---- c. exact data: every target, whole matrix ------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("t", TARGETS, ids=pid)
def test_exact_integer_data(gemm, oracle, sms, t):
    sh = shape_for(t, sms)
    _, ind, outd, _ = KINDS[t.kind]
    g = torch.Generator(device="cuda").manual_seed(zlib.crc32(t.id.encode()))
    A, B = small_ints(sh.m, sh.k, ind, g), small_ints(sh.k, sh.n, ind, g)
    P = A.double() @ B.double()                       # integers far below 2^53: exact in any order
    rq = None
    if t.kind == "s8rq":
        scales, bias = requant_params(sh.m, 5)
        rq = (torch.from_numpy(scales).cuda(), torch.from_numpy(bias).cuda())
    C, Cbuf = padded(sh.m, sh.n, outd, SENTINEL[outd])
    force(gemm.lib, t)
    call(gemm, t, A, B, C, rq)
    assert gemm.last_kernel() == t.kernel
    check_schedule(gemm, t, sh)
    rows = check_rows(sh)
    a_rows, b = A[torch.from_numpy(rows).cuda()].cpu(), B.contiguous().cpu()
    if ind == "s8":
        oracle_rows = _libs.ref_s8(oracle, a_rows.numpy(), b.numpy())
    else:
        oracle_rows = _libs.ref_f64(oracle, a_rows.float().numpy(), b.float().numpy())
    if outd == "f32":
        want = P.float()
        assert np.array_equal(C.cpu().numpy()[rows], oracle_rows.astype(np.float32))
    elif outd == "s32":
        want = P.int()
        assert np.array_equal(C.cpu().numpy()[rows], oracle_rows)
    elif outd == "bf16":                             # exact fp32 accumulation, then one RNE rounding
        want = torch.from_numpy(_libs.round_bf16(oracle, P.float().cpu().numpy())).cuda().bfloat16()
        assert np.array_equal(C.float().cpu().numpy()[rows], _libs.round_bf16(oracle, oracle_rows.astype(np.float32)))
    else:
        want = torch.from_numpy(_libs.requant_s8(oracle, P.int().cpu().numpy(), scales, bias)).cuda()
        assert np.array_equal(C.cpu().numpy()[rows], _libs.requant_s8(oracle, oracle_rows, scales[rows], bias[rows]))
    assert torch.equal(C, want), (t.kernel, (C != want).nonzero()[:8].tolist())
    assert padding_intact(Cbuf, sh.n, SENTINEL[outd])
    if t.kind in SPLIT_MODES:                        # the same kernel from a pre-split B
        pk = gemm.PackedB(B, getattr(gemm, MODE[t.kind]))
        C2, Cbuf2 = padded(sh.m, sh.n, outd, SENTINEL[outd])
        call(gemm, t, A, None, C2, packed=pk)
        pk.close()
        assert gemm.last_kernel() == t.kernel
        check_schedule(gemm, t, sh)
        assert torch.equal(C2, want) and padding_intact(Cbuf2, sh.n, SENTINEL[outd])


# ---- d. random data: every target, row subset against the oracle within the per-mode bars ---------------------------
TOL = {"tf32": TOL_TF32, "bf16": TOL_BF16, "x3": TOL_X3, "x2": TOL_X2, "f16x2": TOL_F16X2}


@gpu
@pytest.mark.parametrize("t", TARGETS, ids=pid)
def test_random_data(gemm, oracle, sms, t):
    sh = shape_for(t, sms)
    outd = KINDS[t.kind][2]
    a, b, A, B = random_operands(oracle, t, sh, 101)
    rq = None
    if t.kind == "s8rq":
        scales, bias = requant_params(sh.m, 7)
        scales *= np.float32(2.0 ** -10)             # full-range int8 accumulators back into [-128, 127] mostly
        rq = (torch.from_numpy(scales).cuda(), torch.from_numpy(bias).cuda())
    C, Cbuf = padded(sh.m, sh.n, outd, SENTINEL[outd])
    force(gemm.lib, t)
    call(gemm, t, A, B, C, rq)
    assert gemm.last_kernel() == t.kernel
    check_schedule(gemm, t, sh)
    rows = check_rows(sh)
    got = C.float().cpu().numpy()[rows] if outd == "bf16" else C.cpu().numpy()[rows]
    if KINDS[t.kind][1] == "s8":
        c32 = _libs.ref_s8(oracle, a[rows], b)
        want = c32 if outd == "s32" else _libs.requant_s8(oracle, c32, scales[rows], bias[rows])
        assert np.array_equal(got, want)
    else:
        ref = _libs.ref_f64(oracle, a[rows], b)
        if outd == "bf16":      # one RNE rounding of the fp32 accumulator: half an ulp = 2^-9 relative, elementwise
            assert np.all(np.abs(got - ref) <= np.abs(ref) * 2.0 ** -8 + TOL_BF16 * np.abs(ref).max())
        else:
            assert rel(got, ref) <= TOL[t.kind], (t.kernel, rel(got, ref))
    assert padding_intact(Cbuf, sh.n, SENTINEL[outd])


# ---- e. epilogue forms across the schedule paths (fp32-output kinds, exact data) ------------------------------------
@gpu
@pytest.mark.parametrize("t", [t for t in TARGETS if t.kind in F32_MODES], ids=pid)
def test_epilogue_forms(gemm, sms, t):
    """C += A*B and C = alpha*A*B + beta*C on an integer C, exact in fp32.  With beta = 0, C starts as NaN: part 0 of a
    K-split tile must not read it and every later part must add to what the earlier ones stored."""
    sh = shape_for(t, sms)
    md = getattr(gemm, MODE[t.kind])
    g = torch.Generator(device="cuda").manual_seed(zlib.crc32(t.id.encode()) + 1)
    A, B = small_ints(sh.m, sh.k, "f32", g), small_ints(sh.k, sh.n, "f32", g)
    P = A.double() @ B.double()
    C0, C0buf = padded(sh.m, sh.n, "f32")
    C0buf.copy_(torch.randint(-64, 65, C0buf.shape, generator=g, device="cuda").float())
    force(gemm.lib, t)
    Cbuf = C0buf.clone()
    C = Cbuf[:, :sh.n]
    gemm.gemm_f32(A, B, out=C, mode=md, accumulate=True)
    assert gemm.last_kernel() == t.kernel
    check_schedule(gemm, t, sh)
    assert torch.equal(C.double(), C0.double() + P) and torch.equal(Cbuf[:, sh.n:], C0buf[:, sh.n:])
    for alpha, beta in ((0.75, 0.5), (-2.0, 0.0), (0.0, 1.0)):
        Cbuf = C0buf.clone()
        if beta == 0.0:
            Cbuf.fill_(float("nan"))
        C = Cbuf[:, :sh.n]
        gemm.gemm_f32_ex(alpha, A, B, beta, C, mode=md)
        if alpha != 0.0:
            assert gemm.last_kernel() == t.kernel
            check_schedule(gemm, t, sh)
        want = alpha * P + (beta * C0.double() if beta != 0.0 else 0.0)
        assert torch.equal(C.double(), want), (alpha, beta, (C.double() != want).nonzero()[:8].tolist())
        pad = Cbuf[:, sh.n:]
        assert bool(torch.isnan(pad).all()) if beta == 0.0 else torch.equal(pad, C0buf[:, sh.n:])


# ---- f. bf16 output = RNE of the fp32-output kernel's accumulator, bit for bit --------------------------------------
@gpu
@pytest.mark.parametrize("t", [t for t in TARGETS if t.kind == "bf16o"], ids=pid)
def test_bf16_output_rounding(gemm, oracle, sms, t):
    sh = shape_for(t, sms)
    _, _, A, B = random_operands(oracle, t, sh, 201)
    force(gemm.lib, t)
    if t.path != "halfn":
        gemm.lib.b200_gemm_debug_set_split_tail(0)  # fp32 output would otherwise cut K where bf16 output cannot
    Co = gemm.gemm_bf16(A, B, out_dtype=torch.bfloat16)
    assert gemm.last_kernel() == t.kernel
    so = gemm.last_schedule()
    Cf = gemm.gemm_bf16(A, B, out_dtype=torch.float32)
    assert gemm.last_kernel() == t.kernel.replace("tc_bf16_obf16", "tc_bf16")
    sf = gemm.last_schedule()
    assert so == sf and so["halfn"] == int(t.path == "halfn") and so["split"] == 1, (so, sf)
    want = _libs.round_bf16(oracle, Cf.cpu().numpy())
    assert np.array_equal(Co.float().cpu().numpy(), want)


# ---- g. schedule-only knobs change no bit ------------------------------------------------------------------------
def _knobs(t):
    epi = 2 if t.cfg == "pair4" else 0
    return (("dynamic", lambda L: L.b200_gemm_debug_set_dynamic_sched(1)),
            ("epilogue-4-warps", lambda L: L.b200_gemm_debug_set_epilogue(epi | 2)),
            ("epi-direct", lambda L: L.b200_gemm_debug_set_epilogue(epi | 1)),
            ("pdl-off", lambda L: L.b200_gemm_debug_set_pdl(0)),
            ("pdl-serial-prepass", lambda L: L.b200_gemm_debug_set_pdl(3)),
            ("group-rows-256", lambda L: L.b200_gemm_debug_set_group_rows(256)),
            ("dynamic+group-rows-256", lambda L: (L.b200_gemm_debug_set_dynamic_sched(1),
                                                  L.b200_gemm_debug_set_group_rows(256))))


@gpu
@pytest.mark.parametrize("t", TARGETS, ids=pid)
def test_schedule_knobs_bit_identical(gemm, oracle, sms, t):
    """Dynamic tile scheduler, 4 or 8 epilogue warps, direct epilogue stores, PDL off, the F16X2 pre-pass of B on the
    caller's stream, ragged raster groups, and repeats (the K-split flag slots and the scheduler counters rotate)
    only move work between SMs: any difference is a race or a stale read."""
    sh = shape_for(t, sms)
    outd = KINDS[t.kind][2]
    _, _, A, B = random_operands(oracle, t, sh, 301)
    rq = None
    if t.kind == "s8rq":
        scales, bias = requant_params(sh.m, 9)
        rq = (torch.from_numpy(scales * np.float32(2.0 ** -10)).cuda(), torch.from_numpy(bias).cuda())
    L = gemm.lib

    def run():
        C, _ = padded(sh.m, sh.n, outd, SENTINEL[outd])
        return call(gemm, t, A, B, C, rq)

    force(L, t)
    base = run()
    check_schedule(gemm, t, sh)
    for name, knob in _knobs(t):
        force(L, t)
        knob(L)
        for rep in range(2):
            C = run()
            dyn = int(name.startswith("dynamic"))
            if name == "epilogue-4-warps" and t.cfg == "pair" and t.kind not in SPLIT_MODES:
                assert gemm.last_kernel() == t.kernel[:-len("_e8")]
                check_schedule(gemm, t, sh, epilogue_warps=4)
            else:
                assert gemm.last_kernel() == t.kernel, name
                check_schedule(gemm, t, sh, dynamic=dyn)
            assert torch.equal(C, base), (name, rep, (C != base).nonzero()[:8].tolist())
        reset_hooks(L)
    force(L, t)
    assert torch.equal(run(), base)


# ---- h. strict FFMA: both kernels, half tiles on and off ---------------------------------------------------------
def ffma_shape(variant, sms):
    bn, slots = (256, sms) if variant >> 1 else (128, 2 * sms)
    tm, tn = factor(slots + 1, slots + slots // 2, 128, bn, variant)   # a partial last round of at most half the slots
    return Shape(tm * 128 - 45, tn * bn - 19, 301, 128, tm, tn, slots), bn


@gpu
@pytest.mark.parametrize("variant", sorted(FFMA_TARGETS))
def test_strict_ffma_variants(gemm, oracle, sms, variant):
    """C = A*B and C += A*B bit-exact against the sequential-k FMA chain, at ragged shapes with a partial last round
    (issued as half tiles when bit 0 is set)."""
    sh, bn = ffma_shape(variant, sms)
    a, b, c0 = _libs.gen_f32(oracle, sh.m, sh.k, 11), _libs.gen_f32(oracle, sh.k, sh.n, 12), _libs.gen_f32(oracle, sh.m, sh.n, 13)
    A, _ = padded(sh.m, sh.k, "f32")
    B, _ = padded(sh.k, sh.n, "f32")
    A.copy_(torch.from_numpy(a))
    B.copy_(torch.from_numpy(b))
    gemm.lib.b200_gemm_debug_set_ffma_variant(variant)
    rows = check_rows(sh)
    tiles = sh.tiles_m * sh.tiles_n
    halves = variant & 1
    full = tiles - tiles % sh.units if halves else tiles
    want_sched = dict(tile_m=128, bn=bn, cta_group=1, epilogue_warps=0, tiles=tiles, grid_units=full + 2 * (tiles - full),
                      full_tiles=full, split=1, halfn=halves, dynamic=0)
    for acc in (False, True):
        C, Cbuf = padded(sh.m, sh.n, "f32", SENTINEL["f32"])
        if acc:
            C.copy_(torch.from_numpy(c0))
        gemm.gemm_f32(A, B, out=C, mode=gemm.F32_STRICT, accumulate=acc)
        assert gemm.last_kernel() == FFMA_TARGETS[variant]
        assert gemm.last_schedule() == want_sched
        want = _libs.ref_f32_fma(oracle, a[rows], b, c0[rows] if acc else None)
        assert np.array_equal(C.cpu().numpy()[rows], want), acc
        assert padding_intact(Cbuf, sh.n, SENTINEL["f32"])


@gpu
def test_strict_ffma_variants_agree(gemm, oracle, sms):
    """Every element is the same sequential-k chain in both kernels, whole tiles or half tiles: the whole matrix agrees."""
    sh, _ = ffma_shape(1, sms)
    A, _ = padded(sh.m, sh.k, "f32")
    B, _ = padded(sh.k, sh.n, "f32")
    A.copy_(torch.from_numpy(_libs.gen_f32(oracle, sh.m, sh.k, 14)))
    B.copy_(torch.from_numpy(_libs.gen_f32(oracle, sh.k, sh.n, 15)))
    outs = []
    for v in sorted(FFMA_TARGETS):
        gemm.lib.b200_gemm_debug_set_ffma_variant(v)
        outs.append(gemm.gemm_f32(A, B, mode=gemm.F32_STRICT))
        assert gemm.last_kernel() == FFMA_TARGETS[v]
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


# ---- i. generic path; bf16 output through the tensor cores with an odd ldc ---------------------------------------------
@gpu
@pytest.mark.parametrize("name,out", GENERIC_TARGETS, ids=lambda x: x)
def test_generic_kernels(gemm, oracle, name, out):
    """Operands at a 16-byte misaligned base: the CUDA-core kernels, against the oracle; they report no schedule."""
    m, n, k = 150, 201, 133
    g = torch.Generator(device="cuda").manual_seed(3)
    if out in ("strict", "tf32"):
        a, b = _libs.gen_f32(oracle, m, k + 1, 16), _libs.gen_f32(oracle, k + 1, n + 1, 17)
        A, B = torch.from_numpy(a).cuda()[:, 1:], torch.from_numpy(b).cuda()[1:, 1:]
        C = gemm.gemm_f32(A, B, mode=gemm.F32_STRICT if out == "strict" else gemm.F32_TF32)
        ref = _libs.ref_f32_fma(oracle, np.ascontiguousarray(a[:, 1:]), np.ascontiguousarray(b[1:, 1:]))
        if out == "strict":
            assert np.array_equal(C.cpu().numpy(), ref)
        else:
            t = _libs.ref_f64(oracle, np.ascontiguousarray(a[:, 1:]), np.ascontiguousarray(b[1:, 1:]))
            assert rel(C.cpu().numpy(), t) <= TOL_TF32
    elif out in ("f32", "bf16"):
        Abuf = torch.randint(-4, 5, (m, k + 1), generator=g, device="cuda").bfloat16()
        Bbuf = torch.randint(-4, 5, (k, n), generator=g, device="cuda").bfloat16()
        A, B = Abuf[:, 1:], Bbuf
        C = gemm.gemm_bf16(A, B, out_dtype=torch.float32 if out == "f32" else torch.bfloat16)
        P = _libs.ref_f64(oracle, A.float().cpu().numpy(), B.float().cpu().numpy()).astype(np.float32)
        want = P if out == "f32" else _libs.round_bf16(oracle, P)
        assert np.array_equal(C.float().cpu().numpy(), want)
    else:
        a, b = _libs.gen_s8(oracle, m, k + 1, 18), _libs.gen_s8(oracle, k, n, 19)
        A, B = torch.from_numpy(a).cuda()[:, 1:], torch.from_numpy(b).cuda()
        c32 = _libs.ref_s8(oracle, np.ascontiguousarray(a[:, 1:]), b)
        if out == "s32":
            assert np.array_equal(gemm.gemm_s8s32(A, B).cpu().numpy(), c32)
        else:
            scales, bias = requant_params(m, 11)
            C = gemm.gemm_s8s8_requant(A, B, torch.from_numpy(scales).cuda(), torch.from_numpy(bias).cuda())
            assert np.array_equal(C.cpu().numpy(), _libs.requant_s8(oracle, c32, scales, bias))
    assert gemm.last_kernel() == name
    assert gemm.last_schedule() is None


@gpu
@pytest.mark.parametrize("cfg", ["128", "256", "pair"])
def test_bf16_output_odd_ldc(gemm, oracle, sms, cfg):
    """bf16 output with ldc = n + 3 (rows not 16-byte aligned: element stores) on the tensor-core path: exact, and the
    three padding columns of every row untouched."""
    t = Target("bf16o", cfg, "halfn")
    sh = shape_for(t, sms)
    g = torch.Generator(device="cuda").manual_seed(4)
    A, B = small_ints(sh.m, sh.k, "bf16", g), small_ints(sh.k, sh.n, "bf16", g)
    Cbuf = torch.full((sh.m, sh.n + 3), -7.0, dtype=torch.bfloat16, device="cuda")
    force(gemm.lib, t)
    gemm.gemm_bf16(A, B, out=Cbuf[:, :sh.n])
    assert gemm.last_kernel() == t.kernel
    check_schedule(gemm, t, sh)
    P = (A.double() @ B.double()).float().cpu().numpy()
    assert np.array_equal(Cbuf[:, :sh.n].float().cpu().numpy(), _libs.round_bf16(oracle, P))
    assert (Cbuf[:, sh.n:] == -7.0).all()
