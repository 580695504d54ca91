"""The bf16 tensor-core GEMMs (gemm_tcgen05.cu, gemm_skinny.cu) and the fused residual GEMM + LayerNorm (gemm_ln.cu) against
float64, through the kernel-level entries m3pc_gemm_bf16_problems and m3pc_gemm_ln_bf16_grouped.

Every GEMM case is one description -- a list of problems (M, N, K, flags, rows_per_group, bias or not) and the instance each is
expected to run on.  From it the test builds the call and a float64 reference on the same bf16 operands; the call reports which
kernel ran each problem ({kind, a, b, launch}), and the report must match the case.  Two inputs per case:

  random  per-element bar |C - ref| <= A_BAR * S + G (+ 2^-8 |ref| for bf16 outputs), where S = sum_k |a_k w_k| + |bias| + |table|
          + |residual| is computed in float64, G is the documented error of the kernel's GELU form (GELU_BAR) and 2^-8 |ref| is the
          bf16 rounding of the result (half an ulp at the bottom of a binade);
  exact   integer operands, bias, table and residual: A is one-hot over (row mod K), so every sum is an exact fp32 integer of
          magnitude <= 256 and the output must match bit for bit (GELU is dropped from the flags for this input).  A wrong row,
          column, problem, k-block, stage, table group or residual row is then an error of at least 1.

Every output has GUARD rows before and after it holding a NaN-payload pattern that must come back bit-identical; outputs start
as NaN (bf16 / fp32 without a residual) and must end finite; table buffers carry NaN rows past their last group; A, W, bias and
table must be byte-identical after the call.
"""
import ctypes as C
from dataclasses import dataclass, field

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
GUARD = 64
GELU, RES, RELU, TAB, F32 = 1, 2, 4, 8, 16
SKINNY, SINGLE, PAIR = 0, 1, 2
A_BAR = 1e-6  # fp32 accumulation and epilogue (B200: largest measured fp32-output error 0.031 x the bar at 8e-6); printed per case
# documented error of the GELU forms (common.cuh gelu_erf_fast: within 2e-6 of erf-GELU; tcgen05.cuh gelu_erf_tanh: 2.5e-5 with an
# exact tanh, plus tanh.approx's 2^-11 relative on tanh, i.e. 2^-12 |x| on GELU)
GELU_BAR = {SKINNY: lambda x: 2e-6 * (1 + x.abs()), SINGLE: lambda x: 2e-6 * (1 + x.abs()), PAIR: lambda x: 2.5e-5 + 2.0 ** -12 * x.abs()}
GUARD_F32 = 0x7FC0A5A5  # NaN payloads that no kernel writes
GUARD_BF16 = 0x7FA5


@pytest.fixture(scope="module")
def lib():
    from m3pc_b200 import _native
    return _native.lib()


@pytest.fixture(scope="module")
def nat():
    from m3pc_b200 import _native
    return _native


@dataclass
class Prob:
    M: int
    N: int
    K: int
    flags: int = 0
    rpg: int = 1
    bias: bool = True


@dataclass
class GemmCase:
    name: str
    probs: list
    expect: list  # (kind, a, b) per problem
    launches: int = None  # launches of the call, when the case is about grouping
    id: str = field(init=False)

    def __post_init__(self):
        self.id = self.name


def gcase(name, probs, expect, launches=None):
    probs = [p if isinstance(p, Prob) else Prob(*p) for p in probs]
    expect = expect if isinstance(expect, list) else [expect] * len(probs)
    return GemmCase(name, probs, expect, launches)


def out_f32(flags):
    return bool(flags & (RES | F32))


def guarded(rows, cols, dtype, fill):
    """(GUARD + rows + GUARD, cols) buffer: guard rows hold the NaN-payload pattern, the rows in between `fill`."""
    buf = torch.empty(rows + 2 * GUARD, cols, device=DEV, dtype=dtype)
    iv = torch.int32 if dtype == torch.float32 else torch.int16
    pat = GUARD_F32 if dtype == torch.float32 else GUARD_BF16
    buf.view(iv).fill_(pat)
    buf[GUARD:GUARD + rows] = fill
    return buf


def guards_intact(buf):
    iv = torch.int32 if buf.dtype == torch.float32 else torch.int16
    pat = GUARD_F32 if buf.dtype == torch.float32 else GUARD_BF16
    g = torch.cat([buf[:GUARD], buf[-GUARD:]]).view(iv)
    return bool((g == pat).all())


def bits(t):
    return t.view(torch.int32 if t.element_size() == 4 else torch.int16).clone()


def make_operands(p, g, exact):
    """A, W (bf16), bias, table (fp32, NaN rows past the last group), residual (fp32) of one problem."""
    M, N, K = p.M, p.N, p.K
    n_grp = -(-M // p.rpg)
    if exact:
        A = torch.zeros(M, K, device=DEV)
        r = torch.arange(M, device=DEV)
        A[r, r % K] = (1 + (r // K) % 3).float()
        W = torch.randint(-8, 9, (N, K), device=DEV, generator=g).float()
        bias = torch.randint(-16, 17, (N,), device=DEV, generator=g).float()
        table = torch.randint(-32, 33, (n_grp, N), device=DEV, generator=g).float()
        resid = torch.randint(-64, 65, (M, N), device=DEV, generator=g).float()
    else:
        A = torch.randn(M, K, device=DEV, generator=g)
        W = torch.randn(N, K, device=DEV, generator=g) / K ** 0.5
        bias = torch.randn(N, device=DEV, generator=g)
        table = torch.randn(n_grp, N, device=DEV, generator=g)
        resid = torch.randn(M, N, device=DEV, generator=g)
    tab = None
    if p.flags & TAB:
        tab = torch.full((n_grp + 8, N), float("nan"), device=DEV)
        tab[:n_grp] = table
    return A.bfloat16(), W.bfloat16(), bias if p.bias else None, tab, resid


def reference(p, A, W, bias, tab, resid, flags):
    """float64 C and the bound S of the bar."""
    a, w = A.double(), W.double()
    acc = a @ w.T
    S = a.abs() @ w.abs().T
    if bias is not None:
        acc = acc + bias.double()
        S = S + bias.double().abs()
    if flags & TAB:
        t = tab[:-8].double().repeat_interleave(p.rpg, dim=0)[:p.M]
        acc, S = acc + t, S + t.abs()
    pre = acc
    if flags & GELU:
        acc = torch.nn.functional.gelu(acc)
    if flags & RELU:
        acc = torch.relu(acc)
    if flags & RES:
        acc, S = acc + resid.double(), S + resid.double().abs()
    return acc, S, pre


def run_gemm(lib, nat, c, exact, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    n = len(c.probs)
    ops, outs, arr = [], [], (nat.GemmProblem * n)()
    for i, p in enumerate(c.probs):
        flags = p.flags & ~GELU if exact else p.flags
        A, W, bias, tab, resid = make_operands(p, g, exact)
        if flags & RES:
            Cb = guarded(p.M, p.N, torch.float32, resid)
        else:
            Cb = guarded(p.M, p.N, torch.float32 if out_f32(flags) else torch.bfloat16, float("nan"))
        ops.append((A, W, bias, tab, resid, flags, [bits(t) for t in (A, W, bias, tab) if t is not None]))
        outs.append(Cb)
        arr[i] = nat.GemmProblem(A.data_ptr(), W.data_ptr(), bias.data_ptr() if bias is not None else None,
                                 tab.data_ptr() if tab is not None else None, Cb[GUARD:].data_ptr(), p.M, p.N, p.K, p.rpg, flags)
    rep = (C.c_int32 * (4 * n))()
    nat.check(lib.m3pc_gemm_bf16_problems(arr, n, rep, None), c.name)
    torch.cuda.synchronize()
    report = [tuple(rep[4 * i:4 * i + 4]) for i in range(n)]
    worst = 0.0
    for i, (p, (A, W, bias, tab, resid, flags, before), Cb) in enumerate(zip(c.probs, ops, outs)):
        where = f"{c.name} problem {i} {p} {'exact' if exact else 'random'}"
        assert report[i][:3] == tuple(c.expect[i]), (where, report[i])
        assert guards_intact(Cb), where
        assert all(torch.equal(b0, bits(t)) for b0, t in zip(before, [t for t in (A, W, bias, tab) if t is not None])), \
            f"{where}: a read-only operand changed"
        out = Cb[GUARD:GUARD + p.M]
        assert torch.isfinite(out.float()).all(), where
        ref, S, pre = reference(p, A, W, bias, tab, resid, flags)
        if exact:
            assert ref.abs().max() <= 256
            assert torch.equal(out.double(), ref), f"{where}: {int((out.double() != ref).sum())} elements differ"
            continue
        bar = A_BAR * S
        if flags & GELU:
            bar = bar + GELU_BAR[report[i][0]](pre)
        if not out_f32(flags):
            bar = bar + 2.0 ** -8 * ref.abs()
        err = (out.double() - ref).abs()
        ratio = float((err / bar).max())
        worst = max(worst, ratio)
        assert ratio <= 1.0, f"{where}: error {ratio:.3g} x the bar"
    return report, worst


def check_case(lib, nat, c):
    report, worst = run_gemm(lib, nat, c, False, 1)
    run_gemm(lib, nat, c, True, 2)
    if c.launches is not None:
        assert 1 + max(r[3] for r in report) == c.launches, report
    print(f"\n{c.name}: report {report}, largest error / bar {worst:.3f}")


# ---- every reachable instance ---------------------------------------------------------------------------------------------------
INSTANCE_CASES = [gcase(f"skinny_M{M}_K{K}", [(M, 256, K)], (SKINNY, 0, 0)) for M in (1, 17, 32) for K in (64, 512, 2048, 4096)
                  if M * K * 2 <= 160 * 1024]
INSTANCE_CASES += [
    gcase("single_M32_K4096", [(32, 256, 4096)], (SINGLE, 128, 2)),  # 32 rows whose A panel does not fit the skinny kernel
    gcase("single_M33", [(33, 512, 512)], (SINGLE, 128, 2)),
    gcase("single_M64", [(64, 1536, 512)], (SINGLE, 128, 2)),
    gcase("single_M128", [(128, 512, 2048)], (SINGLE, 128, 2)),
    gcase("single_M129_N384", [(129, 384, 512)], (SINGLE, 128, 2)),  # 2 m-tiles: one cluster, the second CTA's tile is 1 row
    gcase("single_M257_N640", [(257, 640, 512)], (SINGLE, 128, 2)),  # 3 m-tiles: the second cluster's second CTA is beyond M
    gcase("single_M257_N384_K2048", [(257, 384, 2048)], (SINGLE, 128, 2)),
    gcase("single_128x4x1", [(513, 3200, 64)], (SINGLE, 128, 1)),
    gcase("pair_M129", [(129, 256, 256)], (PAIR, 0, 1)),
    gcase("pair_M257", [(257, 512, 512)], (PAIR, 0, 1)),
    gcase("pair_M4099", [(4099, 1024, 512)], (PAIR, 0, 1)),
    gcase("pair_strided", [(32768, 512, 2048)], (PAIR, 1, 1)),
]

# ---- every epilogue on each kernel ------------------------------------------------------------------------------------------------
EPILOGUES = [("none_nobias", 0, 1, False), ("gelu", GELU, 1, True), ("relu", RELU, 1, True), ("gelu_relu", GELU | RELU, 1, True),
             ("res", RES, 1, True), ("res_gelu", RES | GELU, 1, True), ("tab1", TAB, 1, True), ("tabB", TAB, None, True),
             ("tab7", TAB, 7, True), ("f32", F32, 1, True), ("tab_f32", TAB | F32, None, True), ("gelu_f32", GELU | F32, 1, True)]
KERNELS = [("skinny", (17, 512, 512), (SKINNY, 0, 0)), ("single", (257, 640, 512), (SINGLE, 128, 2)),
           ("single_cl1", (513, 3200, 64), (SINGLE, 128, 1)), ("pair", (4099, 512, 512), (PAIR, 0, 1))]
EPILOGUE_CASES = [gcase(f"{kn}_{en}", [Prob(M, N, K, fl, rpg if rpg else max(1, M // 4), b)], ex)
                  for kn, (M, N, K), ex in KERNELS for en, fl, rpg, b in EPILOGUES]

# ---- the engine's grouped lists, and the other ways a group is issued -------------------------------------------------------------
B = 1024
GROUP_CASES = [
    # decoder_embed: one run of kept tokens per problem, X row block = token, table = the run's dec_cvec rows (one per token)
    gcase("decoder_embed_runs", [Prob(3 * B, 512, 512, TAB | F32, B, False), Prob(2 * B, 512, 512, TAB | F32, B, False),
                                 Prob(3 * B, 512, 512, TAB | F32, B, False), Prob(1 * B, 512, 512, TAB | F32, B, False)],
          (PAIR, 0, 4), launches=1),
    gcase("kv_q", [(13 * B, 1024, 512), (12 * B, 512, 512)], (PAIR, 0, 2), launches=1),
    gcase("gelu_heads", [(4 * B, 512, 512, GELU), (3 * B, 512, 512, GELU)], (PAIR, 0, 2), launches=1),
    gcase("twin_critics", [(8 * B, 256, 256, RELU | F32), (8 * B, 256, 256, RELU | F32)], (PAIR, 0, 2), launches=1),
    gcase("group_with_skinny_rows", [(4096, 512, 512), (17, 512, 512, RELU), (32, 256, 64, TAB, 5)], (PAIR, 0, 3), launches=1),
    gcase("group_falls_back_n384", [(4096, 512, 512), (300, 384, 512), (17, 256, 512)],
          [(PAIR, 0, 1), (SINGLE, 128, 2), (SKINNY, 0, 0)], launches=3),
    gcase("five_problems", [(640, 1024, 512), (129, 256, 256), (1000, 2048, 512, GELU), (333, 512, 2048, RES), (2000, 256, 128, RELU)],
          [(PAIR, 0, 4)] * 4 + [(PAIR, 0, 1)], launches=2),
    gcase("nine_problems", [(300 + 97 * i, 256 * (1 + i % 3), 64 * (1 + i % 4), [0, GELU, RELU, F32][i % 4]) for i in range(9)],
          [(PAIR, 0, 4)] * 8 + [(PAIR, 0, 1)], launches=3),
]


@pytest.mark.parametrize("c", INSTANCE_CASES + EPILOGUE_CASES + GROUP_CASES, ids=lambda c: c.id)
def test_gemm_bf16_problems(lib, nat, c):
    check_case(lib, nat, c)


def test_gemm_gelu_forms_meet_their_documented_bounds(lib, nat):
    """GELU|OUT_F32 on a ramp of pre-activations over [-8, 8] (A = identity rows, bias = the ramp): each kernel's GELU form
    against the erf GELU in float64, within the bound its comment states."""
    N, K = 512, 64
    for name, M, kind in (("skinny", 17, SKINNY), ("single", 257, SINGLE), ("pair", 4099, PAIR)):
        x = torch.linspace(-8, 8, M * N, device=DEV, dtype=torch.float64).float().view(M, N)
        A = torch.zeros(M, K, device=DEV, dtype=torch.bfloat16)
        W = torch.zeros(N if name != "single" else 640, K, device=DEV, dtype=torch.bfloat16)
        Nn = W.shape[0]
        table = torch.zeros(M, Nn, device=DEV)
        table[:, :N] = x
        Cb = guarded(M, Nn, torch.float32, float("nan"))
        p = nat.GemmProblem(A.data_ptr(), W.data_ptr(), None, table.data_ptr(), Cb[GUARD:].data_ptr(), M, Nn, K, 1, GELU | TAB | F32)
        rep = (C.c_int32 * 4)()
        nat.check(lib.m3pc_gemm_bf16_problems(C.byref(p), 1, rep, None))
        torch.cuda.synchronize()
        assert rep[0] == kind, (name, list(rep))
        out = Cb[GUARD:GUARD + M, :N].double()
        ref = torch.nn.functional.gelu(x.double())
        ratio = float(((out - ref).abs() / GELU_BAR[kind](x.double())).max())
        print(f"\n{name} GELU: largest error {float((out - ref).abs().max()):.3g}, {ratio:.3f} x its bound")
        assert ratio <= 1.0 and guards_intact(Cb)


def test_same_rows_give_the_same_bits_on_every_tensor_core_path(lib, nat):
    """Without GELU, a row's bits do not depend on the kernel (single-CTA, CTA pair contiguous or strided) nor on the group it runs
    in: the engine's kernel choices rely on it (commit ee132c8: every residual GEMM + LayerNorm through one call)."""
    g = torch.Generator(device=DEV).manual_seed(5)
    K, N = 2048, 512
    A = torch.randn(32768, K, device=DEV, generator=g).bfloat16()
    W = (torch.randn(N, K, device=DEV, generator=g) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=DEV, generator=g)
    A2 = torch.randn(3000, K, device=DEV, generator=g).bfloat16()
    runs = {"single": [128], "contiguous": [4099], "strided": [32768], "grouped": [4099, 3000]}
    expect = {"single": (SINGLE, 128, 2), "contiguous": (PAIR, 0, 1), "strided": (PAIR, 1, 1), "grouped": (PAIR, 0, 2)}
    outs = {}
    for name, Ms in runs.items():
        Cs = [torch.full((M, N), float("nan"), device=DEV, dtype=torch.bfloat16) for M in Ms]
        arr = (nat.GemmProblem * len(Ms))(*[nat.GemmProblem((A if i == 0 else A2).data_ptr(), W.data_ptr(), bias.data_ptr(), None,
                                                            Cm.data_ptr(), M, N, K, 1, RELU) for i, (M, Cm) in enumerate(zip(Ms, Cs))])
        rep = (C.c_int32 * (4 * len(Ms)))()
        nat.check(lib.m3pc_gemm_bf16_problems(arr, len(Ms), rep, None), name)
        torch.cuda.synchronize()
        assert tuple(rep[:3]) == expect[name], (name, list(rep))
        outs[name] = Cs[0]
    for name in ("contiguous", "strided", "grouped"):
        assert torch.equal(bits(outs[name][:128]), bits(outs["single"])), name
    assert torch.equal(bits(outs["strided"][:4099]), bits(outs["contiguous"]))
    assert torch.equal(bits(outs["grouped"]), bits(outs["contiguous"]))


# ---- the fused residual GEMM + LayerNorm ---------------------------------------------------------------------------------------------
LN_A_BAR = 2e-6  # X: fp32 accumulation + bias + residual, per element against the float64 sum's S (B200: largest 0.063 x 8e-6)
LN_Y_BAR = 2e-4  # Y: |Y - LN64(X)| <= 2^-8 |ref| + LN_Y_BAR * max(1, max |ref|), the bar m3pc_layernorm meets on the same X


@pytest.fixture(scope="module")
def unit_rows_option():
    """m3pc_set_option("gemm_ln_unit_rows") needs a handle; the option is process-wide."""
    from m3pc_b200 import synthetic as syn
    from m3pc_b200.engine import engine_from_synthetic
    shape = syn.shipped_shape("hopper")
    eng = engine_from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), max_batch=8)
    yield lambda rows: eng.set_option("gemm_ln_unit_rows", rows)
    eng.set_option("gemm_ln_unit_rows", 0)


@dataclass
class LnSpec:
    M: int
    res: str = "x"  # "x" in place, "r" other fp32 rows, "t" table
    rpg: int = 1


def ln_inputs(specs, K, g, offset=None):
    """Per job: A, W, X0 (the in-place residual or garbage when the residual comes from elsewhere), R, table.  offset: rows with
    mean / std in `offset` and std from 1e-2 to 1e2 (A rows scaled with the row's std), plus one constant row."""
    W = (torch.randn(512, K, device=DEV, generator=g) / K ** 0.5).bfloat16()
    jobs = []
    for s in specs:
        A = torch.randn(s.M, K, device=DEV, generator=g)
        resid = 2.0 * torch.randn(s.M, 512, device=DEV, generator=g) + 0.5
        if offset is not None:
            r = torch.arange(s.M, device=DEV)
            std = 10.0 ** (-2 + 4 * ((r * 7919) % s.M).double() / max(1, s.M - 1))
            off = torch.tensor(offset, device=DEV, dtype=torch.float64)[r % len(offset)]
            A = A * std[:, None].float()
            resid = (std[:, None] * (torch.randn(s.M, 512, device=DEV, generator=g, dtype=torch.float64) + off[:, None])).float()
            A[-1] = 0
            resid[-1] = 1000.0
        n_grp = -(-s.M // s.rpg)
        R = resid.clone() if s.res == "r" else None
        tab = None
        if s.res == "t":
            tab = torch.full((n_grp + 8, 512), float("nan"), device=DEV)
            tab[:n_grp] = torch.randn(n_grp, 512, device=DEV, generator=g) * 2 + 0.5
        X0 = resid if s.res == "x" else torch.full((s.M, 512), float("nan"), device=DEV)
        jobs.append((A.bfloat16(), X0, R, tab))
    return W, jobs


def run_ln(lib, nat, specs, K, W, jobs, bias, gamma, beta):
    n = len(specs)
    arr = (nat.LnJob * n)()
    bufs = []
    for i, (s, (A, X0, R, tab)) in enumerate(zip(specs, jobs)):
        Xb = guarded(s.M, 512, torch.float32, X0)
        Yb = guarded(s.M, 512, torch.bfloat16, float("nan"))
        bufs.append((Xb, Yb))
        arr[i] = nat.LnJob(A.data_ptr(), W.data_ptr(), Xb[GUARD:].data_ptr(), Yb[GUARD:].data_ptr(), tab.data_ptr() if tab is not None else None,
                           R.data_ptr() if R is not None else None, s.rpg, s.M)
    ro = [bits(t) for t in [W, bias, gamma, beta] + [t for (A, X0, R, tab) in jobs for t in (A, R, tab) if t is not None] if t is not None]
    rep = (C.c_int32 * 2)()
    nat.check(lib.m3pc_gemm_ln_bf16_grouped(arr, n, bias.data_ptr() if bias is not None else None, gamma.data_ptr(), beta.data_ptr(), K,
                                            rep, None), "m3pc_gemm_ln_bf16_grouped")
    torch.cuda.synchronize()
    ro_after = [bits(t) for t in [W, bias, gamma, beta] + [t for (A, X0, R, tab) in jobs for t in (A, R, tab) if t is not None] if t is not None]
    assert all(torch.equal(a, b) for a, b in zip(ro, ro_after)), "a read-only operand changed"
    outs = []
    for s, (Xb, Yb) in zip(specs, bufs):
        assert guards_intact(Xb) and guards_intact(Yb), s
        outs.append((Xb[GUARD:GUARD + s.M], Yb[GUARD:GUARD + s.M]))
    return tuple(rep), outs


def ln64(X, gamma, beta):
    return torch.nn.functional.layer_norm(X.double(), (512,), gamma.double(), beta.double(), 1e-5)


def y_excess(Y, ref):
    """max over elements of (|Y - ref| - 2^-8 |ref|), over max(1, max |ref|)."""
    return float(((Y.double() - ref).abs() - 2.0 ** -8 * ref.abs()).max()) / max(1.0, float(ref.abs().max()))


def check_ln(specs, W, jobs, outs, bias, gamma, beta):
    worst = 0.0
    for s, (A, X0, R, tab), (X, Y) in zip(specs, jobs, outs):
        a, w = A.double(), W.double()
        ref, S = a @ w.T, a.abs() @ w.abs().T
        if bias is not None:
            ref, S = ref + bias.double(), S + bias.double().abs()
        res = {"x": X0, "r": R, "t": None if tab is None else tab[:-8].repeat_interleave(s.rpg, dim=0)[:s.M]}[s.res].double()
        ref, S = ref + res, S + res.abs()
        assert torch.isfinite(X).all() and torch.isfinite(Y.float()).all(), s
        ratio = float(((X.double() - ref).abs() / (LN_A_BAR * S)).max())
        worst = max(worst, ratio)
        assert ratio <= 1.0, (s, ratio)
        assert y_excess(Y, ln64(X, gamma, beta)) <= LN_Y_BAR, s
    return worst


def ln_params(g, with_bias=True):
    bias = torch.randn(512, device=DEV, generator=g) if with_bias else None
    return bias, 1 + 0.2 * torch.randn(512, device=DEV, generator=g), 0.2 * torch.randn(512, device=DEV, generator=g)


LN_CASES = [  # (name, K, jobs, bias)
    *[(f"M{M}_K{K}", K, [LnSpec(M)], True) for M in (1, 31, 63, 64, 65, 127, 128, 129, 255, 256, 257, 4000, 26624) for K in (64, 512, 2048)
      if M <= 4000 or K != 64],
    ("R_source", 512, [LnSpec(4000, "r")], True),
    ("table_rpg1", 512, [LnSpec(300, "t", 1)], True),
    ("table_rpg7", 2048, [LnSpec(1000, "t", 7)], True),
    ("table_rpg1024", 512, [LnSpec(4000, "t", 1024)], True),
    ("null_bias", 512, [LnSpec(777)], False),
    ("two_jobs", 512, [LnSpec(300), LnSpec(129, "r")], True),
    ("three_jobs", 2048, [LnSpec(65, "t", 7), LnSpec(4000), LnSpec(1, "r")], True),
    # block_shared_history: the shared tokens' rows from the history table (row / grp), the per-candidate rows in place
    ("shared_history_outproj", 512, [LnSpec(9 * 8, "t", 8), LnSpec(4 * 1024)], True),
    # decode_restricted / restricted_last_layer: runs of needed rows into a compact block, residual from the mask-token table
    # (one row per token: rows_per_group = B) or from the kept tokens' residual-stream rows
    ("restricted_decoder_runs", 512, [LnSpec(4 * 256, "t", 256), LnSpec(3 * 256, "r"), LnSpec(1 * 256, "t", 256), LnSpec(2 * 256, "r")], False),
]


@pytest.mark.parametrize("name,K,specs,with_bias", LN_CASES, ids=[c[0] for c in LN_CASES])
def test_gemm_ln_bf16_grouped(lib, nat, unit_rows_option, name, K, specs, with_bias):
    """X per element against float64, Y against a float64 LayerNorm of the kernel's own X; the same bits alone, in the group and with
    either unit size, and the unit size reported as chosen (automatic) or forced."""
    g = torch.Generator(device=DEV).manual_seed(K + sum(s.M for s in specs))
    bias, gamma, beta = ln_params(g, with_bias)
    W, jobs = ln_inputs(specs, K, g)
    results = {}
    for rows in (0, 128, 256):
        unit_rows_option(rows)
        rep, outs = run_ln(lib, nat, specs, K, W, jobs, bias, gamma, beta)
        if rows:
            assert rep[0] == rows, rep
        results[rows] = (rep, outs)
    unit_rows_option(0)
    worst = check_ln(specs, W, jobs, results[0][1], bias, gamma, beta)
    for rows in (128, 256):
        for (X0, Y0), (X1, Y1) in zip(results[0][1], results[rows][1]):
            assert torch.equal(bits(X0), bits(X1)) and torch.equal(bits(Y0), bits(Y1)), f"unit rows {rows}"
    if len(specs) > 1:
        for i, s in enumerate(specs):  # alone
            rep, outs = run_ln(lib, nat, [s], K, W, [jobs[i]], bias, gamma, beta)
            assert torch.equal(bits(outs[0][0]), bits(results[0][1][i][0])) and torch.equal(bits(outs[0][1]), bits(results[0][1][i][1])), s
    print(f"\n{name}: automatic unit {results[0][0]}, X error / bar {worst:.3f}")


@pytest.mark.parametrize("K", [512, 2048])
def test_gemm_ln_rows_with_large_offsets(lib, nat, K):
    """Rows whose mean is 0 .. 1000 times their spread (std 1e-2 .. 1e2) and one constant row: the fused kernel's Y must meet the
    bar m3pc_layernorm meets on the same X.  A variance taken as E[x^2] - mean^2 in fp32 misses it from mean / std ~ 100 on."""
    g = torch.Generator(device=DEV).manual_seed(11 + K)
    _, gamma, beta = ln_params(g)
    specs = [LnSpec(4000)]
    W, jobs = ln_inputs(specs, K, g, offset=[0, 30, 100, 300, 1000])
    _, outs = run_ln(lib, nat, specs, K, W, jobs, None, gamma, beta)
    X, Y = outs[0]
    ref = ln64(X, gamma, beta)
    Ys = torch.empty(X.shape, device=DEV, dtype=torch.bfloat16)
    nat.check(lib.m3pc_layernorm(X.data_ptr(), gamma.data_ptr(), beta.data_ptr(), Ys.data_ptr(), X.shape[0], 512, 1, None))
    torch.cuda.synchronize()
    fused, alone = y_excess(Y, ref), y_excess(Ys, ref)
    print(f"\nK={K}: Y error beyond bf16 rounding / max(1, max|ref|): fused {fused:.3g}, m3pc_layernorm {alone:.3g}")
    assert alone <= LN_Y_BAR
    assert fused <= LN_Y_BAR
