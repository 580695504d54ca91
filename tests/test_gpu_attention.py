"""The gather-form attention kernels (attention.cu) through m3pc_attention_gather, against float64.

Every case is one description: for each query / key / value token, the source it is read from and a label naming its block of
rows there (Q, K and V of one token share a block, at different columns).  A source has one token kind and one of the engine's
layouts:

  qkv   per batch row, stride 3D, Q / K / V at column 0 / D / 2D   (the QKV activations)
  kv    per batch row, stride 2D, K / V at column 0 / D            (K / V of the restricted decoder layer)
  q     per batch row, stride D                                    (selected queries of the restricted decoder layer)
  c     batch-constant (bstride 0), stride 3D                      (the mask-token table const_qkv)
  g<n>  per group of n batch rows (bdiv n), stride 3D              (the history table of pass 2)

From that description the test builds both the header arrays of the call and the float64 reference (the same rows gathered with
torch indexing; for bf16 the reference uses the same bf16-rounded operands).  Every call reports which kernel instance ran and its
grid; every case names the instance it expects, and the cases reach all 23 instances.  Rows of a source that no token uses are
NaN, so a read outside the described rows shows up in the output.

Inputs: random, and for bf16 two probes that random inputs can miss at these bars --
  onehot  every (batch row, head, query) attends with weight > 1 - 1e-6 to one key, chosen per query, head and query row, at a
          peak score >= 100 (a missing max subtraction overflows); the key's code dimension and the values differ per row, group
          and head, so a wrong row, group, head or K / V pairing gives an O(1) error;
  pad     every real score <= -20 and values around 1: an unmasked zero pad key would dominate and pull the output to 0.
"""
import ctypes as C
import math
import zlib
from dataclasses import dataclass

import pytest
import torch

pytestmark = pytest.mark.gpu

HD = 128
ROW, CONST = 1, 0  # token kinds besides a group size n > 1: one row per batch row, one row for the whole batch
BAR = {False: 1e-5, True: 8e-3}  # fp32 / bf16: max |out - ref| <= BAR * max(1, max |ref|)
GUARD_ROWS = 64
DEV = "cuda"
SH_ROWS = 8  # batch rows per block of the shared-key kernel

LAYOUT = {"qkv": (3, {"q": 0, "k": 1, "v": 2}), "kv": (2, {"k": 0, "v": 1}), "q": (1, {"q": 0}), "c": (3, {"q": 0, "k": 1, "v": 2})}


def src_kind(name):
    return {"qkv": ROW, "kv": ROW, "q": ROW, "c": CONST}[name] if name in LAYOUT else int(name[1:])


def src_layout(name):
    return LAYOUT.get(name, LAYOUT["c"])


def block_rows(kind, B):
    return 1 if kind == CONST else -(-B // kind)


def src_rows(kind, b):  # row of a token's block that batch rows b read
    return torch.zeros_like(b) if kind == CONST else b // kind


def coarser_or_equal(key_kind, query_kind):
    """Within one row of the query's block the key's row does not change."""
    return key_kind == CONST or (query_kind != CONST and key_kind % query_kind == 0)


@dataclass
class Case:
    name: str
    B: int
    q: list  # [(source, label)]
    k: list
    v: list
    n_kv_batch: int
    expect: tuple  # (kind, a, b) of the bf16 launch: 1 = attention_mma_kernel<a, b>, 2 = attention_mma_shared_kernel<a, b>
    H: int = 4
    persistent: bool = None  # shared-key kernel: whether each CTA walks several 8-row blocks

    @property
    def id(self):
        return f"{self.name}-B{self.B}"


def case(name, B, q, k, v=None, n_kv_batch=0, expect=None, H=4, persistent=None):
    return Case(name, B, list(q), list(k), list(k if v is None else v), n_kv_batch, expect, H, persistent)


def seq(src, n, start=0):
    return [(src, start + i) for i in range(n)]


# ---- the engine's two forms ------------------------------------------------------------------------------------------------
def pass2_first_block(B, grp=1024):
    """block_shared_history: 9 history tokens per group of `grp` candidates (table g<grp>), 4 per-candidate tokens (qkv); queries
    in token order, keys with the per-candidate tokens first."""
    g = f"g{grp}"
    return case(f"pass2_first_block_g{grp}", B, seq(g, 9) + seq("qkv", 4, 9), seq("qkv", 4, 9) + seq(g, 9), n_kv_batch=4,
                expect=(2, 1, 1), persistent=B >= 8192)


def restricted_decoder(B, persistent=None):
    """restricted_last_layer at T = 8: 32 decoder tokens, 13 kept (K / V rows of kv), 19 masked (const_qkv rows); 12 needed
    queries, the masked ones from const_qkv, the kept ones from their q row block."""
    kept = [0, 1, 2, 3, 8, 9, 10, 16, 17, 18, 24, 25, 26]
    masked = [j for j in range(32) if j not in kept]
    need = [4, 5, 6, 7, 11, 12, 13, 14, 15, 19, 20, 1]
    q = [("c", j) if j in masked else ("q", qi) for qi, j in enumerate(need)]
    k = [("kv", j) for j in kept] + [("c", j) for j in masked]
    return case("restricted_decoder", B, q, k, n_kv_batch=13, expect=(2, 1, 2), persistent=persistent)


ENGINE_CASES = [pass2_first_block(1024), pass2_first_block(8 * 1024), restricted_decoder(64, False), restricted_decoder(65, False),
                restricted_decoder(8192, True)]


# ---- every shared-key instance, on the persistent path and off it -----------------------------------------------------------
def mixed_queries(n):  # per-row queries at strides 3D and D, batch-constant ones, one per group of 24 rows
    srcs = ["qkv", "c", "g24", "q"]
    return [(srcs[i % 4], i) for i in range(n)]


def batch_keys(n):  # per-batch keys: per-row at strides 3D and 2D, and one per group of 3 rows (K and V move together)
    srcs = ["qkv", "kv", "g3"]
    return [(srcs[i % 3], 100 + i) for i in range(n)]


def shared(name, n_q, n_b, n_c, shared_src, expect, B, H):
    return case(f"{name}_q{n_q}_b{n_b}_{shared_src}x{n_c}_h{H}", B, mixed_queries(n_q), batch_keys(n_b) + seq(shared_src, n_c, 200),
                n_kv_batch=n_b, expect=expect, H=H, persistent=B >= 8192)


SHARED_SHAPES = [  # (name, n_q, n_b, n_c, source of the shared keys, instance, n_head)
    ("shared11", 16, 16, 16, "c", (2, 1, 1), 4),
    ("shared12", 3, 1, 17, "g16", (2, 1, 2), 4),
    ("shared13", 7, 16, 40, "c", (2, 1, 3), 8),
    ("shared21", 1, 17, 8, "c", (2, 2, 1), 4),
    ("shared22", 12, 32, 32, "g8", (2, 2, 2), 4),  # bdiv 8: the kernel restages the shared tiles for every block
    ("shared23", 16, 20, 44, "g96", (2, 2, 3), 4),  # groups of 12 blocks straddle the CTAs' block ranges
]
SHARED_CASES = [shared(n, nq, nb, nc, src, ex, B, H) for (n, nq, nb, nc, src, ex, H) in SHARED_SHAPES
                for B in (72, 8195 if H == 8 else 8192)]


# ---- the per-row kernel: every (query tiles, key tiles), token counts from {1, 16, 17, 33, 48, 49, 64} ----------------------
TOKENS_OF_TILES = {1: (1, 16), 2: (17, 17), 3: (33, 48), 4: (49, 64)}


def per_row(ntq, ntk):
    i = 4 * (ntq - 1) + (ntk - 1)
    n_q, n_kv = TOKENS_OF_TILES[ntq][i % 2], TOKENS_OF_TILES[ntk][(i // 2) % 2]
    qs, ks = ["qkv", "q", "c", "g3"], ["qkv", "kv", "c", "g5"]
    q = [(qs[(j + i) % 4], j) for j in range(n_q)]
    k = [(ks[(j + i) % 4], 100 + j) for j in range(n_kv)]
    return case(f"per_row{ntq}{ntk}_q{n_q}_kv{n_kv}", (1, 63, 200)[i % 3], q, k, expect=(1, ntq, ntk))


PER_ROW_CASES = [per_row(a, b) for a in range(1, 5) for b in range(1, 5)]


# ---- key lists the shared-key kernel must not take --------------------------------------------------------------------------
def fallback_cases():
    dec = restricted_decoder(63)
    k9 = batch_keys(9) + seq("c", 9, 200)
    k_split, v_split = list(k9), list(k9)
    k_split[4], v_split[4] = ("kv", 300), ("qkv", 300)  # one per-row key: K at stride 2D, V at stride 3D
    return [
        case("fallback_below_64_rows", 63, dec.q, dec.k, n_kv_batch=13, expect=(1, 1, 2)),
        case("fallback_7_shared_keys", 8192, mixed_queries(5), batch_keys(9) + seq("c", 7, 200), n_kv_batch=9, expect=(1, 1, 1)),
        case("fallback_bdiv12", 8192, mixed_queries(5), batch_keys(9) + seq("g12", 9, 200), n_kv_batch=9, expect=(1, 1, 2)),
        case("fallback_17_queries", 8192, mixed_queries(17), k9, n_kv_batch=9, expect=(1, 2, 2)),
        case("fallback_no_shared_keys", 200, mixed_queries(16), batch_keys(64), n_kv_batch=64, expect=(1, 1, 4)),
        case("fallback_kv_strides_differ", 8192, mixed_queries(5), k_split, v_split, n_kv_batch=9, expect=(1, 1, 2)),
        # shared keys of mixed forms: the shared-key kernel restages its tiles only when the FIRST shared key's group changes
        case("fallback_mixed_const_group", 8192, mixed_queries(5), batch_keys(9) + seq("c", 4, 200) + seq("g8", 5, 210),
             n_kv_batch=9, expect=(1, 1, 2)),
        case("fallback_mixed_bdiv", 8192, mixed_queries(5), batch_keys(9) + seq("g1024", 4, 200) + seq("g8", 5, 210),
             n_kv_batch=9, expect=(1, 1, 2)),
    ]


FALLBACK_CASES = fallback_cases()
BF16_CASES = ENGINE_CASES + SHARED_CASES + PER_ROW_CASES + FALLBACK_CASES
FP32_CASES = ENGINE_CASES + [case("square64", 200, mixed_queries(64), seq("qkv", 64, 100)), case("single", 1, [("qkv", 0)], [("qkv", 0)])]


def test_cases_reach_every_instance():
    every = {(1, a, b) for a in range(1, 5) for b in range(1, 5)} | {(2, a, b) for a in (1, 2) for b in (1, 2, 3)}
    assert {c.expect for c in BF16_CASES} == every
    for inst in {(2, a, b) for a in (1, 2) for b in (1, 2, 3)}:  # each shared-key instance on and off the persistent path
        assert {c.persistent for c in BF16_CASES if c.expect == inst} == {True, False}, inst
    assert FP32_CASES


# ---- building the operands and the reference --------------------------------------------------------------------------------
class Operands:
    """The sources of a case: one NaN-filled matrix per source name, a block of rows per distinct label."""

    def __init__(self, cs, dtype):
        self.cs, self.D = cs, cs.H * HD
        self.block = {}
        for name, label in cs.q + cs.k + cs.v:
            blocks = self.block.setdefault(name, {})
            blocks.setdefault(label, len(blocks))
        self.src = {}
        for name, blocks in self.block.items():
            rows = len(blocks) * block_rows(src_kind(name), cs.B)
            self.src[name] = torch.full((rows, src_layout(name)[0] * self.D), float("nan"), device=DEV, dtype=dtype)

    def region(self, tok, role):
        """(rows of the token's block x D) view of the token's role (q / k / v) in its source."""
        name, label = tok
        kind, (_, cols) = src_kind(name), src_layout(name)
        n = block_rows(kind, self.cs.B)
        r0, c0 = self.block[name][label] * n, cols[role] * self.D
        return self.src[name][r0:r0 + n, c0:c0 + self.D]

    def header(self, tok, role):
        from m3pc_b200 import _native as nat
        name, _ = tok
        kind, reg = src_kind(name), self.region(tok, role)
        return nat.AttnTok(reg.data_ptr(), 0 if kind == CONST else reg.stride(0), kind if kind > ROW else 0)

    def gather(self, tok, role, b):  # (len(b), H, 128) float64 rows of batch rows b
        return self.region(tok, role)[src_rows(src_kind(tok[0]), b)].double().view(len(b), self.cs.H, HD)

    def tokens(self):  # every (token, role) once; K and V of one key may be one block
        for role, toks in (("q", self.cs.q), ("k", self.cs.k), ("v", self.cs.v)):
            for j, t in enumerate(toks):
                yield role, j, t

    def fill_random(self, g):
        for role, _, t in self.tokens():
            reg = self.region(t, role)
            reg.copy_(torch.randn(reg.shape, device=DEV, generator=g))

    def fill_onehot(self, g, a=32.0, c=40.0):
        """Key j at a row of its block is c * e_(2j + bit), bit random per row and head; query i aims at key t (random per
        query row and head) with a * e_(2t + bit of key t at that batch row) when key t's row is fixed within the query's row,
        else with a * (e_2t + e_2t+1).  Scores: a c / sqrt(128) = 113 for the target, 0 for every other key."""
        cs, H = self.cs, self.cs.H
        n_kv, b = len(cs.k), torch.arange(cs.B, device=DEV)
        bits = []
        for j, t in enumerate(cs.k):
            reg = self.region(t, "k").view(-1, H, HD)
            bit = torch.randint(0, 2, reg.shape[:2], device=DEV, generator=g)
            reg.zero_().scatter_(2, (2 * j + bit)[..., None], c)
            bits.append(bit[src_rows(src_kind(t[0]), b)])  # (B, H): bit of key j at every batch row
        bits = torch.stack(bits)  # (n_kv, B, H)
        for t in cs.v:
            reg = self.region(t, "v")
            reg.copy_(torch.randn(reg.shape, device=DEV, generator=g))
        for t in cs.q:
            qk = src_kind(t[0])
            reg = self.region(t, "q").view(-1, H, HD)
            sq = src_rows(qk, b)
            target = torch.randint(0, n_kv, reg.shape[:2], device=DEV, generator=g)[sq]  # (B, H)
            fine = torch.tensor([coarser_or_equal(src_kind(kt[0]), qk) for kt in cs.k], device=DEV)[target]
            bit = bits.gather(0, target[None])[0]
            vec = torch.zeros(cs.B, H, HD, device=DEV)
            vec.scatter_(2, torch.where(fine, 2 * target + bit, 2 * target)[..., None], a)
            vec.scatter_(2, torch.where(fine, 2 * target + bit, 2 * target + 1)[..., None], a)
            reg[sq] = vec.to(reg.dtype)  # rows shared by several batch rows receive one value

    def fill_pad(self, g):
        """q = 16 e_0 + noise, k = -(16 .. 24) e_0 + noise (noise in the other dimensions): every score <= -20; v ~ 1."""
        for role, _, t in self.tokens():
            reg = self.region(t, role).view(-1, self.cs.H, HD)
            x = torch.randn(reg.shape, device=DEV, generator=g)
            if role == "v":
                reg.copy_(1 + 0.25 * x)
                continue
            x *= 0.5
            x[..., 0] = 16.0 if role == "q" else -(16 + 8 * torch.rand(reg.shape[:2], device=DEV, generator=g))
            reg.copy_(x)

    def reference(self, chunk=2048):
        """fp64 attention of the gathered rows: (n_q * B, D) and, over all (batch row, head, query), the smallest and largest
        top score, the smallest gap between the two top scores and the smallest top softmax weight."""
        cs, out = self.cs, []
        top_lo, top_hi, gap, wmin = math.inf, -math.inf, math.inf, 1.0
        for b0 in range(0, cs.B, chunk):
            b = torch.arange(b0, min(cs.B, b0 + chunk), device=DEV)
            q = torch.stack([self.gather(t, "q", b) for t in cs.q])
            k = torch.stack([self.gather(t, "k", b) for t in cs.k])
            v = torch.stack([self.gather(t, "v", b) for t in cs.v])
            s = torch.einsum("ibhd,jbhd->bhij", q, k) / math.sqrt(HD)
            p = torch.softmax(s, -1)
            out.append(torch.einsum("bhij,jbhd->ibhd", p, v))
            top = s.topk(min(2, len(cs.k)), -1).values
            top_lo, top_hi = min(top_lo, float(top[..., 0].min())), max(top_hi, float(top[..., 0].max()))
            if len(cs.k) > 1:
                gap = min(gap, float((top[..., 0] - top[..., 1]).min()))
            wmin = min(wmin, float(p.max(-1).values.min()))
        ref = torch.cat(out, 1).reshape(len(cs.q) * cs.B, self.D)
        return ref, dict(top_lo=top_lo, top_hi=top_hi, gap=gap, wmin=wmin)


def launch(nat, ops, dst, bf16, **override):
    """m3pc_attention_gather of the case into dst, with any argument replaced by `override`; returns {kind, a, b, grid_x}."""
    cs = ops.cs
    arr = lambda role, toks: (nat.AttnTok * len(toks))(*[ops.header(t, role) for t in toks])
    launched = (C.c_int32 * 4)(-1, -1, -1, -1)
    args = dict(q=arr("q", cs.q), n_q=len(cs.q), k=arr("k", cs.k), v=arr("v", cs.v), n_kv=len(cs.k),
                n_kv_batch=cs.n_kv_batch, B=cs.B, H=cs.H, out=dst.data_ptr())
    args.update(override)
    nat.check(nat.lib().m3pc_attention_gather(args["q"], args["n_q"], args["k"], args["v"], args["n_kv"], args["n_kv_batch"], args["B"],
                                              args["H"], args["out"], int(bf16), launched, None), "m3pc_attention_gather")
    return tuple(launched)


def run_case(nat, cs, bf16, inputs):
    dtype = torch.bfloat16 if bf16 else torch.float32
    g = torch.Generator(device=DEV).manual_seed(zlib.crc32(f"{cs.id} {inputs}".encode()))
    ops = Operands(cs, dtype)
    getattr(ops, f"fill_{inputs}")(g)
    rows = len(cs.q) * cs.B
    out = torch.full((rows + GUARD_ROWS, ops.D), float("nan"), device=DEV, dtype=dtype)
    out[rows:] = torch.randn(GUARD_ROWS, ops.D, device=DEV, generator=g).to(dtype)
    guard = out[rows:].clone()
    kind, a, b, grid_x = launch(nat, ops, out, bf16)
    torch.cuda.synchronize()
    ref, st = ops.reference()
    if inputs == "onehot":  # the probe is what it claims to be
        assert st["top_lo"] >= 100 and st["gap"] >= 14 and st["wmin"] > 1 - 1e-6, st
    if inputs == "pad":
        assert st["top_hi"] <= -20, st
    assert torch.equal(out[rows:].view(torch.int16 if bf16 else torch.int32), guard.view(torch.int16 if bf16 else torch.int32)), \
        "a write past the output"
    res = out[:rows]
    assert bool(torch.isfinite(res).all()), f"{int((~torch.isfinite(res)).any(1).sum())} output rows not finite"
    err = float((res.double() - ref).abs().max()) / max(1.0, float(ref.abs().max()))
    print(f"attention_gather kernel={kind}<{a},{b}> grid={grid_x} {cs.id} {'bf16' if bf16 else 'fp32'} {inputs}: "
          f"err {err:.2e} = {err / BAR[bf16]:.3f} of the bar")
    assert err <= BAR[bf16], (err, cs.id)
    assert (kind, a, b) == (cs.expect if bf16 else (0, 0, 0)), (kind, a, b)
    if kind == 2:
        nblk = -(-cs.B // SH_ROWS)
        assert (grid_x < nblk) if cs.persistent else (grid_x == nblk), (grid_x, nblk)
    elif kind == 0:
        assert grid_x == cs.B * cs.H


@pytest.fixture(scope="module")
def nat():
    from m3pc_b200 import _native
    _native.lib()
    return _native


@pytest.mark.parametrize("inputs", ["random", "onehot", "pad"])
@pytest.mark.parametrize("cs", BF16_CASES, ids=lambda c: c.id)
def test_attention_gather_bf16(nat, cs, inputs):
    run_case(nat, cs, True, inputs)


@pytest.mark.parametrize("cs", FP32_CASES, ids=lambda c: c.id)
def test_attention_gather_fp32(nat, cs):
    run_case(nat, cs, False, "random")


@pytest.mark.parametrize("bf16", [True, False])
def test_attention_gather_rejects_bad_arguments(nat, bf16):
    """Every bad argument fails with M3PC_ERR_INVALID before anything is launched: the output stays untouched."""
    cs = restricted_decoder(64)
    dtype = torch.bfloat16 if bf16 else torch.float32
    ops = Operands(cs, dtype)
    ops.fill_random(torch.Generator(device=DEV).manual_seed(0))
    out = torch.full((len(cs.q) * cs.B + 8, ops.D), float("nan"), device=DEV, dtype=dtype)
    es = out.element_size()
    good = lambda role, toks: [ops.header(t, role) for t in toks]
    arr = lambda hs: (nat.AttnTok * len(hs))(*hs)

    def bad_token(**field):
        hs = good("k", cs.k)
        for f, val in field.items():
            setattr(hs[3], f, val)
        return arr(hs)

    k0 = good("k", cs.k)[0]
    bad = [
        dict(q=None), dict(k=None), dict(v=None), dict(out=None), dict(k=bad_token(ptr=None)),
        dict(n_q=0), dict(n_q=65), dict(n_kv=0), dict(n_kv=65),
        dict(n_kv_batch=-1), dict(n_kv_batch=len(cs.k) + 1),
        dict(B=0), dict(H=0),
        dict(out=out.data_ptr() + es),  # output not 16-byte aligned
        dict(k=bad_token(ptr=k0.ptr + es)),  # token not 16-byte aligned
        dict(k=bad_token(bstride=k0.bstride + 4 if bf16 else k0.bstride + 2)),  # rows not 16-byte aligned
        dict(k=bad_token(bstride=-k0.bstride)), dict(k=bad_token(bdiv=-8)),
    ]
    for override in bad:
        with pytest.raises(ValueError):
            launch(nat, ops, out, bf16, **override)
    torch.cuda.synchronize()
    assert bool(torch.isnan(out.float()).all()), "a rejected call launched"
    assert launch(nat, ops, out, bf16)[0] == (2 if bf16 else 0)  # the same arguments without the fault run
