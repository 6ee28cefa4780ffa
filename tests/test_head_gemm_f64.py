"""The tcgen05 TF32 mask head -- the TMA forward head (head_fused.cu), the register-staged forward head (head_tc.cu) and the
split-K weight gradient (head_bwd_tc.cu: TMA and transposing kernels, no loss / SISDR / WSD folded in, split reduction and
per-utterance pack) -- against a float64 GEMM of the operands the kernels feed the tensor cores, element by element, on every
branch of their launch plans.

Reference.  The operand preparation is restated in float32 (CMVN scale / shift as each kernel computes them, x_hat = x * sc + sh
or (x - mean) * sc, dZ = g * act'(o) times the row-live mask), rounded to TF32 with ``ops.round_tf32`` (cvt.rna), and multiplied
in float64.  Column D_in of x_hat is the ones column, so grad_b is column D_in of the reference.  The folded losses take g from
float64 autograd of the reference loss, rounded to float32.  The restated float32 operand need not equal the kernel's bit for
bit: __fdividef, rsqrtf and a different order of the loss arithmetic move it by a few float32 ulps of its terms.  Where that
moves it across a TF32 rounding midpoint, the kernel's TF32 operand is the neighbour of ours -- one TF32 ulp, 2^-10 of that
operand at most.  Instead of chasing bit-identical operands, every restated operand carries a bound eps on that difference,
and the tolerance adds, per element, the largest product change those flips can cause: sum_r span(a_r) (|b_r| + span(b_r)) +
|a_r| span(b_r), with span(v) = rn(v + eps) - rn(v - eps) (zero for almost every operand).

Tolerance.  |got - ref| <= RTOL * (blocks + 2) * sum_r |a_r b_r| + (flip allowance), per element of grad_W / grad_b and per
output of the forward heads.  `blocks` is the number of 32-wide blocks the kernel accumulates into one fp32 accumulator (rows of
the longest split in the weight gradient, ceil(D_in / 32) in the forward heads); the 2 covers the split reduction or the
per-utterance pack, and the epilogue.  fp32 accumulation error grows with that depth, so the bound does too: it is 1.2e-6 sum|ab|
for one block and at most 34 * RTOL = 1.4e-5 sum|ab| (the one-split-per-utterance case, 1024-row splits), 7.6e-6 for D_in 544.
The forward heads add |b_n| to the sum; Sigmoid scales the bound by its slope, at most 1/4, plus the 2^-20 of its own
approximate exponential and reciprocal; ReLU units inside the bound are skipped.  The leftover output rows of the weight gradient
(D_out % 128 in 1..4) and the "+1" output column of the forward head are fp32 dot products, not tensor-core products: there the
reference takes dZ (and, in the transposing kernel, x_hat) unrounded, and the allowance covers eps itself.  DESIGN section 2's
bound is also asserted against the unrounded operands: |got - ref64| <= 2^-10 sum|ab| + (the tolerance above) + (the eps terms).

Inputs.  Every utterance and feature has its own statistics (means in [-20, 5], scales in [0.3, 4]), so a row that takes its
neighbour's CMVN constants moves x_hat by O(10).  Burst rows (the first and last row of every utterance and of every split,
every row of a 32-row block that straddles an utterance boundary, and for the folded losses the last valid and first padded
frame of every utterance) carry 100 times the gradient.  Padding columns hold NaN; the forward outputs have sentinel guard rows
past row R.  ``record_margin`` asserts for each case that removing any one burst row, moving an utterance's boundary row to the
neighbour's statistics, one valid frame more or fewer (folded losses) and one row of the next utterance (per-utterance
gradients) each move the reference by at least SENSITIVITY tolerances on some element (rank-1 differences).

Measured on one NVIDIA B200 (1000 W power limit), largest (|got - ref| - flip allowance) / ((blocks + 2) sum|ab|) over the cases
of this file (``pytest -s`` prints each as an ERROR line, each margin as a MARGIN line):
  weight gradient, TMA kernel            1.35e-7   leftover row 8.5e-8
  weight gradient, transposing kernel    1.34e-7   leftover rows 1.1e-8
  per-utterance, TMA kernel              1.44e-7   leftover row 8.4e-8
  per-utterance, transposing kernel      1.11e-7   leftover rows 1.8e-8
  folded SISDR, row splits               1.3e-8    folded WSD, row splits 5.6e-8    folded SISDR, per utterance 1.05e-7
  (the folded kernels' leftover row stays inside its eps allowance: below zero)
  forward TMA head                       3.8e-8    "+1" SIMT column 2.9e-9
  forward register-staged head           2.5e-8
  Sigmoid outputs of both forward heads stay inside SIG_ATOL.
RTOL = 4e-7 is 2.8 times the largest, 1.44e-7 (one split of 1001 frames per utterance).  The smallest sensitivity margin is 23.5
tolerances (removing one burst row of the folded SISDR case with 600 utterances); the smallest boundary-row margin is 636.
"""
import math

import pytest
import torch

gpu = pytest.mark.gpu

RTOL = 4e-7                # |got - ref| / sum|ab| per accumulation step (2.8 times the largest measured, see above)
DESIGN_REL = 2.0 ** -10    # DESIGN section 2: each TF32 product carries a relative error <= 2^-10
SIG_ATOL = 2.0 ** -20      # the fused heads' sigmoid: ex2.approx / rcp.approx (__expf / __fdividef in head_tc.cu)
SENSITIVITY = 10.0
SMS_B200 = 148
BM, BK, MAX_UTT, MAX_SIMT, MAX_BROWS = 128, 32, 8, 4, 272
FWD_MAX_COLS, FWD_MAX_WROWS, FWD_RING = 544, 272, 4 * 51200


# ------------------------------------------------------------------------------------------------ launch-plan mirrors
def bwd_plan(B, F, Din, Dout, sms, per_utt=False):
    """plan() of head_bwd_tc.cu: None where the library refuses the shape."""
    R = B * F
    if R <= 0 or F < BK or Din <= 0 or Dout <= 0 or Din + 1 > MAX_BROWS:
        return None
    rem = Dout % BM
    simt = rem if (Dout > BM and 0 < rem <= MAX_SIMT) else 0
    m_tiles = (Dout - simt + BM - 1) // BM
    p = dict(simt_rows=simt, m_tiles=m_tiles, m_rows=m_tiles * BM + simt, b_rows=(Din + 1 + 15) // 16 * 16)
    p["n_tail"] = p["b_rows"] - min(p["b_rows"], 256)
    if per_utt:
        sub = min(max(sms // (B * m_tiles), 1), 4)
        rows = ((F + sub - 1) // sub + BK - 1) // BK * BK
        sub = (F + rows - 1) // rows
        p.update(sub=sub, rows=rows, splits=B * sub, clamped=False,
                 bounds=[(u * F + s * rows, min(u * F + (s + 1) * rows, (u + 1) * F)) for u in range(B) for s in range(sub)])
        return p
    splits = max(sms // m_tiles, 1)
    rows = ((R + splits - 1) // splits + BK - 1) // BK * BK
    max_rows = (MAX_UTT - 2) * F // BK * BK
    clamped = rows > max_rows
    rows = min(rows, max_rows)
    n = (R + rows - 1) // rows
    if n > 65535 or (rows + F - 1) // F + 1 > MAX_UTT:
        return None
    p.update(sub=0, rows=rows, splits=n, clamped=clamped, bounds=[(s * rows, min((s + 1) * rows, R)) for s in range(n)])
    return p


def fwd_plan(B, F, Din, Dout, ld_out, sms, out_aligned=True):
    """Launch shape of se_linear_head_fused (None where se_linear_head_fused_supported refuses the shape)."""
    if B <= 0 or F < 8 or Din > FWD_MAX_COLS or Dout > FWD_MAX_COLS or ld_out < Dout:
        return None
    dout4 = (Dout + 3) // 4 * 4
    if Dout <= FWD_MAX_WROWS and (ld_out if ld_out == dout4 else dout4 + 4) * 4 * BM > FWD_RING:
        return None
    R = B * F
    w_rows = (Dout + 15) // 16 * 16
    tiles128 = (R + BM - 1) // BM
    plus_one = Dout > 256 and (Dout - 1) % 256 == 0
    single = (w_rows + FWD_MAX_WROWS - 1) // FWD_MAX_WROWS
    dual = (w_rows <= 256 or plus_one) and tiles128 * single > sms
    store4 = ld_out % 4 == 0 and out_aligned
    if dual:
        n_split = (Dout - 1) // 256 if plus_one else 1
        slots, direct = 2 * sms, (2 if store4 else 1)
    else:
        n_split, slots = single, sms
        direct = (2 if store4 else 1) if n_split > 1 else 0
    waves = (tiles128 * n_split + slots - 1) // slots
    want = max(waves * slots // n_split, 1)
    rows = min(((R + want - 1) // want + 7) // 8 * 8, BM)
    if rows > F:
        rows = F // 8 * 8
    bulk = 1 if (not direct and ld_out == dout4 and out_aligned) else 0
    return dict(dual=dual, plus_one=dual and plus_one, n_split=n_split, direct_out=direct, bulk_out=bulk, tile_rows=rows,
                tiles=(R + rows - 1) // rows, sld=ld_out if bulk else dout4 + 4)


# ------------------------------------------------------------------------------------------------ cases
# backward: (B, F, D_in, D_out, act, cmvn, route); route "tma" = se_linear_head_bwd_fused on padded rows with stat_sums,
# "tc" = se_linear_head_bwd_tc on dense rows with mean / std, "tc_off" = the same on padded rows whose base is one float off
BWD = [
    (600, 40, 257, 257, "Sigmoid", True, "tma"),     # clamp: 108 splits x 2 tiles, splits % 4 = 0
    (1024, 32, 257, 257, "Identity", True, "tma"),   # clamp: 171 x 2, F = 32, splits % 4 = 3
    (900, 40, 129, 129, "ReLU", True, "tma"),        # clamp: 161 x 1, splits % 4 = 1
    (2, 32, 271, 257, "Identity", True, "tma"),      # D_in 271 (n_tail 16), splits % 4 = 2
    (1, 32, 257, 257, "Sigmoid", True, "tma"),       # one split
    (4, 96, 257, 385, "Identity", True, "tma"),      # 3 m-tiles + 1 SIMT row
    (5, 64, 120, 201, "Sigmoid", False, "tma"),      # no CMVN
    (600, 40, 257, 257, "Identity", True, "tc"),     # transposing kernel past one wave
    (900, 40, 129, 129, "Sigmoid", True, "tc_off"),
    (3, 33, 255, 130, "Identity", True, "tc"),       # 2 SIMT rows, D_in 255 (n_tail 0), F = 33
    (5, 64, 120, 131, "Sigmoid", True, "tc"),        # 3 SIMT rows, F a multiple of 32
    (7, 40, 201, 132, "ReLU", True, "tc"),           # 4 SIMT rows
    (2, 32, 271, 257, "Sigmoid", True, "tc"),
    (4, 96, 257, 385, "Identity", True, "tc_off"),
]
# per-utterance gradients: (B, F, D_in, D_out, act, cmvn, route); cmvn "meanstd" / "sums" / None; route "tma" (padded rows)
# or "tc" (dense rows)
EMB = [
    (44, 1001, 201, 201, "Sigmoid", "meanstd", "tma"),   # sub 1
    (32, 1001, 201, 201, "Identity", "sums", "tma"),     # sub 2, short last part
    (4, 96, 257, 385, "Identity", None, "tma"),          # sub 3
    (12, 1001, 201, 201, "Identity", "meanstd", "tma"),  # sub 4, short last part
    (5, 94, 129, 131, "Sigmoid", "meanstd", "tc"),       # sub 3, short last part, 3 SIMT rows
]
# folded objectives: (loss, B, F, D, act, hop, per_utt)
LOSS = [
    ("sisdr", 600, 40, 257, "Sigmoid", 256, False),     # clamp; sample lengths
    ("sisdr", 5, 64, 129, "Identity", 0, False),        # frame counts
    ("wsd", 900, 40, 129, "Sigmoid", 0, False),         # clamp, splits % 4 = 1
    ("wsd", 3, 101, 257, "Identity", 160, False),
    ("sisdr", 5, 94, 129, "Identity", 160, True),       # per-utterance, sub 3
    ("sisdr", 12, 1001, 201, "Sigmoid", 0, True),       # per-utterance, sub 4
]
# forward TMA head: (B, F, D_in, D_out, act, ld_out, out_offset_floats, cmvn)
FWD = [
    (2, 40, 257, 257, "Identity", 260, 0, True),       # one slab, bulk store
    (2, 40, 257, 257, "Identity", 257, 0, True),       # one slab, staging tile with per-row stores
    (2, 40, 257, 257, "Sigmoid", 260, 1, True),        # staging tile into an unaligned output
    (148, 128, 129, 129, "ReLU", 132, 0, True),        # tile_rows 128
    (150, 130, 201, 201, "Identity", 204, 0, True),    # dual, direct stores (2)
    (150, 130, 201, 201, "Sigmoid", 204, 1, False),    # dual, unaligned output: direct stores (1)
    (150, 130, 257, 257, "Identity", 260, 0, True),    # dual + SIMT column
    (64, 251, 513, 513, "Identity", 513, 0, True),     # dual + SIMT column, ld_out % 4 != 0: direct (1)
    (3, 40, 257, 300, "Identity", 300, 0, True),       # two slabs, direct (2)
    (2, 40, 257, 513, "Identity", 516, 0, True),       # two slabs at 513
    (1, 8, 544, 544, "Identity", 544, 0, True),        # D_in = D_out = 544, F = 8
    (3, 9, 544, 272, "Identity", 272, 0, True),        # F = 9: tiles straddle utterances
]
# forward register-staged head (se_linear_head_fwd_strided, precision 1): (B, F, D_in, D_out, act, vec, want_pred)
FWD_TC = [
    (3, 40, 257, 257, "Identity", True, True),         # 2 column chunks, predicted_out
    (2, 64, 120, 201, "Sigmoid", False, False),        # scalar loads, 1 chunk
    (1, 77, 513, 513, "Identity", True, False),        # 3 chunks
    (2, 50, 1025, 1025, "Identity", False, True),      # 5 chunks (n_fft 2048)
]


def bwd_branches(sms):
    """Branch labels that the case lists reach at `sms` SMs."""
    got = set()
    for B, F, Din, Dout, _, _, route in BWD:
        p = bwd_plan(B, F, Din, Dout, sms)
        kern = "tma" if route == "tma" else "tc"
        if p["clamped"] and p["splits"] * p["m_tiles"] > sms:
            got.add(f"{kern}:clamp>wave")
        got.add(f"{kern}:m_tiles{p['m_tiles']}")
        got.add(f"{kern}:n_tail{'>0' if p['n_tail'] else '=0'}")
        if kern == "tc":
            got.add(f"tc:simt{p['simt_rows']}")
        if p["splits"] == 1:
            got.add(f"{kern}:one_split")
        got.add(f"splits%4={p['splits'] % 4}")
        got.add(f"F={F}" if F in (32, 33) else ("F%32=0" if F % 32 == 0 else "F other"))
    for B, F, Din, Dout, _, _, route in EMB:
        p = bwd_plan(B, F, Din, Dout, sms, per_utt=True)
        got.add(f"emb:sub{p['sub']}")
        if F % p["rows"]:
            got.add("emb:short_last")
    for loss, B, F, D, _, hop, per_utt in LOSS:
        p = bwd_plan(B, F, D, D, sms, per_utt)
        got.add(f"{loss}:{'emb' if per_utt else 'rows'}:sub{p['sub']}" if per_utt else f"{loss}:rows")
    for B, F, Din, Dout, _, ld_out, off, _ in FWD:
        p = fwd_plan(B, F, Din, Dout, ld_out, sms, off % 4 == 0)
        if not p["dual"] and p["n_split"] == 1:
            got.add("fwd:single:bulk" if p["bulk_out"] else "fwd:single:staging")
        got.add(f"fwd:direct{p['direct_out']}")
        if p["dual"]:
            got.add("fwd:dual+1" if p["plus_one"] else "fwd:dual")
        if p["n_split"] == 2:
            got.add(f"fwd:n_split2@{Dout}")
        if p["tile_rows"] == 128:
            got.add("fwd:tile_rows128")
        if F % p["tile_rows"]:
            got.add("fwd:tile_straddles")
        if Din == 544:
            got.add("fwd:Din544")
    for B, F, Din, Dout, _, vec, _ in FWD_TC:
        got.add(f"tc_fwd:chunks{(Dout + 255) // 256}")
        got.add("tc_fwd:vec" if vec else "tc_fwd:scalar")
    return got


REQUIRED = {"tma:clamp>wave", "tc:clamp>wave", "tc:simt2", "tc:simt3", "tc:simt4", "tma:m_tiles3", "tc:m_tiles3",
            "tma:n_tail>0", "tc:n_tail>0", "tc:n_tail=0", "tma:one_split", "F=32", "F=33", "F%32=0",
            "splits%4=0", "splits%4=1", "splits%4=2", "splits%4=3", "emb:sub1", "emb:sub2", "emb:sub3", "emb:sub4",
            "emb:short_last", "sisdr:rows", "wsd:rows", "sisdr:emb:sub3", "sisdr:emb:sub4",
            "fwd:single:bulk", "fwd:single:staging", "fwd:direct0", "fwd:direct1", "fwd:direct2", "fwd:dual", "fwd:dual+1",
            "fwd:n_split2@300", "fwd:n_split2@513", "fwd:n_split2@544", "fwd:Din544", "fwd:tile_rows128",
            "fwd:tile_straddles", "tc_fwd:chunks1", "tc_fwd:chunks2", "tc_fwd:chunks3", "tc_fwd:chunks5", "tc_fwd:vec",
            "tc_fwd:scalar"}


def lib():
    from speech_enhancement_by_s3prl_b200 import _lib
    return _lib.load()


def device_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else SMS_B200


# ------------------------------------------------------------------------------------------------ CPU tests
def test_plan_mirror_matches_the_library_workspaces():
    """The Python mirror of plan() gives the library's workspace size for every backward and per-utterance case, and refuses
    what the library refuses."""
    L, sms = lib(), device_sms()
    for B, F, Din, Dout, *_ in BWD + [(B, F, D, D) for _, B, F, D, _, _, pu in LOSS if not pu]:
        p = bwd_plan(B, F, Din, Dout, sms)
        assert L.se_linear_head_bwd_tc_workspace(B, F, Din, Dout) == p["splits"] * p["m_rows"] * MAX_BROWS, (B, F, Din, Dout)
    for B, F, Din, Dout, *_ in EMB + [(B, F, D, D) for _, B, F, D, _, _, pu in LOSS if pu]:
        p = bwd_plan(B, F, Din, Dout, sms, per_utt=True)
        assert L.se_head_grad_embeddings_workspace(B, F, Din, Dout) == p["splits"] * p["m_rows"] * MAX_BROWS, (B, F, Din, Dout)
    for shape in ((2, 32, 272, 257), (2, 31, 257, 257), (3, 64, 300, 129)):
        assert bwd_plan(*shape, sms) is None and L.se_linear_head_bwd_tc_workspace(*shape) == 0
        assert bwd_plan(*shape, sms, per_utt=True) is None and L.se_head_grad_embeddings_workspace(*shape) == 0
    # SIMT rows 2 - 4 exist only in the transposing kernel: the folded-loss (TMA-only) entry points refuse them
    for B, F, Din, Dout, *_ in BWD:
        p = bwd_plan(B, F, Din, Dout, sms)
        ld = (max(Din, Dout) + 3) // 4 * 4
        assert L.se_linear_head_bwd_sisdr_supported(B, F, Din, Dout, ld, ld, ld, ld) == (1 if p["simt_rows"] <= 1 else 0)
    for B, F, Din, Dout, _, ld_out, off, _ in FWD:
        assert L.se_linear_head_fused_supported(B, F, Din, Dout, (Din + 3) // 4 * 4, (Din + 3) // 4 * 4, ld_out) == 1
    for shape in ((2, 40, 545, 257), (2, 40, 257, 545), (2, 7, 257, 257)):
        assert fwd_plan(*shape, 548, sms) is None and L.se_linear_head_fused_supported(*shape, 548, 548, 548) == 0


def test_case_list_covers_every_branch():
    got = bwd_branches(SMS_B200)
    assert REQUIRED <= got, sorted(REQUIRED - got)
    # the shapes of the issue table land where the table says
    assert [bwd_plan(*s, SMS_B200)["splits"] for s in ((600, 40, 257, 257), (1024, 32, 257, 257), (900, 40, 129, 129))] == [108, 171, 161]
    assert [bwd_plan(*s, SMS_B200, per_utt=True)["sub"] for s in ((44, 1001, 201, 201), (32, 1001, 201, 201), (4, 96, 257, 385),
                                                                 (12, 1001, 201, 201), (5, 94, 129, 129))] == [1, 2, 3, 4, 3]


# ------------------------------------------------------------------------------------------------ reference helpers
def rn(v):
    from speech_enhancement_by_s3prl_b200 import ops
    return ops.round_tf32(v.float().contiguous())


def span(v32, eps):
    """Width of the TF32 values the kernel's operand can round to when it lies within eps of v32 (0 almost everywhere)."""
    if eps is None:
        return None
    lo = rn((v32.double() - eps).float())
    hi = rn((v32.double() + eps).float())
    s = (hi.double() - lo.double())
    return s if bool((s != 0).any()) else None


def ulp_eps(v32, k=1.0):
    return v32.double().abs() * (k * 2.0 ** -23)


class Operands:
    """A (R, N) float32 restated operand with its eps bound: `t` = TF32 value fed to the reference, `v` = unrounded."""

    def __init__(self, v32, eps=None):
        self.v = v32.float()
        self.eps = eps
        self.t = rn(self.v).double()
        self.sp = span(self.v, eps)

    @classmethod
    def of(cls, v, t, eps, sp):
        o = cls.__new__(cls)
        o.v, o.t, o.eps, o.sp = v, t, eps, sp
        return o

    def map(self, f):
        """The same operand with `f` (a slice or a transpose) applied to each of its tensors."""
        g = lambda a: None if a is None else f(a)
        return Operands.of(f(self.v), f(self.t), g(self.eps), g(self.sp))

    def unrounded(self):
        """The operand as the fp32 SIMT dot products read it: no TF32 rounding, so the restated value differs from the
        kernel's by eps itself."""
        return Operands.of(self.v, self.v.double(), self.eps, None if self.eps is None else 2.0 * self.eps)


def activate(z, act):
    if act == "Sigmoid":
        return torch.sigmoid(z)
    if act == "ReLU":
        return z.clamp_min(0.0)
    return z


def bwd_check(got, A, X, name, p, transposing):
    """grad_W | grad_b (D_out, D_in + 1) against the reference.  The leftover output rows past the tensor-core tiles are fp32
    dot products: on unrounded dZ, and on unrounded x_hat in the transposing kernel (the TMA kernel reads its TF32 tile)."""
    n_left = p["m_tiles"] * BM if p["simt_rows"] else got.shape[0]
    blocks = -(-p["rows"] // BK)                                 # 32-row blocks accumulated into one fp32 accumulator
    _, tol = gemm_check(got[:n_left], A.map(lambda a: a[:, :n_left]), X, name, blocks=blocks)
    if n_left == got.shape[0]:
        return tol
    _, tol_s = gemm_check(got[n_left:], A.map(lambda a: a[:, n_left:]).unrounded(), X.unrounded() if transposing else X,
                          name + ":simt_rows", blocks=blocks)
    return torch.cat([tol, tol_s])


def gemm_check(got, A, Bop, name, act="Identity", add=None, blocks=1):
    """got (N, K) against act(A^T B + add) (A: R x N, B: R x K, contracted over R) with `blocks` 32-wide blocks accumulated into
    one fp32 accumulator; the tolerance counts blocks + 2 accumulation steps (the +2: the split reduction and the epilogue).
    Returns (reference pre-activation, pre-activation tolerance) and records the largest measured error ratio under `name`."""
    z = A.t.t() @ Bop.t
    S = A.t.abs().t() @ Bop.t.abs()
    allow = torch.zeros_like(S)
    if A.sp is not None:
        allow += A.sp.t() @ (Bop.t.abs() + (Bop.sp if Bop.sp is not None else 0))
    if Bop.sp is not None:
        allow += A.t.abs().t() @ Bop.sp
    if add is not None:
        z, S = z + add, S + add.abs()
    S = S * (blocks + 2)                                         # the tolerance grows with the accumulation depth
    tol = RTOL * S + allow
    got = got.double()
    # DESIGN section 2 against the unrounded operands
    z64 = A.v.double().t() @ Bop.v.double()
    S64 = A.v.double().abs().t() @ Bop.v.double().abs()
    E = torch.zeros_like(S64)
    if A.eps is not None:
        E += A.eps.t() @ (Bop.v.double().abs() + (Bop.eps if Bop.eps is not None else 0))
    if Bop.eps is not None:
        E += A.v.double().abs().t() @ Bop.eps
    if add is not None:
        z64 = z64 + add
    dtol = DESIGN_REL * S64 + 1.01 * E + tol
    if act == "Sigmoid":
        check(got, torch.sigmoid(z), 0.25 * S, 0.25 * allow + SIG_ATOL, 0.25 * tol + SIG_ATOL, name + ":sigmoid")
        dd, dtol = (got - torch.sigmoid(z64)).abs(), 0.25 * dtol + SIG_ATOL
    elif act == "ReLU":
        live = z.abs() > tol
        check(got, z.clamp_min(0.0), S, allow, tol, name, mask=live)
        dd = torch.where(z64.abs() > dtol, (got - z64.clamp_min(0.0)).abs(), torch.zeros_like(got))
    else:
        check(got, z, S, allow, tol, name)
        dd = (got - z64).abs()
    assert bool((dd <= dtol).all()), f"{name}: DESIGN section 2 bound broken by {(dd - dtol).max().item():.3e}"
    return z, tol


def act_tol(tol, act):
    return 0.25 * tol + SIG_ATOL if act == "Sigmoid" else tol


def check(got, ref, S, allow, tol, name, mask=None):
    err = (got - ref).abs()
    bad = ~(err <= tol)
    if mask is not None:
        bad &= mask
    ratio = ((err - allow) / S.clamp_min(1e-300))
    if mask is not None:
        ratio = torch.where(mask, ratio, torch.zeros_like(ratio))
    r = ratio.max().item()
    print(f"ERROR {name} {r:.3e}")                               # pytest -s: the numbers recorded in the module docstring
    if bool(bad.any()):
        idx = torch.nonzero(bad)[0].tolist()
        raise AssertionError(f"{name}: {int(bad.sum())} elements outside the bound; first {idx}: got {got[tuple(idx)].item():.9g} "
                             f"ref {ref[tuple(idx)].item():.9g} tol {tol[tuple(idx)].item():.3e} (ratio {r:.3e})")


def record_margin(name, m):
    print(f"MARGIN {name} {m:.1f}")
    assert m >= SENSITIVITY, f"{name}: a one-row mistake moves the reference by only {m:.2f} tolerances"


def rank1_margin(a_rows, b_rows, tol, chunk=256):
    """min over rows r of max_{n,k} |a_r[n] b_r[k]| / tol[n, k] (a_rows (M, N), b_rows (M, K))."""
    inv = (1.0 / tol).float()
    best = math.inf
    for i in range(0, a_rows.shape[0], chunk):
        a, b = a_rows[i:i + chunk].float().abs(), b_rows[i:i + chunk].float().abs()
        m = torch.einsum("mn,mk,nk->mnk", a, b, inv).amax((1, 2))
        best = min(best, m.min().item())
    return best


# ------------------------------------------------------------------------------------------------ inputs
def make_features(B, F, D, g):
    """log-power-like features: every (utterance, feature) has its own mean in [-20, 5] and scale in [0.3, 4]."""
    mu = torch.rand(B, 1, D, generator=g) * 25 - 20
    sd = 0.3 * (4 / 0.3) ** torch.rand(B, 1, D, generator=g)
    return mu + sd * torch.randn(B, F, D, generator=g)


def padded(t, LD, offset=0):
    """(B, F, D) -> device tensor (B, F, LD): NaN in the padding columns, its base `offset` floats into a NaN-filled buffer.
    Returns (tensor, LD)."""
    B, F, D = t.shape
    buf = torch.full((B * F * LD + 8,), float("nan"), device="cuda")
    v = buf[offset:offset + B * F * LD].view(B, F, LD)
    v[..., :D] = t.cuda()
    return v, LD


def burst_rows(B, F, plan, per_utt=False):
    R = B * F
    rows = set()
    for u in range(B):
        rows.update((u * F, u * F + F - 1))
    for ra, rb in plan["bounds"]:
        if rb <= ra:
            continue
        rows.update((ra, rb - 1))
        for r0 in range(ra, rb, BK):
            r1 = min(r0 + BK, rb)
            if r0 // F != (r1 - 1) // F:
                rows.update(range(r0, r1))
    return torch.tensor(sorted(r for r in rows if r < R), dtype=torch.long)


def cmvn_restate(x, B, F, cmvn, mode, sums=None, mean=None, std=None, eps=1e-6):
    """x (B, F, D) float32 device -> Operands of x_hat (R, D + 1) with the ones column, as the kernel `mode` computes it.
    mode: "fma" (TMA kernels: fmaf(x, sc, sh)), "sub" (transposing kernel: (x - mean) * sc), "rcp" (head_tc.cu: (x - mean) *
    __fdividef(1, std + eps)).  Also returns the per-utterance (sc, sh) float32 tables (B, D) for the sensitivity checks."""
    D = x.shape[2]
    x32 = x.float()
    sc_eps_rel = 0.0
    if cmvn == "sums":
        s1, s2 = sums[:, :D, 0], sums[:, :D, 1]
        m64 = s1 * (1.0 / F)
        var = ((s2 - s1 * m64) * (1.0 / (F - 1))).float()
        sc = 1.0 / (var.clamp_min(0).sqrt() + torch.tensor(eps, dtype=torch.float32))
        mf = m64.float()
        sc_eps_rel = 2.0 ** -21                                  # __fdividef: 2 ulp
    elif cmvn == "meanstd":
        mf = mean[:, :D].float()
        sc = 1.0 / (std[:, :D].float() + torch.tensor(eps, dtype=torch.float32))
        if mode == "rcp":
            sc_eps_rel = 2.0 ** -21
    else:
        mf = torch.zeros(B, D, device=x.device)
        sc = torch.ones(B, D, device=x.device)
    sh = (-mf * sc).float()
    if cmvn is None:
        v = x32
        eps_t = None
    elif mode == "fma":
        v = (x32.double() * sc[:, None].double() + sh[:, None].double()).float()
        # the kernel's shift is -mean * (its own scale): a scale off by d moves x * sc + sh by d |x_hat|, plus the rounding of the
        # shift, which may then land on the other side of a float32 rounding boundary
        eps_t = ulp_eps(v) + sc_eps_rel * v.double().abs()
        if sc_eps_rel:
            eps_t = eps_t + 2.0 ** -23 * (mf * sc)[:, None].double().abs()
    else:
        d = (x32 - mf[:, None]).float()
        v = (d * sc[:, None]).float()
        eps_t = ulp_eps(v) + sc_eps_rel * sc[:, None].double() * d.double().abs()
    R = B * F
    ones = torch.ones(R, 1, device=x.device)
    vv = torch.cat([v.reshape(R, D), ones], 1)
    ee = None if eps_t is None else torch.cat([eps_t.reshape(R, D), torch.zeros(R, 1, device=x.device, dtype=torch.float64)], 1)
    return Operands(vv, ee), (mf, sc, sh)


def xhat_with_stats(x_rows, mf, sc, sh, mode):
    """x_hat of rows x_rows (M, D) under the statistics (M, D) of another utterance (float32, mode as cmvn_restate)."""
    if mode == "fma":
        v = (x_rows.double() * sc.double() + sh.double()).float()
    else:
        v = ((x_rows - mf).float() * sc).float()
    return torch.cat([v, torch.ones(v.shape[0], 1, device=v.device)], 1)


def dact32(g, o, act):
    if act == "Sigmoid":
        return (g * (o * (1.0 - o))).float()
    if act == "ReLU":
        return torch.where(o > 0, g, torch.zeros_like(g))
    return g.float()


def make_head_operands(B, F, Dout, act, g):
    off = torch.rand(B, F, Dout, generator=g)
    if act == "ReLU":
        off = (off - 0.3).clamp_min(0.0)
    grad = torch.randn(B, F, Dout, generator=g)
    return off, grad


# ------------------------------------------------------------------------------------------------ GPU: plan coverage and trace
@pytest.fixture(scope="module")
def se():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import speech_enhancement_by_s3prl_b200 as pkg
    return pkg


@gpu
def test_case_list_covers_every_branch_on_this_device(se):
    got = bwd_branches(device_sms())
    assert REQUIRED <= got, sorted(REQUIRED - got)


@gpu
@pytest.mark.parametrize("case", [FWD[0], FWD[6], FWD[10]], ids=lambda c: f"{c[0]}x{c[1]}-{c[2]}-{c[3]}")
def test_forward_grid_matches_the_plan(se, case):
    """se_set_trace: every CTA of the TMA head records kernel id 2 once; the count is tiles x column slabs of the mirror."""
    from speech_enhancement_by_s3prl_b200 import ops
    B, F, Din, Dout, act, ld_out, off, _ = case
    p = fwd_plan(B, F, Din, Dout, ld_out, device_sms(), off % 4 == 0)
    L = lib()
    ldx = ops.round4(Din)
    x = torch.randn(B * F, ldx, device="cuda")
    W = torch.zeros(Dout, ldx, device="cuda")
    out = torch.empty(B * F * ld_out + 8, device="cuda")
    grid = p["tiles"] * p["n_split"]
    # room for every CTA the library could launch, whatever the mirror says: tiles of >= 8 rows, <= 2 column slabs, and
    # 7 records per CTA (marks 11 - 16 and the closing record)
    cap = 8 * 2 * -(-(B * F) // 8)
    buf = torch.zeros(1 + 4 * cap, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    L.se_set_trace(buf.data_ptr())
    try:
        rc = L.se_linear_head_fused(x.data_ptr(), ldx, None, 0, 1e-6, W.data_ptr(), ldx, None, B, F, Din, Dout, ops.ACT[act],
                                    out.data_ptr() + 4 * off, ld_out, ops._stream())
        torch.cuda.synchronize()
    finally:
        L.se_set_trace(None)
    assert rc == 0
    n = int(buf[0].item())
    assert n <= cap
    rec = buf[1:1 + 4 * n].view(n, 4).cpu()
    ids = rec[:, 0] >> 32
    blocks = (rec[ids == 2, 0] & 0xFFFFFFFF).tolist()
    assert len(blocks) == grid and sorted(blocks) == list(range(grid))


def boundary_moves(B, F, stats, x_rows_of, mode):
    """Rows that sit on an utterance boundary, with x_hat under the neighbouring utterance's statistics minus their own:
    (rows, difference (M, D + 1)).  stats = (mean, sc, sh) per utterance (B, D)."""
    mf, sc, sh = stats
    rows, nb = [], []
    for u in range(B):
        if u > 0:
            rows.append(u * F)
            nb.append(u - 1)
        if u < B - 1:
            rows.append(u * F + F - 1)
            nb.append(u + 1)
    if not rows:
        return None, None
    rows = torch.tensor(rows, dtype=torch.long)
    nb = torch.tensor(nb, dtype=torch.long, device="cuda")
    xr = x_rows_of(rows)
    own = torch.div(rows, F, rounding_mode="floor").cuda()
    moved = xhat_with_stats(xr, mf[nb], sc[nb], sh[nb], mode).double()
    mine = xhat_with_stats(xr, mf[own], sc[own], sh[own], mode).double()
    return rows, rn(moved).double() - rn(mine).double()


def ctypes_ws(n):
    return torch.empty(max(int(n), 1), device="cuda")


# ------------------------------------------------------------------------------------------------ GPU: weight gradient
@gpu
@pytest.mark.parametrize("case", BWD, ids=lambda c: f"{c[6]}-{c[0]}x{c[1]}-{c[2]}-{c[3]}-{c[4]}-{'cmvn' if c[5] else 'raw'}")
def test_weight_gradient_matches_float64(se, case):
    """se_linear_head_bwd_fused (TMA kernel) and se_linear_head_bwd_tc (transposing kernel) + the split reduction."""
    from speech_enhancement_by_s3prl_b200 import ops
    B, F, Din, Dout, act, cmvn, route = case
    p = bwd_plan(B, F, Din, Dout, device_sms())
    g = torch.Generator().manual_seed(B * 7919 + F * 31 + Din * 3 + Dout)
    x = make_features(B, F, Din, g)
    off, grad = make_head_operands(B, F, Dout, act, g)
    R = B * F
    burst = burst_rows(B, F, p)
    grad.view(R, Dout)[burst] *= 100.0
    L = lib()
    if route == "tma":
        LDx, LDo = ops.round4(Din), ops.round4(Dout)
        xf, _ = padded(x, LDx)
        of, _ = padded(off, LDo)
        gf, _ = padded(grad, LDo)
        sums = ops.feature_sums(xf, Din) if cmvn else None
        gw, gb = ops.linear_head_bwd_fused(xf, Din, sums, 1e-6, of, gf, Dout, act)
        X, stats = cmvn_restate(x.cuda(), B, F, "sums" if cmvn else None, "fma", sums=sums)
    else:
        shift = 1 if route == "tc_off" else 0
        LDx, LDo = (ops.round4(Din), ops.round4(Dout)) if shift else (Din, Dout)
        xf, _ = padded(x, LDx, shift)
        of, _ = padded(off, LDo, shift)
        gf, _ = padded(grad, LDo, shift)
        mean, std = x.mean(1).cuda(), x.std(1).cuda()
        ws = ctypes_ws(L.se_linear_head_bwd_tc_workspace(B, F, Din, Dout))
        gw, gb = torch.empty(Dout, Din, device="cuda"), torch.empty(Dout, device="cuda")
        rc = L.se_linear_head_bwd_tc(xf.data_ptr(), LDx, mean.data_ptr(), std.data_ptr(), Din, 1e-6, of.data_ptr(), gf.data_ptr(), LDo,
                                     B, F, Din, Dout, ops.ACT[act], ws.data_ptr(), ws.numel(), gw.data_ptr(), gb.data_ptr(), ops._stream())
        assert rc == 0, lib_error()
        X, stats = cmvn_restate(x.cuda(), B, F, "meanstd", "sub", mean=mean, std=std)
    torch.cuda.synchronize()
    A = Operands(dact32(grad.cuda(), off.cuda(), act).reshape(R, Dout))
    got = torch.cat([gw, gb[:, None]], 1)
    assert torch.isfinite(got).all()
    kern = "bwd_tma" if route == "tma" else "bwd_transposing"
    tol = bwd_check(got, A, X, kern, p, route != "tma")
    name = f"{kern} {B}x{F}-{Din}-{Dout}"
    record_margin(name + " burst", rank1_margin(A.t[burst.cuda()], X.t[burst.cuda()], tol))
    if cmvn:
        rows, diff = boundary_moves(B, F, stats, lambda r: x.view(R, Din)[r].cuda(), "fma" if route == "tma" else "sub")
        if rows is not None:
            record_margin(name + " boundary", rank1_margin(A.t[rows.cuda()], diff, tol))


def lib_error():
    from speech_enhancement_by_s3prl_b200 import _lib
    return _lib.last_error()


# ------------------------------------------------------------------------------------------------ GPU: per-utterance gradients
def per_utt_checks(out, A, X, B, F, Din, Dout, name, p, transposing=False):
    """Row u of `out` against the utterance's own rows; returns the tolerance of every utterance."""
    P = Dout * Din
    tols = []
    for u in range(B):
        sl = slice(u * F, (u + 1) * F)
        got = torch.cat([out[u, :P].view(Dout, Din), out[u, P:][:, None]], 1)
        tols.append(bwd_check(got, A.map(lambda a: a[sl]), X.map(lambda a: a[sl]), name, p, transposing))
    return tols


def per_utt_margins(name, A, X, tols, B, F, burst, rows=None, diff=None):
    m_burst = m_next = m_bnd = math.inf
    bset = burst.tolist()
    for u in range(B):
        br = torch.tensor([r for r in bset if u * F <= r < (u + 1) * F], dtype=torch.long, device="cuda")
        m_burst = min(m_burst, rank1_margin(A.t[br], X.t[br], tols[u]))
        if u + 1 < B:                                            # one row of the next utterance counted in
            r = torch.tensor([(u + 1) * F], device="cuda")
            m_next = min(m_next, rank1_margin(A.t[r], X.t[r], tols[u]))
        if rows is not None:
            sel = torch.nonzero((rows >= u * F) & (rows < (u + 1) * F)).flatten()
            if len(sel):
                m_bnd = min(m_bnd, rank1_margin(A.t[rows[sel].cuda()], diff[sel.cuda()], tols[u]))
    record_margin(name + " burst", m_burst)
    if B > 1:
        record_margin(name + " next-utterance row", m_next)
    if rows is not None:
        record_margin(name + " boundary", m_bnd)


@gpu
@pytest.mark.parametrize("case", EMB, ids=lambda c: f"{c[6]}-{c[0]}x{c[1]}-{c[2]}-{c[3]}-{c[4]}-{c[5]}")
def test_per_utterance_gradients_match_float64(se, case):
    """se_head_grad_embeddings: one split per (utterance, part), partials packed per utterance in a fixed order."""
    from speech_enhancement_by_s3prl_b200 import ops
    B, F, Din, Dout, act, cmvn, route = case
    p = bwd_plan(B, F, Din, Dout, device_sms(), per_utt=True)
    g = torch.Generator().manual_seed(B * 131 + F * 17 + Din + 5 * Dout)
    x = make_features(B, F, Din, g) if cmvn else torch.randn(B, F, Din, generator=g)
    off, grad = make_head_operands(B, F, Dout, act, g)
    R = B * F
    burst = burst_rows(B, F, p)
    grad.view(R, Dout)[burst] *= 100.0
    L = lib()
    LDx, LDo = (ops.round4(Din), ops.round4(Dout)) if route == "tma" else (Din, Dout)
    xf, _ = padded(x, LDx)
    of, _ = padded(off, LDo)
    gf, _ = padded(grad, LDo)
    mean = std = sums = None
    if cmvn == "meanstd":
        mean, std = x.mean(1).cuda(), x.std(1).cuda()
    elif cmvn == "sums":
        sums = ops.feature_sums(xf, Din)
    ws = ctypes_ws(L.se_head_grad_embeddings_workspace(B, F, Din, Dout))
    out = torch.empty(B, Dout * Din + Dout, device="cuda")
    ld_stats = Din if mean is not None else (sums.shape[1] if sums is not None else 0)
    rc = L.se_head_grad_embeddings(xf.data_ptr(), LDx, ops._p(mean), ops._p(std), ops._p(sums), ld_stats, 1e-6, of.data_ptr(),
                                   gf.data_ptr(), LDo, B, F, Din, Dout, ops.ACT[act], ws.data_ptr(), ws.numel(), out.data_ptr(), ops._stream())
    assert rc == 0, lib_error()
    torch.cuda.synchronize()
    mode = "fma" if route == "tma" else "sub"
    X, stats = cmvn_restate(x.cuda(), B, F, cmvn, mode, sums=sums, mean=mean, std=std)
    A = Operands(dact32(grad.cuda(), off.cuda(), act).reshape(R, Dout))
    assert torch.isfinite(out).all()
    kern = "per_utt_tma" if route == "tma" else "per_utt_transposing"
    tols = per_utt_checks(out, A, X, B, F, Din, Dout, kern, p, route != "tma")
    rows = diff = None
    if cmvn:
        rows, diff = boundary_moves(B, F, stats, lambda r: x.view(R, Din)[r].cuda(), mode)
    per_utt_margins(f"{kern} {B}x{F}-{Din}-{Dout}", A, X, tols, B, F, burst, rows, diff)


# ------------------------------------------------------------------------------------------------ GPU: folded objectives
def loss_frames(B, F, g):
    """Valid frames per utterance: all of them, a length beyond F (clamped), frames that end exactly on a 32-row block of the
    batch, mid-block, one frame, and random ones."""
    fr = torch.randint(1, F + 1, (B,), generator=g)
    for u in range(B):
        k = u % 6
        if k == 0:
            fr[u] = F
        elif k == 1:
            fr[u] = F + 3
        elif k == 2:
            v = (-u * F) % BK
            fr[u] = v if 0 < v <= F else BK
        elif k == 3:
            fr[u] = min(F, ((-u * F) % BK) + BK // 2) or 1
        elif k == 4:
            fr[u] = 1
    return fr


def sisdr_grad64(off, inp, tar, frames, go, eps=1e-10):
    """d (sum_u go * loss_u) / d offset of objective.SISDR on predicted = offset * linear_inp, float64 autograd, and the
    per-element scale of the kernel's two-term expression (for the operand eps)."""
    B, F, D = off.shape
    o64 = off.double().requires_grad_(True)
    x64, t64 = inp.double(), tar.double()
    m = (torch.arange(F, device=off.device)[None, :] < frames[:, None]).double()[..., None]
    src, tgt = (o64 * x64).clamp_min(0).sqrt() * m, t64.clamp_min(0).sqrt() * m
    al = (src * tgt).sum((1, 2)) / ((tgt ** 2).sum((1, 2)) + eps)
    num = ((al[:, None, None] * tgt) ** 2).sum((1, 2))
    den = ((al[:, None, None] * tgt - src) ** 2).sum((1, 2)) + eps
    loss = -10 * torch.log10(num / den + eps)
    (loss.sum() * go).backward()
    with torch.no_grad():                                        # sisdr_coef of head_bwd_tc.cu
        st, tt, ss = (src * tgt).sum((1, 2)), (tgt ** 2).sum((1, 2)), (src ** 2).sum((1, 2))
        a = st / (tt + eps)
        Aa = a * a * tt
        Dd = a * a * tt - 2 * a * st + ss + eps
        kap = -10.0 / (math.log(10.0) * (Aa / Dd + eps) * Dd * Dd)
        ca = 2 * a * tt / (tt + eps)
        cd = 2 * (a * tt - st) / (tt + eps) - 2 * a
        cx, cy = (go * kap * (ca * Dd - Aa * cd))[:, None, None], (go * kap * (-2 * Aa))[:, None, None]
        pi = o64.detach() * x64
        scale = (cx.abs() * t64.sqrt() + cy.abs() * pi.sqrt()) * 0.5 * x64 / pi.sqrt()
    return o64.grad, scale


def wsd_grad64(off, inp, tar, frames, energy64, thres, alpha):
    B, F, D = off.shape
    m = (torch.arange(F, device=off.device)[None, :] < frames[:, None]).double()[..., None]
    voiced = (10 * torch.log10(energy64 + 1e-10) > thres).double()[..., None]
    G, X, S = off.double(), inp.double(), tar.double()
    n = (X - S).clamp_min(0)
    g = (alpha * 2 * (S - G * S) * (-S) * voiced + (1 - alpha) * 2 * G * n * n) * m / B
    big = torch.maximum(X.abs(), S.abs())
    scale = (alpha * 2 * (S.abs() + (G * S).abs()) * S.abs() + (1 - alpha) * 2 * G.abs() * (n + 2.0 ** -22 * big) ** 2) * m / B
    return g, scale


def live_only(rows, diff, live):
    """The boundary rows inside the valid frames (a padded frame carries no gradient to move)."""
    keep = live.reshape(-1)[rows.cuda()]
    return rows[keep.cpu()], diff[keep]


@gpu
@pytest.mark.parametrize("case", LOSS, ids=lambda c: f"{c[0]}-{'per_utt' if c[6] else 'rows'}-{c[1]}x{c[2]}-{c[3]}-{c[4]}-hop{c[5]}")
def test_folded_objective_gradient_matches_float64(se, case):
    """se_linear_head_bwd_sisdr / _wsd and se_head_grad_embeddings_sisdr: d loss / d offset rebuilt inside the TMA kernel."""
    from speech_enhancement_by_s3prl_b200 import ops
    loss, B, F, D, act, hop, per_utt = case
    p = bwd_plan(B, F, D, D, device_sms(), per_utt)
    g = torch.Generator().manual_seed(B * 977 + F * 13 + D + hop)
    x = make_features(B, F, D, g)
    off = torch.rand(B, F, D, generator=g) * 0.9 + 0.05
    R = B * F
    fr = loss_frames(B, F, g)
    # the burst rows here also include the last valid frame and the first padded one of every utterance
    ends = [u * F + min(int(v), F) - 1 for u, v in enumerate(fr)] + [u * F + int(v) for u, v in enumerate(fr) if v < F]
    burst = torch.tensor(sorted(set(burst_rows(B, F, p).tolist()) | set(ends)), dtype=torch.long)
    if loss == "sisdr":
        inp, tar = torch.randn(B, F, D, generator=g) ** 2 + 1e-3, torch.randn(B, F, D, generator=g) ** 2 + 1e-3
        inp.view(R, D)[burst] *= 100.0
        tar.view(R, D)[burst] *= 100.0
    else:
        level = 10.0 ** (-4.0 * torch.rand(B, F, 1, generator=g))
        level.view(R)[burst] = 1.0                               # burst rows at the loud end of the 40 dB spread
        tar = (torch.rand(B, F, D, generator=g) ** 4) * 3.0 * level
        inp = tar + (torch.rand(B, F, D, generator=g) - 0.3).clamp_min(-0.2) * tar.mean(-1, keepdim=True)
        inp.view(R, D)[burst] *= 10.0
        tar.view(R, D)[burst] *= 10.0
        # keep every frame energy at least 1 dB away from the voicing threshold: a frame within 1 dB is decided by the
        # rounding of its fp32 energy, not by the kernel
        e = tar.double().sum(-1)
        thres = 10 * torch.log10(e.max() + 1e-10) - 30.0
        near = (10 * torch.log10(e + 1e-10) - thres).abs() < 1.0
        tar[near] *= 10.0 ** -0.25
        inp[near] *= 10.0 ** -0.25
    lens = ((fr - 1) * hop + torch.randint(0, max(hop, 1), (B,), generator=g)) if hop else fr.clone()
    frames = fr.clamp_max(F).cuda()
    LD = ops.round4(D)
    xf, _ = padded(x, LD)
    of, _ = padded(off, LD)
    inf_, _ = padded(inp, LD)
    tf, _ = padded(tar, LD)
    lens_d = lens.cuda()
    sums = ops.feature_sums(xf, D)
    assert ops.linear_head_bwd_sisdr_supported(B, F, D, D, LD, LD, LD, LD)
    L = lib()
    alpha = 0.5
    if loss == "sisdr":
        sums3 = ops.sisdr_mask_step(of, inf_, tf, lens_d, hop, D, want_grad=False)[3]
        if per_utt:
            ws = ctypes_ws(L.se_head_grad_embeddings_workspace(B, F, D, D))
            out = torch.empty(B, D * D + D, device="cuda")
            rc = L.se_head_grad_embeddings_sisdr(xf.data_ptr(), LD, sums.data_ptr(), sums.shape[1], 1e-6, of.data_ptr(), LD,
                                                 inf_.data_ptr(), LD, tf.data_ptr(), LD, lens_d.data_ptr(), hop, sums3.data_ptr(),
                                                 1e-10, B, F, D, D, ops.ACT[act], ws.data_ptr(), ws.numel(), out.data_ptr(), ops._stream())
            assert rc == 0, lib_error()
        else:
            gw, gb = ops.linear_head_bwd_sisdr(xf, D, sums, 1e-6, of, inf_, tf, lens_d, hop,
                                               sums3, D, act)
        grad_of = lambda fr_: sisdr_grad64(off.cuda(), inp.cuda(), tar.cuda(), fr_, 1.0 if per_utt else 1.0 / B)
    else:
        energy, emax = ops.wsd_energy(tf, D)
        gw, gb = ops.linear_head_bwd_wsd(xf, D, sums, 1e-6, of, inf_, tf, lens_d, hop,
                                         energy, emax, D, act, alpha=alpha, db_interval=30.0)
        e64 = tar.cuda().double().sum(-1)
        thres = 10 * math.log10(float(emax.item()) + 1e-10) - 30.0
        assert ((10 * torch.log10(e64 + 1e-10) - thres).abs() >= 1.0).all()
        grad_of = lambda fr_: wsd_grad64(off.cuda(), inp.cuda(), tar.cuda(), fr_, e64, thres, alpha)
    torch.cuda.synchronize()
    g64, gscale = grad_of(frames)
    o32 = off.cuda()
    g32 = g64.float()
    slope = o32.double() * (1 - o32.double()) if act == "Sigmoid" else torch.ones_like(o32, dtype=torch.float64)
    dz = dact32(g32, o32, act)
    live = (torch.arange(F, device="cuda")[None, :] < frames[:, None])[..., None]
    eps = ((2.0 ** -18 * gscale + ulp_eps(g32)) * slope + ulp_eps(dz, 2.0)) * live
    A = Operands(dz.reshape(R, D), eps.reshape(R, D))
    burst = burst[live.reshape(R)[burst.cuda()].cpu()]
    X, stats = cmvn_restate(x.cuda(), B, F, "sums", "fma", sums=sums)
    kern = f"{loss}_{'per_utt' if per_utt else 'rows'}"
    name = f"{kern} {B}x{F}-{D}"
    # one valid frame more / fewer: the rows of dZ that would appear / vanish
    g_more, _ = grad_of((frames + 1).clamp_max(F))
    dz_more = dact32(g_more.float(), o32, act).reshape(R, D)
    u_all = torch.arange(B, device="cuda")
    last = u_all * F + frames - 1
    has_next = frames < F
    nxt = (u_all * F + frames)[has_next]
    if per_utt:
        tols = per_utt_checks(out, A, X, B, F, D, D, kern, p)
        rows, diff = live_only(*boundary_moves(B, F, stats, lambda r: x.view(R, D)[r].cuda(), "fma"), live)
        per_utt_margins(name, A, X, tols, B, F, burst, rows, diff)
        m_less = min(rank1_margin(A.t[last[u:u + 1]], X.t[last[u:u + 1]], tols[u]) for u in range(B))
        m_more = min([rank1_margin(rn(dz_more[r:r + 1]).double(), X.t[r:r + 1], tols[int(r) // F]) for r in nxt.tolist()] or [math.inf])
    else:
        got = torch.cat([gw, gb[:, None]], 1)
        assert torch.isfinite(got).all()
        tol = bwd_check(got, A, X, kern, p, False)
        record_margin(name + " burst", rank1_margin(A.t[burst.cuda()], X.t[burst.cuda()], tol))
        rows, diff = live_only(*boundary_moves(B, F, stats, lambda r: x.view(R, D)[r].cuda(), "fma"), live)
        record_margin(name + " boundary", rank1_margin(A.t[rows.cuda()], diff, tol))
        m_less = rank1_margin(A.t[last], X.t[last], tol)
        m_more = rank1_margin(rn(dz_more[nxt]).double(), X.t[nxt], tol) if len(nxt) else math.inf
    record_margin(name + " frame fewer", m_less)
    record_margin(name + " frame more", m_more)


# ------------------------------------------------------------------------------------------------ GPU: forward heads
SENTINEL = -7.25


def out_buffer(R, ld_out, shift, guard_rows=2, pre=8):
    buf = torch.full((pre + shift + (R + guard_rows) * ld_out,), SENTINEL, device="cuda")
    return buf, pre + shift


def check_guards(buf, start, R, ld_out):
    assert (buf[:start] == SENTINEL).all(), "the head wrote before its output"
    assert (buf[start + R * ld_out:] == SENTINEL).all(), "the head wrote past row R"


def forward_margins(name, z, tol, act, X_rows_of, stats, W_t, B, F, mode):
    rows, diff = boundary_moves(B, F, stats, X_rows_of, mode)
    if rows is None:
        return
    rr = rows.cuda()
    dz = diff[:, :-1] @ W_t                                      # (M, Dout): the pre-activation move
    z0 = z[rr]
    move = (activate(z0 + dz, act) - activate(z0, act)).abs()
    record_margin(name + " boundary", (move / act_tol(tol[rr], act)).amax(1).min().item())


@gpu
@pytest.mark.parametrize("case", FWD, ids=lambda c: f"{c[0]}x{c[1]}-{c[2]}-{c[3]}-{c[4]}-ld{c[5]}-off{c[6]}")
def test_tma_forward_head_matches_float64(se, case):
    """se_linear_head_fused through the C ABI: the output stride and base pointer chosen by the caller."""
    from speech_enhancement_by_s3prl_b200 import ops
    B, F, Din, Dout, act, ld_out, shift, cmvn = case
    p = fwd_plan(B, F, Din, Dout, ld_out, device_sms(), shift % 4 == 0)
    g = torch.Generator().manual_seed(B * 71 + F + Din * 7 + Dout + ld_out)
    x = make_features(B, F, Din, g) if cmvn else torch.randn(B, F, Din, generator=g)
    R = B * F
    LDx = ops.round4(Din)
    xf, _ = padded(x, LDx)
    W = torch.full((Dout, LDx), float("nan"))
    W[:, :Din] = torch.randn(Dout, Din, generator=g) * (0.5 / math.sqrt(Din))
    W = ops.round_tf32(W.cuda())
    b = (torch.randn(Dout, generator=g) * 0.5).cuda()
    sums = ops.feature_sums(xf, Din) if cmvn else None
    buf, start = out_buffer(R, ld_out, shift)
    L = lib()
    assert L.se_linear_head_fused_supported(B, F, Din, Dout, LDx, LDx, ld_out) == 1
    rc = L.se_linear_head_fused(xf.data_ptr(), LDx, ops._p(sums), 0 if sums is None else sums.shape[1], 1e-6, W.data_ptr(), LDx,
                                b.data_ptr(), B, F, Din, Dout, ops.ACT[act], buf.data_ptr() + 4 * start, ld_out, ops._stream())
    assert rc == 0, lib_error()
    torch.cuda.synchronize()
    check_guards(buf, start, R, ld_out)
    got = buf[start:start + R * ld_out].view(R, ld_out)[:, :Dout]
    assert torch.isfinite(got).all()
    X, stats = cmvn_restate(x.cuda(), B, F, "sums" if cmvn else None, "fma", sums=sums)
    Xt = X.map(lambda a: a[:, :Din].t())                        # (D_in, R): contracted over the features
    Wop = Operands(W[:, :Din].t())
    kern = "fwd_tma" + (":simt_column" if p["plus_one"] else "")
    kb = -(-Din // BK)
    z, tol = gemm_check(got, Xt, Wop, "fwd_tma", act=act, add=b.double()[None, :], blocks=kb)
    if p["plus_one"]:                                            # the fp32 SIMT column on its own
        gemm_check(got[:, -1:], Xt, Operands(W[-1:, :Din].t()), kern, act=act, add=b.double()[None, -1:], blocks=kb)
    if cmvn:
        forward_margins(f"fwd_tma {B}x{F}-{Din}-{Dout}", z, tol, act, lambda r: x.view(R, Din)[r].cuda(), stats,
                        W[:, :Din].double().t(), B, F, "fma")


@gpu
@pytest.mark.parametrize("case", FWD_TC, ids=lambda c: f"{c[0]}x{c[1]}-{c[2]}-{c[3]}-{c[4]}-{'vec' if c[5] else 'scalar'}")
def test_register_staged_forward_head_matches_float64(se, case):
    """se_linear_head_fwd_strided with precision 1 (head_tc.cu): 128-row tiles across many utterances, column chunks of <= 256."""
    from speech_enhancement_by_s3prl_b200 import ops
    B, F, Din, Dout, act, vec, want_pred = case
    g = torch.Generator().manual_seed(B * 53 + F + Din + 3 * Dout)
    x = make_features(B, F, Din, g)
    R = B * F
    shift = 0 if vec else 1
    LDx = ops.round4(Din)
    xf, _ = padded(x, LDx, shift)
    W = torch.full((Dout, LDx), float("nan"))
    W[:, :Din] = torch.randn(Dout, Din, generator=g) * (0.5 / math.sqrt(Din))
    Wd = W.cuda()
    b = (torch.randn(Dout, generator=g) * 0.5).cuda()
    mean = torch.full((B, LDx), float("nan"), device="cuda")
    std = torch.full((B, LDx), float("nan"), device="cuda")
    mean[:, :Din], std[:, :Din] = x.mean(1).cuda(), x.std(1).cuda()
    ld_out = ops.round4(Dout)
    buf, start = out_buffer(R, ld_out, 0)
    lin = pbuf = None
    if want_pred:
        lin = torch.rand(R, ld_out, device="cuda")
        pbuf, _ = out_buffer(R, ld_out, 0)
    rc = lib().se_linear_head_fwd_strided(xf.data_ptr(), LDx, mean.data_ptr(), std.data_ptr(), LDx, 1e-6, Wd.data_ptr(), LDx,
                                          b.data_ptr(), B, F, Din, Dout, ops.ACT[act], ops._p(lin), buf.data_ptr() + 4 * start,
                                          None if pbuf is None else pbuf.data_ptr() + 4 * start, ld_out, 1, ops._stream())
    assert rc == 0, lib_error()
    torch.cuda.synchronize()
    check_guards(buf, start, R, ld_out)
    got = buf[start:start + R * ld_out].view(R, ld_out)[:, :Dout]
    assert torch.isfinite(got).all()
    if want_pred:
        check_guards(pbuf, start, R, ld_out)
        pred = pbuf[start:start + R * ld_out].view(R, ld_out)[:, :Dout]
        assert torch.equal(pred, lin[:, :Dout] * got)
    X, stats = cmvn_restate(x.cuda(), B, F, "meanstd", "rcp", mean=mean, std=std)
    Xt = X.map(lambda a: a[:, :Din].t())                        # (D_in, R): contracted over the features
    Wr = rn(Wd[:, :Din])
    z, tol = gemm_check(got, Xt, Operands(Wr.t()), "fwd_register_staged", act=act, add=b.double()[None, :], blocks=-(-Din // BK))
    forward_margins(f"fwd_register_staged {B}x{F}-{Din}-{Dout}", z, tol, act, lambda r: x.view(R, Din)[r].cuda(), stats,
                    Wr.double().t(), B, F, "sub")
