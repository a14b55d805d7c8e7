"""Every GEMM of the five fused update engines, kernel by kernel, against float64 computed from the kernel's own inputs.

Isolation.  Each engine runs one ``update()`` with learning rate 0 and tau 0: Adam's step size is 0 and polyak is the identity, so
``params`` and ``targets`` come back bit-identical (asserted).  Every phase of the step then read the same, known weights, and the order
of the phases inside a step no longer matters.  The ``grads`` block holds every gradient the step formed, and the workspace holds the
activations of the last phase, found through a Python mirror of the workspace layout (``td3_carve``, ``bcq_carve``, ``ma_carve``, checked
against ``cstr_*_workspace_bytes``).  Two fresh engines per case: a critic-only step (delay 2) for the critic-phase slots, and a policy
step (delay 1) for the actor-phase slots.  SAC always takes a policy step, so its critic phase is read from a copy of the workspace
taken in the ``allreduce`` hook between the phases.

Each kernel output is compared on every element with a float64 reference computed from the workspace values the kernel read, against a
bound derived from the kernel's arithmetic (U = 2^-24, the float32 unit roundoff; ULP = 2^-23):

* float32 FFMA (``td3_gemm_kernel``, split-K partials, ``td3_splitk_finish_kernel``, the ``td3_finalize_kernel`` slab sum, every layer-1
  and head kernel): a dot product of length k accumulated in any order errs by at most k * U * sum|a*b|; each split-K partial or slab
  adds one rounding, the bias one more:  (k + splits + 2) * U * (sum|a*b| + |bias|).
* ``gemm="tensor"`` (``td3_gemm_tc_kernel``, three bf16 planes): the reference emulates the documented arithmetic exactly.  Planes are
  cut by truncation as ``split_store`` does (x1 = x & 0xffff0000, r = x - x1, x2 = hi16(r), x3 = hi16(r - x2)) and the six products
  a1b1 + a1b2 + a2b1 + a2b2 + a1b3 + a3b1 are summed in float64.  What is left is accumulation: each bf16 x bf16 product is exact in
  fp32, and the tensor core's accumulation truncates, so every MMA may lose up to MMA_ULPS fp32 ulps of the running sum, which is at
  most sum|a*b|, and these errors all point the same way.  One ulp per MMA (the rollout tests' model) was exceeded once (1.05 of it,
  a 32 x 32 weight gradient over 64 rows); the bound allows two, one for aligning the addends and one for the result.  Six MMAs per
  K = 16 step, two steps per K = 32 stage:  2 * MMA_ULPS * 6 * ceil(k / 32) * ULP * sum|a*b|, plus (splits - 1) * U * sum|a*b| for the
  slab sum and U * (sum|a*b| + |bias|) for the epilogue.  Dropping a1b3 and a3b1 moves a product by up to 2^-15 of |a*b|, which the
  small-K cases see.
* ``gemm="bf16"`` (plain bf16 operands): operands rounded to nearest even as ``cvt.rn.bf16x2`` does, products summed in float64; one MMA
  per K = 16 step, so 2 * MMA_ULPS * ceil(k / 32) * ULP * sum|a*b| plus the same slab and epilogue terms.  This is the mode's per-step bar.
* skinny weight gradients (``td3_skinny_wgrad_kernel`` + the finalize job): 8 rows per warp, 8 warps, then the chunk sums in four
  interleaved accumulators: (19 + ceil(chunks / 4)) * U * sum|x*y|.
* heads: the critic head's dz2 = dq * w3 is one rounding; ``mlp_head_bwd_kernel`` and the actor backward heads are out + 1 roundings.
* ReLU is 1-Lipschitz, so the bounds carry through it; the backward masks are the kernel's own (``h > 0`` on the workspace values).
* The decoder's layer-1 weight gradient (``wgrad_gemm_direct`` over the 4 + L wide input) reads a dz1 the encoder's backward overwrote.
  Its reference is the float64 chain from the decoder's head, and the bound adds the propagated error of the two GEMMs before it, taken
  against the exact product: (k + 10) * U (fp32), 4 * U + the accumulation term (tensor: the dropped plane terms), 2^-8 + the
  accumulation term (bf16: two operand roundings).

``python -m pytest -s`` prints the largest |error| / bound per kernel output, engine, mode and case.  A branch mirror of
``launch_gemm``'s split-K decision, ``choose_splits`` and ``tc_tile`` (csrc/cstr_td3.cu, cstr_td3_tc.cuh) shows that the cases reach
every branch in every mode.
"""
import collections

import numpy as np
import pytest
import torch

import td3_util as TU

gpu = pytest.mark.gpu

f32, f64 = np.float32, np.float64
U = 2.0 ** -24
ULP = 2.0 ** -23
MMA_ULPS = 2  # fp32 ulps of sum|a*b| one tcgen05 MMA may lose to its truncating accumulation
BM, BN, BK = 128, 64, 16          # td3_gemm_kernel's CTA tile
TC_BM, TC_KC = 128, 32            # td3_gemm_tc_kernel: rows per CTA, K per stage
MAX_SPLITS, SKINNY_ROWS, OBS, ACT = 16, 64, 4, 2
B200_SMS = 148
MODES = ("fp32", "tensor", "bf16")


def cdiv(a, b):
    return -(-a // b)


def pad4(n):
    return (n + 3) & ~3


# ---- workspace mirrors ---------------------------------------------------------------------------------------------------------------
class _Bump:
    """The bump allocator of carve() / Bump: every slot padded to 4 floats."""

    def __init__(self):
        self.o, self.slots = 0, {}

    def take(self, name, n):
        self.slots[name] = self.o
        self.o += pad4(n)


def _mlp_scratch(b, rows, hm, z, ny):
    cap = MAX_SPLITS * z * pad4(hm * hm)
    b.take("slabs", cap)
    b.take("skinny", 3 * cdiv(rows, SKINNY_ROWS) * z * (ny + 1) * cdiv(hm, 32) * 32)
    return cap


def td3_carve(B, H1, H2):
    """carve() in csrc/cstr_td3.cu (TD3 and SAC): (slots, floats, capacity of the split-K slabs)."""
    b = _Bump()
    rb = cdiv(B, 8)
    cap = MAX_SPLITS * 2 * pad4(H1 * H2)
    for name, n in (("h1", 2 * B * H1), ("h2", 2 * B * H2), ("dz1", 2 * B * H1), ("dz2", 2 * B * H2), ("t_h1", 2 * B * H1), ("t_h2", 2 * B * H2),
                    ("a_h1", B * H1), ("a_h2", B * H2), ("next_act", 2 * B), ("a_pi", 2 * B), ("target", B), ("dq", 2 * B), ("dpre", 2 * B),
                    ("loss_partial", 2 * rb), ("slabs", cap), ("skinny", 3 * cdiv(B, SKINNY_ROWS) * 2 * (OBS + ACT + 1) * cdiv(max(H1, H2), 32) * 32),
                    ("scalars", 8), ("logp", B), ("next_logp", B), ("std_eps", 2 * B), ("raw_log_std", 2 * B), ("dpre4", 4 * B), ("lp_partial", rb)):
        b.take(name, n)
    return b.slots, b.o, cap


def bcq_carve(B, L, Hv, Hp, H1, H2, K=10):
    """bcq_carve() in csrc/cstr_bcq.cuh."""
    b = _Bump()
    R = B * K
    for name, n in (("e_h1", B * Hv), ("e_h2", B * Hv), ("e_y", B * 2 * L), ("std", B * L), ("eps", B * L), ("xdec", B * (4 + L)),
                    ("d_h1", B * Hv), ("d_h2", B * Hv), ("recon", B * 2), ("d_dy", B * 2), ("v_dz2", B * Hv), ("v_dz1", B * Hv), ("dzl", B * L),
                    ("e_dy", B * 2 * L), ("zc", R * L), ("c_h1", R * Hv), ("c_h2", R * Hv), ("cand", R * 2), ("p_h1", R * Hp), ("p_h2", R * Hp),
                    ("xi", R * 2), ("cand_p", R * 2), ("t_h1", 2 * R * H1), ("t_h2", 2 * R * H2), ("t_q", 2 * R), ("h1", 2 * B * H1), ("h2", 2 * B * H2),
                    ("dz1", 2 * B * H1), ("dz2", 2 * B * H2), ("target", B), ("dq", 2 * B), ("loss_partial", 2 * cdiv(B, 8)), ("za", B * L), ("a0", B * 2),
                    ("a", B * 2), ("pre", B * 2), ("da", B * 2), ("p_dy", B * 2), ("p_dz2", B * Hp), ("p_dz1", B * Hp), ("scalars", 8)):
        b.take(name, n)
    cap = _mlp_scratch(b, R, max(Hv, Hp, H1, H2, 2 * L), 2, OBS + ACT)
    return b.slots, b.o, cap


def ma_carve(B, H1, H2):
    """ma_carve() in csrc/cstr_ma.cuh."""
    b = _Bump()
    for name, n in (("a_h1", 2 * B * H1), ("a_h2", 2 * B * H2), ("a_y", 2 * B), ("next_act", 2 * B), ("t_h1", 2 * B * H1), ("t_h2", 2 * B * H2),
                    ("target", B), ("h1", 2 * B * H1), ("h2", 2 * B * H2), ("dz1", 2 * B * H1), ("dz2", 2 * B * H2), ("dq", 2 * B),
                    ("loss_partial", 2 * cdiv(B, 8)), ("joint", 2 * B), ("da", B), ("a_dy", B), ("a_dz2", B * H2), ("a_dz1", B * H1), ("scalars", 16)):
        b.take(name, n)
    cap = _mlp_scratch(b, B, max(H1, H2), 2, OBS + ACT)
    return b.slots, b.o, cap


# ---- branch mirrors of launch_gemm / choose_splits / tc_tile -------------------------------------------------------------------------
def tc_tile(N):
    """(n_tile, n_tiles, tmem_cols)"""
    n_tiles = cdiv(N, 256)
    n_tile = (cdiv(N, n_tiles) + 15) & ~15
    tmem = 32
    while tmem < n_tile:
        tmem <<= 1
    return n_tile, n_tiles, tmem


def choose_splits(B, H1, H2, Z, tc, sms):
    tiles = cdiv(H2, TC_BM) * tc_tile(H1)[1] * Z if tc else cdiv(H2, BM) * cdiv(H1, BN) * Z
    best, best_cost, s = 1, None, 1
    while s <= MAX_SPLITS and s * 32 <= B + 31:
        cost = cdiv(tiles * s, sms) * cdiv(cdiv(B, s), BK) + 2 * s
        if best_cost is None or cost < best_cost:
            best, best_cost = s, cost
        s += 1
    return best


def ffma_split(M, N, K, Z, cap, sms):
    """launch_gemm's split-K decision for an FFMA forward / dgrad: (splits, clips that bound s)."""
    s, clips, per = (2 * sms) // (cdiv(N, BN) * cdiv(M, BM) * Z), set(), Z * M * N
    if s > 8:
        s = 8
        clips.add("clip 8")
    if s > K // (2 * BK):
        s = K // (2 * BK)
        clips.add("clip K")
    if per > 0 and s > cap // per:
        s = cap // per
        clips.add("clip cap")
    if s >= 2:
        kps = cdiv(cdiv(K, s), BK) * BK
        return cdiv(K, kps), clips
    return 1, clips


def branches(notes, mode, sms):
    """The launch_gemm / choose_splits / tc_tile branches and kernel variants a list of GEMM notes reaches in one mode."""
    hit = set()
    tc = mode != "fp32"
    for n in notes:
        if n[0] == "layer1":
            hit.add(("in", n[1]))
            if n[2]:
                hit.add("periodic")
            continue
        if n[0] == "direct":
            hit.add("direct")
            continue
        role, M, N, K, Z, cap = n
        hit.add(("Z", Z))
        if M % BM:
            hit.add("M tail")
        kslab = K
        if role == "wgrad":
            s = choose_splits(K, N, M, Z, tc, sms)
            kslab = cdiv(K, s)
            hit.add("w1" if s == 1 else "w16" if s == 16 else "w2-15")
            if s > 1 and K % s:
                hit.add("ragged slabs")
            if K < 16:
                hit.add("B<16")
        if tc:
            _, n_tiles, tmem = tc_tile(N)
            hit.update({("tmem", tmem), "one tile" if n_tiles == 1 else "several tiles"})
            if N % 16:
                hit.add("N tail 16")
            if kslab % TC_KC:
                hit.add("K tail 32")
        else:
            if N % BN:
                hit.add("N tail 64")
            if kslab % BK:
                hit.add("K tail 16")
            if role != "wgrad":
                s, clips = ffma_split(M, N, K, Z, cap, sms)
                hit.add("split" if s >= 2 else "no split")
                hit.update(clips)
    return hit


COMMON = {("Z", 1), ("Z", 2), "M tail", "w1", "w2-15", "w16", "ragged slabs", "B<16", "direct", ("in", 2), ("in", 3), ("in", 4), ("in", 6),
          ("in", "4+L"), "periodic"}
REQUIRED = {"fp32": COMMON | {"no split", "split", "clip 8", "clip K", "clip cap", "N tail 64", "K tail 16"},
            "tensor": COMMON | {"one tile", "several tiles", "N tail 16", "K tail 32", ("tmem", 32), ("tmem", 64), ("tmem", 128), ("tmem", 256)}}
REQUIRED["bf16"] = REQUIRED["tensor"]


# ---- the cases, and the GEMMs each one checks ------------------------------------------------------------------------------------------
TD3_CASES = [([400, 300], 1, 2), ([400, 300], 7, 2), ([400, 300], 130, 2), ([400, 300], 256, 2), ([400, 300], 4096, 2), ([36, 20], 37, 2),
             ([4, 4], 3, 2), ([16, 16], 16, 2), ([20, 260], 641, 2), ([256, 256], 256, 2), ([512, 512], 300, 2), ([1024, 768], 64, 2),
             ([16, 16], 20000, 2), ([64, 48], 5, 2), ([32, 60], 33, 2), ([400, 300], 256, 1), ([36, 20], 37, 1), ([16, 16], 3, 1)]
SAC_CASES = [([256, 256], 256), ([36, 20], 100), ([132, 260], 641)]
BCQ_CASES = [(32, 64, 64, [400, 300], 256), (12, 700, 400, [400, 300], 100), (8, 36, 20, [36, 20], 37), (8, 32, 32, [64, 64], 100),
             (8, 32, 32, [128, 128], 64)]
MA_CASES = [([400, 300], 256, True, 2), ([400, 300], 256, False, 2), ([36, 20], 37, True, 1), ([36, 20], 37, False, 1), ([400, 300], 256, True, 1),
            ([36, 20], 37, False, 2)]


def _fwd(M, H1, H2, Z, cap):
    return ("fwd", M, H2, H1, Z, cap)


def _bwd(M, H1, H2, Z, cap, wgrad=True):
    return [("dgrad", M, H1, H2, Z, cap)] + ([("wgrad", H2, H1, M, Z, cap)] if wgrad else [])


def td3_plan(arch, B, nc):
    H1, H2 = arch
    cap = td3_carve(B, H1, H2)[2]
    crit = [("layer1", 6, False)] * (2 * nc) + [_fwd(B, H1, H2, nc, cap)] * 2 + _bwd(B, H1, H2, nc, cap)
    pol = [("layer1", 4, False), ("layer1", 6, False), _fwd(B, H1, H2, 1, cap), _fwd(B, H1, H2, 1, cap)] + _bwd(B, H1, H2, 1, cap, False) + _bwd(B, H1, H2, 1, cap)
    return [("layer1", 4, False), _fwd(B, H1, H2, 1, cap)] + crit + pol


def sac_plan(arch, B):
    H1, H2 = arch
    cap = td3_carve(B, H1, H2)[2]
    crit = [("layer1", 4, False), _fwd(B, H1, H2, 1, cap)] + [("layer1", 6, False)] * 4 + [_fwd(B, H1, H2, 2, cap)] * 2 + _bwd(B, H1, H2, 2, cap)
    act = [("layer1", 6, False)] * 2 + [_fwd(B, H1, H2, 2, cap)] + _bwd(B, H1, H2, 2, cap, False) + _bwd(B, H1, H2, 1, cap)
    return crit + act


def bcq_plan(L, Hv, Hp, arch, B):
    H1, H2 = arch
    R, cap = 10 * B, bcq_carve(B, L, Hv, Hp, H1, H2)[2]
    vae = [("layer1", 6, False), _fwd(B, Hv, Hv, 1, cap), ("layer1", "4+L", False), _fwd(B, Hv, Hv, 1, cap)] + _bwd(B, Hv, Hv, 1, cap) + [("direct",)] * 2
    cand = [("layer1", "4+L", True), _fwd(R, Hv, Hv, 1, cap), ("layer1", 6, True), _fwd(R, Hp, Hp, 1, cap)] + [("layer1", 6, True)] * 2 + [_fwd(R, H1, H2, 2, cap)]
    crit = [("layer1", 6, False)] * 2 + [_fwd(B, H1, H2, 2, cap)] + _bwd(B, H1, H2, 2, cap)
    act = [("layer1", "4+L", False), _fwd(B, Hv, Hv, 1, cap), ("layer1", 6, False), _fwd(B, Hp, Hp, 1, cap), ("layer1", 6, False), _fwd(B, H1, H2, 1, cap)]
    act += _bwd(B, H1, H2, 1, cap, False) + _bwd(B, Hp, Hp, 1, cap)
    return vae + cand + crit + act


def ma_plan(arch, B, centralised, nc):
    H1, H2 = arch
    cap, ci = ma_carve(B, H1, H2)[2], 6 if centralised else 3
    crit = [("layer1", 2, False)] * 2 + [_fwd(B, H1, H2, 2, cap)] + [("layer1", ci, False)] * (2 * nc) + [_fwd(B, H1, H2, nc, cap)] * 2 + _bwd(B, H1, H2, nc, cap)
    act = [("layer1", 2, False)] * 2 + [_fwd(B, H1, H2, 2, cap), ("layer1", ci, False), _fwd(B, H1, H2, 1, cap)] + _bwd(B, H1, H2, 1, cap, False)
    return crit + act + _bwd(B, H1, H2, 1, cap)


def all_plans():
    return ([td3_plan(a, b, nc) for a, b, nc in TD3_CASES] + [sac_plan(a, b) for a, b in SAC_CASES] + [bcq_plan(*c) for c in BCQ_CASES]
            + [ma_plan(*c) for c in MA_CASES])


# ---- CPU: the mirrors against the library ----------------------------------------------------------------------------------------------
def test_workspace_mirrors_match_the_library(pkg):
    """The slot layout the GPU tests read is the library's: the mirrors' sizes equal cstr_{td3,sac,bcq,ma}_workspace_bytes over a grid."""
    from ctypes import byref

    L = pkg._lib
    lib = L.load()
    for H1, H2 in ((4, 4), (36, 20), (400, 300), (20, 260), (1024, 768)):
        for B in (1, 7, 64, 65, 641, 4096):
            want = td3_carve(B, H1, H2)[1] * 4
            assert lib.cstr_td3_workspace_bytes(byref(L.Td3Config(h1=H1, h2=H2, batch=B, policy_delay=2, gemm_mode=0, n_critics=2))) == want
            assert lib.cstr_sac_workspace_bytes(byref(L.SacConfig(h1=H1, h2=H2, batch=B, target_update_interval=1, gemm_mode=0))) == want
            for cen, nc in ((1, 2), (0, 1)):
                cfg = L.MaConfig(centralised=cen, h1=H1, h2=H2, batch=B, policy_delay=2, n_critics=nc, gemm_mode=0)
                assert lib.cstr_ma_workspace_bytes(byref(cfg)) == ma_carve(B, H1, H2)[1] * 4
    for Lt, Hv, Hp, H1, H2 in ((32, 64, 64, 400, 300), (12, 700, 400, 400, 300), (8, 36, 20, 36, 20), (64, 8, 8, 8, 8), (4, 4, 4, 4, 4)):
        for B in (1, 37, 100, 256):
            for K in (1, 10):
                cfg = L.BcqConfig(latent=Lt, vae_hidden=Hv, pert_hidden=Hp, h1=H1, h2=H2, batch=B, actor_delay=2, n_candidates=K, gemm_mode=0)
                assert lib.cstr_bcq_workspace_bytes(byref(cfg)) == bcq_carve(B, Lt, Hv, Hp, H1, H2, K)[1] * 4


@pytest.mark.parametrize("mode", MODES)
def test_cases_reach_every_gemm_branch_on_a_b200(mode):
    """With the B200's 148 SMs, the sweep below reaches every launch_gemm / choose_splits / tc_tile branch listed in REQUIRED."""
    hit = set().union(*(branches(p, mode, B200_SMS) for p in all_plans()))
    assert REQUIRED[mode] <= hit, sorted(map(str, REQUIRED[mode] - hit))


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_cases_reach_every_gemm_branch_on_this_device(mode):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    hit = set().union(*(branches(p, mode, sms) for p in all_plans()))
    assert REQUIRED[mode] <= hit, sorted(map(str, REQUIRED[mode] - hit))


# ---- float64 references ----------------------------------------------------------------------------------------------------------------
def _bf16(x):
    """float32 -> bfloat16, round to nearest even (cvt.rn.bf16x2.f32), as float64."""
    u = np.ascontiguousarray(x, f32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(f32).astype(f64)


def _planes(x):
    """split_store's three bf16 planes by truncation: x1 = hi16(x), x2 = hi16(x - x1), x3 = hi16(x - x1 - x2) (residuals exact in fp32)."""
    x = np.ascontiguousarray(x, f32)
    hi = lambda v: (np.ascontiguousarray(v, f32).view(np.uint32) & np.uint32(0xFFFF0000)).view(f32)  # noqa: E731
    x1 = hi(x)
    r = x - x1
    x2 = hi(r)
    return x1.astype(f64), x2.astype(f64), hi(r - x2).astype(f64)


def _mma(A, Bm, mode):
    """A (M, K) @ Bm (K, N) as the kernel forms it, in float64, and sum|a*b| (the scale of the accumulation bound)."""
    A, Bm = np.asarray(A, f32), np.asarray(Bm, f32)
    absd = np.abs(A).astype(f64) @ np.abs(Bm).astype(f64)
    if mode == "fp32":
        return A.astype(f64) @ Bm.astype(f64), absd
    if mode == "bf16":
        a, b = _bf16(A), _bf16(Bm)
        return a @ b, np.abs(a) @ np.abs(b)
    a1, a2, a3 = _planes(A)
    b1, b2, b3 = _planes(Bm)
    return a1 @ (b1 + b2 + b3) + a2 @ (b1 + b2) + a3 @ b1, absd  # the six products; each partial sum of planes is exact in float64


def _acc_bound(mode, k, splits, absd):
    if mode == "fp32":
        return (k + splits + 2) * U * absd
    per_step = 6 if mode == "tensor" else 1
    return 2 * MMA_ULPS * per_step * cdiv(k, TC_KC) * ULP * absd + (splits - 1) * U * absd


def _exact_err(mode, k, absd):
    """How far the kernel's GEMM may lie from the EXACT product (not from its emulation): for the chained decoder reference."""
    if mode == "fp32":
        return (k + 10) * U * absd
    if mode == "tensor":
        return (4 * U + 12 * MMA_ULPS * cdiv(k, TC_KC) * ULP) * absd
    return (2.0 ** -8 + 2 * MMA_ULPS * cdiv(k, TC_KC) * ULP) * absd


def _skinny_depth(B):
    return 19 + cdiv(cdiv(B, SKINNY_ROWS), 4)


class Check:
    """Collects max |error| / bound per kernel output; fails at the end with every output over its bound."""

    def __init__(self, mode, sms, name):
        self.mode, self.sms, self.name = mode, sms, name
        self.ratio = collections.OrderedDict()
        self.notes = []

    def put(self, label, got, ref, bound):
        got = np.asarray(got, f64)
        assert got.shape == ref.shape, (label, got.shape, ref.shape)
        d = np.abs(got - ref)
        r = np.where(bound > 0, d / np.where(bound > 0, bound, 1.0), np.where(d > 0, np.inf, 0.0))
        self.ratio[label] = max(self.ratio.get(label, 0.0), float(r.max()) if r.size else 0.0)

    def layer1(self, label, x, W1, b1, got, periodic=False, width=None):
        self.notes.append(("layer1", width or x.shape[1], periodic))
        x, W1, b1 = np.asarray(x, f64), np.asarray(W1, f64), np.asarray(b1, f64)
        self.put(label, got, np.maximum(x @ W1.T + b1, 0.0), (x.shape[1] + 2) * U * (np.abs(x) @ np.abs(W1).T + np.abs(b1)))

    def fwd(self, label, h1, nets, got, cap):
        """FWD: h2[z] = relu(h1[z] @ W2[z]^T + b2[z]) for one Z-batched launch."""
        Z, M, K = h1.shape
        N = nets[0][2].shape[0]
        self.notes.append(("fwd", M, N, K, Z, cap))
        s = ffma_split(M, N, K, Z, cap, self.sms)[0] if self.mode == "fp32" else 1
        for z in range(Z):
            v, absd = _mma(h1[z], nets[z][2].T, self.mode)
            b = np.asarray(nets[z][3], f64)
            e = _acc_bound(self.mode, K, s, absd + np.abs(b)) + (0 if self.mode == "fp32" else U * (absd + np.abs(b)))
            self.put(f"{label}[{z}]", got[z], np.maximum(v + b, 0.0), e)

    def dgrad(self, label, dz2, nets, h1, got, cap):
        """DGRAD: dz1[z] = (dz2[z] @ W2[z]) * (h1[z] > 0)."""
        Z, M, K = dz2.shape
        N = nets[0][2].shape[1]
        self.notes.append(("dgrad", M, N, K, Z, cap))
        s = ffma_split(M, N, K, Z, cap, self.sms)[0] if self.mode == "fp32" else 1
        for z in range(Z):
            v, absd = _mma(dz2[z], nets[z][2], self.mode)
            self.put(f"{label}[{z}]", got[z], np.where(h1[z] > 0, v, 0.0), np.where(h1[z] > 0, _acc_bound(self.mode, K, s, absd), 0.0))

    def wgrad(self, label, dz2, h1, got, cap):
        """WGRAD: dW2[z] = dz2[z]^T @ h1[z], split over the batch into slabs that td3_finalize_kernel sums."""
        Z, K, M = dz2.shape
        N = h1.shape[2]
        self.notes.append(("wgrad", M, N, K, Z, cap))
        s = choose_splits(K, N, M, Z, self.mode != "fp32", self.sms)
        for z in range(Z):
            v, absd = _mma(dz2[z].T, h1[z], self.mode)
            self.put(f"{label}[{z}]", got[z], v, _acc_bound(self.mode, cdiv(K, s), s, absd))

    def direct(self, label, A, Bm, got):
        """wgrad_gemm_direct: C = A^T @ Bm over the batch, FFMA in every mode, one split."""
        self.notes.append(("direct",))
        v, absd = _mma(np.asarray(A).T, Bm, "fp32")
        self.put(label, got, v, (A.shape[0] + 3) * U * absd)

    def skinny(self, label, X, Y, got):
        """td3_skinny_wgrad_kernel + its finalize job: X^T @ Y, or the column sum of X when Y is None."""
        X = np.asarray(X, f64)
        Y = np.ones((X.shape[0], 1)) if Y is None else np.asarray(Y, f64).reshape(X.shape[0], -1)
        v = X.T @ Y
        e = _skinny_depth(X.shape[0]) * U * (np.abs(X).T @ np.abs(Y))
        self.put(label, np.asarray(got, f64).reshape(v.shape), v, e)

    def head_bwd(self, label, dy, W3, h2, got):
        """dz2 = (dy @ W3) * (h2 > 0): the critic head (one output: one rounding), the actor backward heads, mlp_head_bwd_kernel."""
        dy, W3 = np.asarray(dy, f64).reshape(h2.shape[0], -1), np.asarray(W3, f64)
        v = dy @ W3
        e = (dy.shape[1] + 1) * U * (np.abs(dy) @ np.abs(W3))
        self.put(label, got, np.where(h2 > 0, v, 0.0), np.where(h2 > 0, e, 0.0))

    def net_grads(self, label, g, x, dz1, dz2, hx, hy, w1=True):
        """The skinny gradients of one net: db2, dW1 (when x is narrow), db1, dW3 = hy^T hx, db3."""
        self.skinny(f"{label}.db2", dz2, None, g[3])
        if w1:
            self.skinny(f"{label}.dW1", dz1, x, g[0])
        self.skinny(f"{label}.db1", dz1, None, g[1])
        self.skinny(f"{label}.dW3", hx, hy, g[4].T)
        self.skinny(f"{label}.db3", hy, None, g[5])

    def finish(self, plan):
        for k, v in self.ratio.items():
            print(f"{self.name:44s} {k:28s} {v:.3g}")
        assert collections.Counter(self.notes) == collections.Counter(plan), "the checks and the coverage plan disagree"
        bad = {k: v for k, v in self.ratio.items() if not v <= 1.0}
        assert not bad, f"{self.name}: outputs over their bound (error / bound): {bad}"


# ---- engine plumbing ---------------------------------------------------------------------------------------------------------------------
def _np_views(eng, block):
    return {k: [t.cpu().numpy() for t in v] for k, v in eng.views(block).items()}


class _Ws:
    def __init__(self, flat, slots):
        self.flat, self.slots = flat, slots

    def __call__(self, name, *shape, skip=0):
        o = self.slots[name] + skip
        return self.flat[o:o + int(np.prod(shape))].reshape(shape).astype(f32)


def _frozen_update(eng, run):
    """Run one update and assert that learning rate 0 / tau 0 left params and targets bit-identical."""
    p0, t0 = eng.params.clone(), eng.targets.clone()
    run()
    torch.cuda.synchronize()
    assert torch.equal(eng.params, p0) and torch.equal(eng.targets, t0), "learning rate 0 / tau 0 changed the weights"
    return eng._workspace.cpu().numpy()


def _batch(rng, B):
    return (rng.uniform(-1, 1, (B, 4)).astype(f32), rng.uniform(-1, 1, (B, 2)).astype(f32), rng.uniform(-1, 1, (B, 4)).astype(f32),
            (rng.random((B, 1)) < 0.1).astype(f32), rng.normal(size=(B, 1)).astype(f32))


def _mlp(rng, i, h1, h2, o):
    out = []
    for fi, fo in ((i, h1), (h1, h2), (h2, o)):
        b = 1.0 / np.sqrt(fi)
        out += [rng.uniform(-b, b, (fo, fi)).astype(f32), rng.uniform(-b, b, fo).astype(f32)]
    return out


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _critic_phase(chk, ws, tag, x, xt, critics, t_nets, B, H1, H2, nz, G, cap, grads=True):
    """Target critics on xt, critics on x, their head and backward: the critic step every engine shares (slots t_h*, h*, dq, dz*)."""
    t_h1, t_h2 = ws("t_h1", nz, B, H1), ws("t_h2", nz, B, H2)
    for z in range(nz):
        chk.layer1(f"{tag}t.h1[{z}]", xt, t_nets[z][0], t_nets[z][1], t_h1[z])
    chk.fwd(f"{tag}t.h2", t_h1, t_nets, t_h2, cap)
    h1, h2, dz1, dz2, dq = ws("h1", nz, B, H1), ws("h2", nz, B, H2), ws("dz1", nz, B, H1), ws("dz2", nz, B, H2), ws("dq", nz, B)
    for z in range(nz):
        chk.layer1(f"{tag}.h1[{z}]", x, critics[z][0], critics[z][1], h1[z])
    chk.fwd(f"{tag}.h2", h1, critics, h2, cap)
    for z in range(nz):
        chk.head_bwd(f"{tag}.dz2[{z}]", dq[z], critics[z][4], h2[z], dz2[z])
    chk.dgrad(f"{tag}.dz1", dz2, critics, h1, dz1, cap)
    if grads:
        chk.wgrad(f"{tag}.dW2", dz2, h1, np.stack([g[2] for g in G]), cap)
        for z in range(nz):
            chk.net_grads(f"{tag}[{z}]", G[z], x, dz1[z], dz2[z], h2[z], dq[z])


def _policy_eval(chk, ws, tag, x, critic, B, H1, H2, cap):
    """Critic 0 on the policy's actions (slab 0 of h*, dz*) and its backward to dz1 (no weight gradients)."""
    h1, h2, dz1, dz2, dq = ws("h1", 1, B, H1), ws("h2", 1, B, H2), ws("dz1", 1, B, H1), ws("dz2", 1, B, H2), ws("dq", B)
    chk.layer1(f"{tag}.h1", x, critic[0], critic[1], h1[0])
    chk.fwd(f"{tag}.h2", h1, [critic], h2, cap)
    chk.head_bwd(f"{tag}.dz2", dq, critic[4], h2[0], dz2[0])
    chk.dgrad(f"{tag}.dz1", dz2, [critic], h1, dz1, cap)


def _net_backward(chk, tag, x, net, g, h1, h2, dy, dz2, dz1, cap):
    """One net's backward from its head: dz2, dz1, dW2 and the skinny gradients."""
    chk.head_bwd(f"{tag}.dz2", dy, net[4], h2, dz2)
    chk.dgrad(f"{tag}.dz1", dz2[None], [net], h1[None], dz1[None], cap)
    chk.wgrad(f"{tag}.dW2", dz2[None], h1[None], g[2][None], cap)
    chk.net_grads(tag, g, x, dz1, dz2, h2, dy)


# ---- GPU: TD3 / DDPG ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("arch,B,nc", TD3_CASES, ids=[f"{a[0]}x{a[1]}-B{b}-nc{n}" for a, b, n in TD3_CASES])
def test_td3_gemms_vs_float64(pkg, arch, B, nc, mode):
    H1, H2 = arch
    slots, _, cap = td3_carve(B, H1, H2)
    chk = Check(mode, _sms(), f"td3 {H1}x{H2} B{B} nc{nc} {mode}")
    for delay in (2, 1):
        rng = np.random.default_rng(B * 7 + H1 + delay)
        nets = TU.random_nets(rng, H1, H2)
        eng = pkg.FusedTD3Update(arch, B, gemm=mode, policy_delay=delay, learning_rate=0.0, tau=0.0, n_critics=nc)
        eng.load_nets(nets)
        obs, act, nobs, dones, rew = batch = _batch(rng, B)
        noise = rng.normal(0, 0.2, (B, 2)).astype(f32)
        ws = _Ws(_frozen_update(eng, lambda: eng.update(batch, noise=noise)), slots)
        P, G = _np_views(eng, "params"), _np_views(eng, "grads")
        actor, critics = P["actor"], [P["critic0"], P["critic1"]][:nc]
        a_h1, a_h2 = ws("a_h1", 1, B, H1), ws("a_h2", 1, B, H2)
        if delay == 2:  # critic-only step: the target actor, the target critics, the critics and their gradients
            chk.layer1("actor_t.h1", nobs, actor[0], actor[1], a_h1[0])
            chk.fwd("actor_t.h2", a_h1, [actor], a_h2, cap)
            xt = np.concatenate([nobs, ws("next_act", B, 2)], 1)
            _critic_phase(chk, ws, "critic", np.concatenate([obs, act], 1), xt, critics, critics, B, H1, H2, nc,
                          [G["critic0"], G["critic1"]][:nc], cap)
        else:  # policy step: the actor on obs, critic 0 on its actions, the backward into the actor and its gradients
            chk.layer1("actor.h1", obs, actor[0], actor[1], a_h1[0])
            chk.fwd("actor.h2", a_h1, [actor], a_h2, cap)
            _policy_eval(chk, ws, "critic0.pi", np.concatenate([obs, ws("a_pi", B, 2)], 1), critics[0], B, H1, H2, cap)
            _net_backward(chk, "actor", obs, actor, G["actor"], a_h1[0], a_h2[0], ws("dpre", B, 2), ws("dz2", B, H2, skip=B * H2),
                          ws("dz1", B, H1, skip=B * H1), cap)
    chk.finish(td3_plan(arch, B, nc))


# ---- GPU: SAC ----------------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("arch,B", SAC_CASES, ids=[f"{a[0]}x{a[1]}-B{b}" for a, b in SAC_CASES])
def test_sac_gemms_vs_float64(pkg, arch, B, mode):
    H1, H2 = arch
    slots, _, cap = td3_carve(B, H1, H2)
    chk = Check(mode, _sms(), f"sac {H1}x{H2} B{B} {mode}")
    rng = np.random.default_rng(B + H1)
    eng = pkg.FusedSACUpdate(arch, B, gemm=mode, learning_rate=0.0, tau=0.0)
    eng.load_nets(TU.random_sac_nets(rng, H1, H2))
    obs, act, nobs, dones, rew = batch = _batch(rng, B)
    e1, e2 = rng.normal(size=(B, 2)).astype(f32), rng.normal(size=(B, 2)).astype(f32)
    snap = []

    def hook(flat):  # between the critic and the actor phase: the critic-phase slots before the actor phase reuses them
        if not snap:
            torch.cuda.synchronize()
            snap.append(eng._workspace.cpu().numpy())

    end = _Ws(_frozen_update(eng, lambda: eng.update(batch, eps_pi=e1, eps_next=e2, allreduce=hook)), slots)
    ws = _Ws(snap[0], slots)
    P, G = _np_views(eng, "params"), _np_views(eng, "grads")
    actor, critics = P["actor"], [P["critic0"], P["critic1"]]
    a_h1, a_h2 = ws("a_h1", 1, B, H1), ws("a_h2", 1, B, H2)
    chk.layer1("actor.h1", obs, actor[0], actor[1], a_h1[0])
    chk.fwd("actor.h2", a_h1, [actor], a_h2, cap)
    xt = np.concatenate([nobs, ws("next_act", B, 2)], 1)
    _critic_phase(chk, ws, "critic", np.concatenate([obs, act], 1), xt, critics, critics, B, H1, H2, 2, [G["critic0"], G["critic1"]], cap)
    # actor phase: both critics on (obs, a_pi), the min-q head's dz2, then the backward into the actor (its dz2 / dz1 in t_h2 / t_h1)
    x = np.concatenate([obs, end("a_pi", B, 2)], 1)
    h1, h2, dz1, dz2 = end("h1", 2, B, H1), end("h2", 2, B, H2), end("dz1", 2, B, H1), end("dz2", 2, B, H2)
    for z in range(2):
        chk.layer1(f"critic.pi.h1[{z}]", x, critics[z][0], critics[z][1], h1[z])
    chk.fwd("critic.pi.h2", h1, critics, h2, cap)
    chk.dgrad("critic.pi.dz1", dz2, critics, h1, dz1, cap)
    _net_backward(chk, "actor", obs, actor, G["actor"], end("a_h1", B, H1), end("a_h2", B, H2), end("dpre4", B, 4), end("t_h2", B, H2),
                  end("t_h1", B, H1), cap)
    chk.finish(sac_plan(arch, B))


# ---- GPU: BCQ ----------------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("L,Hv,Hp,arch,B", BCQ_CASES, ids=[f"L{c[0]}-{c[1]}-{c[2]}-{c[3][0]}x{c[3][1]}-B{c[4]}" for c in BCQ_CASES])
def test_bcq_gemms_vs_float64(pkg, L, Hv, Hp, arch, B, mode):
    H1, H2 = arch
    R = 10 * B
    slots, _, cap = bcq_carve(B, L, Hv, Hp, H1, H2)
    chk = Check(mode, _sms(), f"bcq L{L} {Hv}/{Hp} {H1}x{H2} B{B} {mode}")
    for delay in (2, 1):
        rng = np.random.default_rng(L + B + delay)
        nets = {"vae_enc": _mlp(rng, 6, Hv, Hv, 2 * L), "vae_dec": _mlp(rng, 4 + L, Hv, Hv, 2), "pert": _mlp(rng, 6, Hp, Hp, 2),
                "critic0": _mlp(rng, 6, H1, H2, 1), "critic1": _mlp(rng, 6, H1, H2, 1)}
        eng = pkg.FusedBCQUpdate(L, Hv, Hp, arch, B, gemm=mode, actor_delay=delay, learning_rate=0.0, tau=0.0)
        eng.load_nets(nets)
        obs, act, nobs, dones, rew = batch = _batch(rng, B)
        eps, zn, za = rng.normal(size=(B, L)).astype(f32), rng.normal(size=(R, L)).astype(f32), rng.normal(size=(B, L)).astype(f32)
        ws = _Ws(_frozen_update(eng, lambda: eng.update(batch, eps_vae=eps, z_next=zn, z_actor=za)), slots)
        P, G = _np_views(eng, "params"), _np_views(eng, "grads")
        enc, dec, pert, critics = P["vae_enc"], P["vae_dec"], P["pert"], [P["critic0"], P["critic1"]]
        if delay == 2:
            # VAE: encoder forward, decoder forward on [obs | z], the encoder's backward (its wide head through wgrad_gemm_direct)
            x = np.concatenate([obs, act], 1)
            e_h1, e_h2 = ws("e_h1", 1, B, Hv), ws("e_h2", 1, B, Hv)
            chk.layer1("enc.h1", x, enc[0], enc[1], e_h1[0])
            chk.fwd("enc.h2", e_h1, [enc], e_h2, cap)
            xdec = ws("xdec", B, 4 + L)
            d_h1, d_h2 = ws("d_h1", 1, B, Hv), ws("d_h2", 1, B, Hv)
            chk.layer1("dec.h1", xdec, dec[0], dec[1], d_h1[0], width="4+L")
            chk.fwd("dec.h2", d_h1, [dec], d_h2, cap)
            e_dy, v_dz2, v_dz1, ge = ws("e_dy", B, 2 * L), ws("v_dz2", B, Hv), ws("v_dz1", B, Hv), G["vae_enc"]
            chk.head_bwd("enc.dz2", e_dy, enc[4], e_h2[0], v_dz2)
            chk.dgrad("enc.dz1", v_dz2[None], [enc], e_h1, v_dz1[None], cap)
            chk.wgrad("enc.dW2", v_dz2[None], e_h1, ge[2][None], cap)
            chk.direct("enc.dW3", e_dy, e_h2[0], ge[4])
            chk.net_grads("enc", ge, x, v_dz1, v_dz2, e_h2[0], e_dy)
            # the decoder's layer-1 gradient over the 4 + L wide input: its dz1 was overwritten, so the reference is the float64 chain
            d_dy, W3, W2 = ws("d_dy", B, 2).astype(f64), dec[4].astype(f64), dec[2].astype(f64)
            m2, m1 = d_h2[0] > 0, d_h1[0] > 0
            dz2 = np.where(m2, d_dy @ W3, 0.0)
            e2 = np.where(m2, 3 * U * (np.abs(d_dy) @ np.abs(W3)), 0.0)
            dz1 = np.where(m1, dz2 @ W2, 0.0)
            e1 = np.where(m1, e2 @ np.abs(W2) + _exact_err(mode, Hv, (np.abs(dz2) + e2) @ np.abs(W2)), 0.0)
            xa = np.abs(xdec.astype(f64))
            chk.notes.append(("direct",))
            chk.put("dec.dW1 (chain)", G["vae_dec"][0], dz1.T @ xdec, e1.T @ xa + (B + 3) * U * ((np.abs(dz1) + e1).T @ xa))
            chk.put("dec.db1 (chain)", G["vae_dec"][1], dz1.sum(0), e1.sum(0) + _skinny_depth(B) * U * (np.abs(dz1) + e1).sum(0))
            # candidates: R = 10 B rows whose state part repeats next_obs with period B
            nrep = np.tile(nobs, (10, 1))
            c_h1, c_h2 = ws("c_h1", 1, R, Hv), ws("c_h2", 1, R, Hv)
            chk.layer1("cand.dec.h1", np.concatenate([nrep, ws("zc", R, L)], 1), dec[0], dec[1], c_h1[0], periodic=True, width="4+L")
            chk.fwd("cand.dec.h2", c_h1, [dec], c_h2, cap)
            p_h1, p_h2 = ws("p_h1", 1, R, Hp), ws("p_h2", 1, R, Hp)
            chk.layer1("cand.pert.h1", np.concatenate([nrep, ws("cand", R, 2)], 1), pert[0], pert[1], p_h1[0], periodic=True)
            chk.fwd("cand.pert.h2", p_h1, [pert], p_h2, cap)
            xq = np.concatenate([nrep, ws("cand_p", R, 2)], 1)
            t_h1, t_h2 = ws("t_h1", 2, R, H1), ws("t_h2", 2, R, H2)
            for z in range(2):
                chk.layer1(f"cand.critic_t.h1[{z}]", xq, critics[z][0], critics[z][1], t_h1[z], periodic=True)
            chk.fwd("cand.critic_t.h2", t_h1, critics, t_h2, cap)
            # critics: TD3's twin-critic step (their target-critic slots hold the candidates, checked above)
            x = np.concatenate([obs, act], 1)
            h1, h2, dz1, dz2, dq = ws("h1", 2, B, H1), ws("h2", 2, B, H2), ws("dz1", 2, B, H1), ws("dz2", 2, B, H2), ws("dq", 2, B)
            for z in range(2):
                chk.layer1(f"critic.h1[{z}]", x, critics[z][0], critics[z][1], h1[z])
                chk.head_bwd(f"critic.dz2[{z}]", dq[z], critics[z][4], h2[z], dz2[z])
            chk.fwd("critic.h2", h1, critics, h2, cap)
            chk.dgrad("critic.dz1", dz2, critics, h1, dz1, cap)
            chk.wgrad("critic.dW2", dz2, h1, np.stack([G["critic0"][2], G["critic1"][2]]), cap)
            for z in range(2):
                chk.net_grads(f"critic[{z}]", G[f"critic{z}"], x, dz1[z], dz2[z], h2[z], dq[z])
        else:  # the perturbation step: decoder on [obs | z], perturbation net, critic 0 on the perturbed action, the backward into pert
            d_h1, d_h2 = ws("d_h1", 1, B, Hv), ws("d_h2", 1, B, Hv)
            chk.layer1("actor.dec.h1", np.concatenate([obs, ws("za", B, L)], 1), dec[0], dec[1], d_h1[0], width="4+L")
            chk.fwd("actor.dec.h2", d_h1, [dec], d_h2, cap)
            xp = np.concatenate([obs, ws("a0", B, 2)], 1)
            p_h1, p_h2 = ws("p_h1", 1, B, Hp), ws("p_h2", 1, B, Hp)
            chk.layer1("pert.h1", xp, pert[0], pert[1], p_h1[0])
            chk.fwd("pert.h2", p_h1, [pert], p_h2, cap)
            _policy_eval(chk, ws, "critic0.pi", np.concatenate([obs, ws("a", B, 2)], 1), critics[0], B, H1, H2, cap)
            _net_backward(chk, "pert", xp, pert, G["pert"], p_h1[0], p_h2[0], ws("p_dy", B, 2), ws("p_dz2", B, Hp), ws("p_dz1", B, Hp), cap)
    chk.finish(bcq_plan(L, Hv, Hp, arch, B))


# ---- GPU: MADDPG / IDDPG -------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("arch,B,centralised,nc", MA_CASES, ids=[f"{a[0]}x{a[1]}-B{b}-{'ma' if c else 'i'}ddpg-nc{n}" for a, b, c, n in MA_CASES])
def test_multiagent_gemms_vs_float64(pkg, arch, B, centralised, nc, mode):
    """Agent 1's phases are the last of the step, so its slots are the ones the workspace holds."""
    H1, H2 = arch
    slots, _, cap = ma_carve(B, H1, H2)
    chk = Check(mode, _sms(), f"{'ma' if centralised else 'i'}ddpg {H1}x{H2} B{B} nc{nc} {mode}")
    ci = 6 if centralised else 3

    def src(X, A):  # agent 1's critic input
        return np.concatenate([X, A], 1) if centralised else np.concatenate([X[:, 2:4], A[:, 1:2]], 1)

    for delay in (2, 1):
        rng = np.random.default_rng(B + H1 + delay + 10 * centralised)
        names = [f"actor{i}" for i in range(2)] + [f"critic{i}_{k}" for i in range(2) for k in range(nc)]
        nets = {n: _mlp(rng, 2, H1, H2, 1) if n.startswith("actor") else _mlp(rng, ci, H1, H2, 1) for n in names}
        eng = pkg.FusedMultiAgentUpdate(arch, B, centralised, gemm=mode, policy_delay=delay, actor_lrs=[0.0, 0.0], critic_lrs=[0.0, 0.0], tau=0.0,
                                        n_critics=nc)
        eng.load_nets(nets)
        obs, act, nobs, dones, rew = batch = _batch(rng, B)
        noise = rng.normal(0, 0.2, (2, B)).astype(f32)
        ws = _Ws(_frozen_update(eng, lambda: eng.update(batch, noise=noise)), slots)
        P, G = _np_views(eng, "params"), _np_views(eng, "grads")
        actors, critics = [P["actor0"], P["actor1"]], [P[f"critic1_{k}"] for k in range(nc)]
        a_h1, a_h2 = ws("a_h1", 2, B, H1), ws("a_h2", 2, B, H2)
        if delay == 2:  # target actors (actor z on observation slice z), then agent 1's critic step
            for z in range(2):
                chk.layer1(f"actor_t.h1[{z}]", nobs[:, 2 * z:2 * z + 2], actors[z][0], actors[z][1], a_h1[z])
            chk.fwd("actor_t.h2", a_h1, actors, a_h2, cap)
            _critic_phase(chk, ws, "critic1", src(obs, act), src(nobs, ws("next_act", B, 2)), critics, critics, B, H1, H2, nc,
                          [G[f"critic1_{k}"] for k in range(nc)], cap)
        else:  # agent 1's actor step: every actor on agent 1's slice, critic (1, 0) on the joint action, the backward into actor 1
            x = obs[:, 2:4]
            for z in range(2):
                chk.layer1(f"actors.h1[{z}]", x, actors[z][0], actors[z][1], a_h1[z])
            chk.fwd("actors.h2", a_h1, actors, a_h2, cap)
            _policy_eval(chk, ws, "critic1_0.pi", src(obs, ws("joint", B, 2)), critics[0], B, H1, H2, cap)
            _net_backward(chk, "actor1", x, actors[1], G["actor1"], a_h1[1], a_h2[1], ws("a_dy", B, 1), ws("a_dz2", B, H2), ws("a_dz1", B, H1), cap)
    chk.finish(ma_plan(arch, B, centralised, nc))
