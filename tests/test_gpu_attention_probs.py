"""Relative-position attention checked probability by probability against float64.

The other attention tests compare the context P V for random V under a norm tolerance, which averages an error in one
key over the row and an error in one row over the tensor.  Here the operands are chosen so that the kernels compute
every score exactly, and V is one-hot, so that each element of the context is one probability P[b, h, i, j]:

  * q + u, q + v, k and the positional rows p are integers in {-1, 0, 1} (pad columns dk..dkp-1 zero), except for the
    fixed query component and the poisoned / spiked key rows below, which are integers <= 256;
  * head h of launch r gets v[j] = e_c for the keys j = (w_rh + c) mod T, c < dk, and v = 0 elsewhere, so that
    ctx[b, i, h, c] = P[b, h, i, (w_rh + c) mod T].  The windows of the heads are spread over the keys and move by dk
    per launch; ceil(T / dk) launches show every head every key.

Every probed element is compared with the float64 probability; masked keys and padded query rows must be exact zeros.

Why the bound is relative 2^-7 (tensor-core kernels; line numbers in conformer-nemo_b200/csrc):
  1. Content term: bf16 x bf16 products of integers <= 256 summed into fp32 (attention_tc.cu:249,
     attention_tc128.cu:275) -- exact.
  2. Position term: (q + v) / 16 becomes fp16 (attention_tc.cu:321-326, attention_tcp.cu:405-410,
     attention_tc128.cu:337-339) and p becomes fp16 (attn_pos_f16, attention_tc.cu:509-523; elementwise.cu:553-554)
     -- exact for these values.  The G MMA accumulates in fp16 (attention_common.cuh:57-61, attention_tc.cu:267,302):
     for valid rows it only holds multiples of 2^-4 of magnitude <= dk / 16 <= 8 -- exact.  s + 16 g is one
     fma.rn.f32.f16 (ptx.cuh:296-300; attention_tc.cu:389-393) -- exact.
  3. Masked keys are -inf before the maximum (attention_tc.cu:395-399), so ex2 gives exact zeros for them.
  4. The exponent fma(s, scale, -fl(m scale)) (attention_tc.cu:409,418; attention_tcp.cu:503,509;
     attention_tc128.cu:417,424; ptx.cuh:275-283) and ex2.approx.ftz (attention_common.cuh:14-18) have fp32 errors
     only: scale_log2 is log2(e)/sqrt(dk) rounded to fp32 (attention_tc.cu:577), a relative error of at most 3 2^-24
     of the exponent, i.e. below 2^-19 of P while the exponents of a row span less than 20 nats; ex2.approx is within
     about 2^-22.
  5. P rounded to bf16, round half up (attention_tc.cu:422, attention_tcp.cu:511, attention_tc128.cu:427): relative
     error <= u / (1 + u), u = 2^-8.
  6. P V with one-hot V adds one non-zero product into fp32 (attention_tc.cu:259) -- exact.  The rescales by alpha
     (attention_tc.cu:410,447-451; attention_tcp.cu:504,533-534; attention_tc128.cu:418,451-455), the normaliser l,
     summed in fp32 from the unrounded exponentials (attention_tc.cu:429, attention_tcp.cu:517,
     attention_tc128.cu:431), and the set merge (attention_tc.cu:476-479, attention_tcp.cu:569-572; tc128 has one set,
     :463) are fp32: a few 2^-24 roundings per key tile and softmax set.
  7. ctx rounded to bf16, round to nearest (attention_tc.cu:486-489, attention_tcp.cu:579-582,
     attention_tc128.cu:470-472; ptx.cuh:361-364): relative error <= u / (1 + u).
Two bf16 roundings compose to at most 2u - u^2 (+ O(u^3)) = 2^-7 - 2^-16.  Steps 4 and 6 add about 2^-18 at
T <= 1100; at T = 7500 (59 key tiles per set) they reach the u^2 = 2^-16 of slack only if every one of them rounds
the same way.  Hence |got - P| <= 2^-7 P.  The absolute floor 2^-40 is far below the smallest probability of any case
(the check asserts a factor 2^10), so it never hides a relative error.  The fp32 CUDA-core kernel (attention_simt.cu:56-80:
exact fp32 dot products of integers, one division by fl(sqrt(dk)), expf, an fp32 sum of at most T terms, one
multiplication) stays far inside 1e-5 for T <= 1100.

Shifting a key by one position changes its score by about one nat (the entries' spread), i.e. its probability by
far more than 2^-7.  test_checker_rejects_injected_defects shows on the CPU that the checker fails for the defects a
norm test misses, and test_checker_accepts_kernel_rounding that it passes the float64 reference rounded the way the
kernels round."""
import math

import pytest
import torch

from gpu_util import op_attention
from test_gpu_attention import torch_reference

BN = 64  # keys per tile of the tensor-core kernels
REL_TC = 2.0 ** -7
REL_SIMT = 1e-5
FLOOR = 2.0 ** -40
POISON_KEY, POISON_QUERY = 256.0, 64.0

# kernel name -> (tensor cores, padded head width, CFB_ATTN_PERSIST).  dkp 128 always runs attention_tc128.cu.
KERNELS = {
    "tc": (True, 64, "0"),      # attention_tc.cu, one CTA per (query tile, head, sequence)
    "tcp": (True, 64, "1"),     # attention_tcp.cu, persistent
    "tc128": (True, 128, None),  # attention_tc128.cu
    "simt64": (False, 64, None),  # attention_simt.cu
    "simt128": (False, 128, None),
}
KERNEL_SYMBOL = {"tc": "rel_attn_tc_kernel", "tcp": "rel_attn_tcp_kernel", "tc128": "rel_attn_tc128_kernel",
                 "simt64": "rel_attn_simt_kernel", "simt128": "rel_attn_simt_kernel"}
DK_FOR = {64: [16, 44, 64], 128: [66, 96, 128]}
MODES = ["content", "position", "both"]
T_GRID = [1, 2, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257, 383, 384, 385, 512, 513, 700, 1100]


# ------------------------------------------------------------------------------------------------------ inputs
def lengths_for(T, seed):
    """T, T-1, 0, 1 and the tile edges 63/64/65, 127/128/129 that fit, and one random length."""
    lens = []
    for n in (T, T - 1, 0, 1, 63, 64, 65, 127, 128, 129):
        if 0 <= n <= T and n not in lens:
            lens.append(n)
    lens.append(int(torch.randint(0, T + 1, (1,), generator=torch.Generator().manual_seed(seed))))
    return lens


def make_inputs(B, T, H, dk, lens, mode, seed, spikes=()):
    """float64 CPU tensors q+u, q+v, k (B, H, T, dk) and p (H, 2T-1, dk) with entries in {-1, 0, 1}; qu = 0 in the
    position mode, qv = 0 in the content mode.  Valid queries have qu[.., 0] = 1 wherever the content term is used.
    Poisoned padding: key rows j >= len are (256, 0, ...), which would swamp every valid probability if they leaked
    into the maximum, the normaliser or P V; query rows i >= len hold +-64.  spikes: (b, j) keys whose fixed component
    is round(12 sqrt(dk)), 12 nats above the other scores of every valid query."""
    g = torch.Generator().manual_seed(seed)

    def tern(*shape):
        return torch.randint(-1, 2, shape, generator=g).double()

    qu, qv, k, p = tern(B, H, T, dk), tern(B, H, T, dk), tern(B, H, T, dk), tern(H, 2 * T - 1, dk)
    if mode == "position":
        qu.zero_()
    else:
        qu[..., 0] = 1.0
    if mode == "content":
        qv.zero_()
    pad = (torch.arange(T)[None] >= torch.tensor(lens)[:, None])[:, None, :, None]
    qu = torch.where(pad, POISON_QUERY * tern(B, H, T, dk), qu)
    qv = torch.where(pad, POISON_QUERY * tern(B, H, T, dk), qv)
    poison = torch.zeros(dk, dtype=torch.float64)
    poison[0] = POISON_KEY
    k = torch.where(pad, poison, k)
    for b, j in spikes:
        k[b, :, j, 0] = float(round(12 * math.sqrt(dk)))
    return qu, qv, k, p


def scores(qu, qv, k, p, i0, i1, shift=None):
    """float64 scores (B, H, i1-i0, T) of query rows i0..i1-1, the position term indexed directly as p[T-1+j-i].
    shift (for the checker's self-test only): a (i1-i0,) offset added to that index."""
    B, H, T, dk = qu.shape
    i = torch.arange(i0, i1, device=qu.device)
    j = torch.arange(T, device=qu.device)
    idx = T - 1 + j[None, :] - i[:, None]
    if shift is not None:
        idx = (idx + shift[:, None]).clamp(0, 2 * T - 2)
    ac = qu[:, :, i0:i1] @ k.transpose(-1, -2)
    bd = (qv[:, :, i0:i1] @ p.transpose(-1, -2)).gather(-1, idx.expand(B, H, -1, -1))
    return (ac + bd) / math.sqrt(dk)


def masked(s, lens):
    """scores with keys j >= len at -inf (the rows of padded queries are left as they are)"""
    T = s.shape[-1]
    return s.masked_fill(torch.arange(T, device=s.device) >= lens.to(s.device)[:, None, None, None], float("-inf"))


def softmax_rows(s, lens, i0):
    """masked softmax; query rows i >= len are zero (multi_head_attention.py:104-113)"""
    P = torch.softmax(masked(s, lens), -1)
    i = torch.arange(i0, i0 + s.shape[2], device=s.device)
    valid = (i[None, :] < lens.to(s.device)[:, None])[:, None, :, None]
    return torch.where(valid, P, torch.zeros((), dtype=P.dtype, device=P.device))


def ref_probs(qu, qv, k, p, lens, i0, i1):
    return softmax_rows(scores(qu, qv, k, p, i0, i1), lens, i0)


def pack(qu, qv, k, p, dkp, dtype):
    """Device buffers in the layout cfb_op_rel_attention reads: qkv (B T, 4 H dkp) = [q+u | q+v | k | v] (v left zero),
    pos (2T-1, H dkp) a view into a buffer twice as wide whose first half is a poison value."""
    B, H, T, dk = qu.shape
    Dp = H * dkp
    qkv = torch.zeros(B * T, 4, H, dkp, dtype=dtype, device="cuda")
    for n, t in enumerate((qu, qv, k)):
        qkv[:, n, :, :dk] = t.cuda().permute(0, 2, 1, 3).reshape(B * T, H, dk).to(dtype)
    pos = torch.full((2 * T - 1, 2, H, dkp), 7.0, dtype=dtype, device="cuda")
    pos[:, 1] = 0
    pos[:, 1, :, :dk] = p.cuda().permute(1, 0, 2).to(dtype)
    return qkv.view(B * T, 4 * Dp), pos.view(2 * T - 1, 2 * Dp)[:, Dp:]


# ------------------------------------------------------------------------------------------------------ probes
def probe_keys(T, H, dk, r):
    """(H, dk): the key whose probability ctx column c of head h shows in launch r"""
    start = torch.arange(H) * (T // H) + r * dk
    return (start[:, None] + torch.arange(dk)[None]) % T


def n_launches(T, dk):
    return -(-T // dk)


def one_hot_v(keys, B, T, dkp):
    H, dk = keys.shape
    v = torch.zeros(T, H, dkp)
    v[keys, torch.arange(H)[:, None].expand(H, dk), torch.arange(dk)[None].expand(H, dk)] = 1.0
    return v.reshape(1, T, H * dkp).expand(B, T, H * dkp).reshape(B * T, H * dkp)


def run_probes(kernel, qkv, pos, lens, B, T, H, dk, monkeypatch):
    """All launches of one case; returns ([ctx (B, T, H, dkp)], [keys (H, dk)])."""
    use_tc, dkp, persist = KERNELS[kernel]
    if persist is None:
        monkeypatch.delenv("CFB_ATTN_PERSIST", raising=False)
    else:
        monkeypatch.setenv("CFB_ATTN_PERSIST", persist)
    Dp = H * dkp
    lens_d = torch.tensor(lens, dtype=torch.int32, device="cuda")
    ctxs, keys = [], []
    for r in range(n_launches(T, dk)):
        kr = probe_keys(T, H, dk, r)
        qkv[:, 3 * Dp:] = one_hot_v(kr, B, T, dkp).to(device="cuda", dtype=qkv.dtype)
        ctx = torch.full((B * T, Dp), float("nan"), dtype=qkv.dtype, device="cuda")
        op_attention(use_tc, qkv, pos, ctx, lens_d, B, T, H, dk, dkp)
        ctxs.append(ctx.view(B, T, H, dkp))
        keys.append(kr)
    return ctxs, keys


def probe_ctx(P, keys_list, dkp, dtype):
    """What a kernel computing the probabilities P (B, H, T, T) would write in each launch: ctx (B, T, H, dkp)."""
    B, H, T, _ = P.shape
    out = []
    for kr in keys_list:
        dk = kr.shape[1]
        ctx = torch.zeros(B, T, H, dkp, dtype=torch.float64, device=P.device)
        ctx[..., :dk] = P.gather(-1, kr.to(P.device)[None, :, None, :].expand(B, H, T, dk)).permute(0, 2, 1, 3)
        out.append(ctx.to(dtype))
    return out


def check_probes(ctxs, keys_list, ref_rows, lens, dk, rel, chunk=None):
    """Element-wise check of every probe against the float64 probabilities ref_rows(i0, i1) -> (B, H, i1-i0, T):
    |got - P| <= rel P + FLOOR where P > 0, got == 0 exactly where P == 0 (masked keys, padded query rows), pad
    columns dk..dkp-1 exactly zero; every key of every row probed; each valid row's probabilities sum to 1 within
    rel + T FLOOR.  Returns a dict (ok, worst = max |err| / bound, and the pattern of the failing elements)."""
    B, T, H, dkp = ctxs[0].shape
    chunk = chunk or T
    lens_t = torch.tensor(lens)
    worst, n_bad, n_checked, pad_nonzero, unprobed, sum_err = 0.0, 0, 0, 0, 0, 0.0
    min_pos = math.inf
    bad_b, bad_i, bad_j, samples = set(), set(), set(), []
    for i0 in range(0, T, chunk):
        i1 = min(T, i0 + chunk)
        P = ref_rows(i0, i1)
        pos_vals = P[P > 0]
        if pos_vals.numel():
            min_pos = min(min_pos, float(pos_vals.min()))
        got_P = torch.full_like(P, float("nan"))
        ncols = min(dk, T)
        for ctx, kr in zip(ctxs, keys_list):
            got = ctx[:, i0:i1].to(P.device).double().permute(0, 2, 1, 3)  # (B, H, rows, dkp)
            kd = kr.to(P.device)[None, :, None, :].expand(B, H, i1 - i0, dk)
            want = P.gather(-1, kd)
            g = got[..., :dk]
            err = (g - want).abs()
            bound = rel * want + FLOOR
            exact = want == 0
            fail = torch.where(exact, g != 0, ~(err <= bound))
            ratio = torch.where(exact, torch.where(g == 0, 0.0, math.inf), err / bound)
            ratio = torch.nan_to_num(ratio, nan=math.inf)
            worst = max(worst, float(ratio.max()))
            n_checked += fail.numel()
            pad_nonzero += int((got[..., dk:] != 0).sum())
            if fail.any():  # the pattern: which sequences, query rows and keys
                n_bad += int(fail.sum())
                bad_b.update(fail.flatten(1).any(1).nonzero().flatten().tolist())
                bad_i.update((i0 + fail.any(3).any(1).any(0).nonzero().flatten()).tolist())
                bad_j.update(kr[fail.any(2).any(0).cpu()].tolist())
                for b, h, ii, c in fail.nonzero()[:8 - len(samples)].tolist():
                    samples.append(dict(b=b, h=h, i=i0 + ii, j=int(kr[h, c]), got=float(g[b, h, ii, c]),
                                        want=float(want[b, h, ii, c])))
            got_P.scatter_(-1, kd[..., :ncols], g[..., :ncols])
        unprobed += int(torch.isnan(got_P).sum())
        i = torch.arange(i0, i1)
        valid = (i[None, :] < lens_t[:, None])[:, None, :].expand(B, H, -1).to(P.device)
        if valid.any():
            sum_err = max(sum_err, float((got_P.sum(-1) - 1).abs()[valid].max()))
    ok = n_bad == 0 and pad_nonzero == 0 and unprobed == 0 and sum_err <= rel + T * FLOOR
    return dict(ok=ok, worst=worst, n_bad=n_bad, n_checked=n_checked, pad_nonzero=pad_nonzero, unprobed=unprobed,
                sum_err=sum_err, min_pos=min_pos, bad_sequences=sorted(bad_b), bad_rows=sorted(bad_i)[:24],
                n_bad_rows=len(bad_i), bad_keys=sorted(bad_j)[:24], n_bad_keys=len(bad_j), samples=samples)


def assert_ok(res, case):
    assert res["ok"], f"{case}: {res}"
    assert res["min_pos"] >= 2.0 ** 10 * FLOOR, f"{case}: the absolute floor is not far below P_min {res['min_pos']}"
    print(f"probs {case}: worst |err|/bound {res['worst']:.4f} over {res['n_checked']} probes, "
          f"row-sum err {res['sum_err']:.2e}, P_min {res['min_pos']:.2e}")


def check_case(kernel, B, T, H, dk, lens, mode, seed, monkeypatch, spikes=(), chunk=None):
    use_tc, dkp, _ = KERNELS[kernel]
    qu, qv, k, p = make_inputs(B, T, H, dk, lens, mode, seed, spikes)
    qkv, pos = pack(qu, qv, k, p, dkp, torch.bfloat16 if use_tc else torch.float32)
    ctxs, keys = run_probes(kernel, qkv, pos, lens, B, T, H, dk, monkeypatch)
    dev = [t.cuda() for t in (qu, qv, k, p)]
    lens_t = torch.tensor(lens)
    res = check_probes(ctxs, keys, lambda i0, i1: ref_probs(*dev, lens_t, i0, i1), lens, dk,
                       REL_TC if use_tc else REL_SIMT, chunk)
    assert_ok(res, f"{kernel} {mode} B={B} T={T} H={H} dk={dk} lens={lens if B <= 12 else '...'}"
                   f"{' spikes=' + str(list(spikes)) if spikes else ''}")


# ------------------------------------------------------------------------------------------------------ GPU cases
def grid_cases():
    """Every T of the grid in every probe mode for each tensor-core kernel, the head widths taking turns; the
    CUDA-core kernel on a subset of T at both padded widths."""
    cases = []
    for kerns, ts in ((("tc", "tcp", "tc128"), T_GRID), (("simt64", "simt128"), [1, 64, 65, 129, 257, 513, 700])):
        for kern in kerns:
            dks = DK_FOR[KERNELS[kern][1]]
            for ti, T in enumerate(ts):
                for mi, mode in enumerate(MODES):
                    dk = dks[(ti + mi) % 3]
                    cases.append(pytest.param(kern, T, dk, mode, id=f"{kern}-{mode}-T{T}-dk{dk}"))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,T,dk,mode", grid_cases())
def test_probabilities_match_float64(kernel, T, dk, mode, monkeypatch):
    seed = 1000 * T_GRID.index(T) + 10 * MODES.index(mode) + list(KERNELS).index(kernel)
    lens = lengths_for(T, seed)
    check_case(kernel, len(lens), T, 2, dk, lens, mode, seed, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("kernel", ["tcp", "tc"])
def test_more_items_than_sms(kernel, mode, monkeypatch):
    """40 sequences x 3 query tiles x 8 heads = 960 items: the persistent kernel's pipelines and barrier phases carry
    across several items per SM, with empty and one-tile sequences in between."""
    B, T, H = 40, 300, 8
    g = torch.Generator().manual_seed(7)
    lens = torch.randint(0, T + 1, (B,), generator=g).tolist()
    lens[:8] = [T, 0, 1, 64, 65, 128, 129, T - 1]
    check_case(kernel, B, T, H, 64, lens, mode, 70 + MODES.index(mode), monkeypatch)


def spike_keys(lens, where):
    """One spike key per non-empty sequence: in the first key tile, in the last one, or in the last tile of the other
    softmax set (tiles alternate between the two sets of attention_tc.cu / attention_tcp.cu)."""
    out = []
    for b, n in enumerate(lens):
        if n == 0:
            continue
        last = (n - 1) // BN
        tile = {"first": 0, "last": last, "other_last": max(last - 1, 0)}[where]
        out.append((b, min(n - 1, tile * BN + 37)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["content", "both"])
@pytest.mark.parametrize("where", ["first", "last", "other_last"])
@pytest.mark.parametrize("kernel", ["tc", "tcp", "tc128"])
def test_running_max_spike(kernel, where, mode, monkeypatch):
    """A key 12 nats above the rest: the online rescale by alpha, and the merge of the two softmax sets, carry the
    small probabilities of every other key (~e^-12 / len, far above ex2.approx.ftz's flush range)."""
    T, lens = 450, [450, 321, 200, 65]
    check_case(kernel, len(lens), T, 2, KERNELS[kernel][1], lens, mode, 90, monkeypatch, spikes=spike_keys(lens, where))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["tc", "tcp"])
def test_long_sequence_cfg5_shape(kernel, monkeypatch):
    """B = 1, T = 7500, 8 heads of 64: the attention of the long-form workload (5 min of audio, BASELINE.json cfg 5),
    the float64 reference computed on the device 500 query rows at a time."""
    T = 7500
    check_case(kernel, 1, T, 8, 64, [T], "both", 75, monkeypatch, chunk=500)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", list(KERNELS))
def test_each_case_runs_the_kernel_it_names(kernel, monkeypatch):
    """The switches above select the kernel the case names (CUDA kernel names from the profiler)."""
    use_tc, dkp, _ = KERNELS[kernel]
    B, T, H, dk = 1, 130, 2, dkp
    qu, qv, k, p = make_inputs(B, T, H, dk, [T], "both", 3)
    qkv, pos = pack(qu, qv, k, p, dkp, torch.bfloat16 if use_tc else torch.float32)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run_probes(kernel, qkv, pos, [T], B, T, H, dk, monkeypatch)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "rel_attn" in e.name}
    assert names and all(KERNEL_SYMBOL[kernel] in n for n in names), names  # no symbol is a substring of another


# ------------------------------------------------------------------------------------------------------ CPU (no GPU)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B,T,H,dk,lens", [(2, 7, 2, 4, [7, 3]), (3, 70, 2, 16, [70, 65, 0]), (1, 130, 1, 8, [129])])
def test_reference_is_the_rel_shift_restatement(B, T, H, dk, lens, mode):
    """The direct index p[T-1+j-i] equals the pad/view rel_shift of test_gpu_attention.torch_reference (the restatement
    of multi_head_attention.py), probabilities read out through an identity V, also when computed in query chunks."""
    qu, qv, k, p = make_inputs(B, T, H, dk, lens, mode, 5)
    lens_t = torch.tensor(lens)
    want = torch_reference(qu, qv, k, torch.eye(T, dtype=torch.float64).expand(B, H, T, T), p, lens_t).permute(0, 2, 1, 3)
    got = torch.cat([ref_probs(qu, qv, k, p, lens_t, i0, min(T, i0 + 48)) for i0 in range(0, T, 48)], 2)
    assert float((got - want).abs().max()) < 1e-12


def round_half_up_bf16(x):
    """fp32 -> bf16 by adding half an ulp to the bit pattern and truncating (attention_tc.cu:422)"""
    bits = x.float().view(torch.int32).long()
    return ((bits + 0x8000) & 0xFFFF0000).to(torch.int32).view(torch.float32).double()


def emulate_kernel_rounding(s, lens):
    """float64 probabilities rounded the way attention_tc.cu rounds them: two softmax sets over alternating key tiles,
    P = bf16 (round half up) of exp(s - m) with the set's running maximum m after the key's tile, the exact rescale and
    normaliser, and the context rounded to bf16 (nearest even)."""
    B, H, R, T = s.shape
    sm = masked(s, lens)
    n_kt = n_launches(T, BN)
    tiles = torch.nn.functional.pad(sm, (0, n_kt * BN - T), value=-math.inf).view(B, H, R, n_kt, BN)
    m_at = torch.empty(B, H, R, n_kt, dtype=torch.float64)
    tmax = tiles.amax(-1)
    for st in (0, 1):
        m_at[..., st::2] = torch.cummax(tmax[..., st::2], -1).values
    m = tmax.amax(-1, keepdim=True)
    live = tiles > -math.inf
    e = torch.where(live, torch.exp(tiles - torch.where(live, m_at[..., None], 0.0)), 0.0)
    l = torch.exp(sm - m).sum(-1, keepdim=True)
    out = round_half_up_bf16(e) * torch.exp(m_at - m)[..., None]
    out = out.reshape(B, H, R, n_kt * BN)[..., :T] / l
    i = torch.arange(R)
    valid = (i[None, :] < lens[:, None])[:, None, :, None]
    return torch.where(valid, out.bfloat16().double(), 0.0)


SELF_TEST = dict(B=3, T=200, H=2, dk=64, lens=[200, 130, 77])


def self_test_case(mode):
    c = SELF_TEST
    qu, qv, k, p = make_inputs(c["B"], c["T"], c["H"], c["dk"], c["lens"], mode, 11)
    return (qu, qv, k, p), torch.tensor(c["lens"])


def checker_verdict(P_got, P_ref, lens, dk=SELF_TEST["dk"]):
    T = P_ref.shape[-1]
    keys = [probe_keys(T, P_ref.shape[1], dk, r) for r in range(n_launches(T, dk))]
    ctxs = probe_ctx(P_got, keys, 64, torch.float64)
    return check_probes(ctxs, keys, lambda i0, i1: P_ref[:, :, i0:i1], lens.tolist(), dk, REL_TC, chunk=96)


def inject(defect, ops, lens):
    """The probabilities (B, H, T, T) a kernel with this defect would compute"""
    qu, qv, k, p = ops
    T = qu.shape[2]
    P = ref_probs(qu, qv, k, p, lens, 0, T)
    if defect == "rel_shift_off_by_one_in_one_band_block":
        shift = torch.zeros(T, dtype=torch.long)
        shift[64:128] = 1
        return softmax_rows(scores(qu, qv, k, p, 0, T, shift), lens, 0)
    if defect == "last_key_dropped":
        bad = P.clone()
        for b, n in enumerate(lens.tolist()):
            bad[b, :, :n, n - 1] = 0
        return bad / bad.sum(-1, keepdim=True).clamp_min(1e-300)
    if defect == "masked_key_in_normaliser":
        s = scores(qu, qv, k, p, 0, T)
        bad = P.clone()
        for b, n in enumerate(lens.tolist()):
            if n < T:  # the first masked key's weight joins the sum over the valid ones
                sv = s[b, :, :n, :n]
                mx = sv.amax(-1, keepdim=True)
                extra = torch.exp(s[b, :, :n, n:n + 1] - mx) / torch.exp(sv - mx).sum(-1, keepdim=True)
                bad[b, :, :n] = P[b, :, :n] / (1 + extra)
        return bad
    if defect == "v_tiles_swapped":
        bad = P.clone()
        bad[..., 64:128], bad[..., 128:192] = P[..., 128:192], P[..., 64:128]
        return bad
    if defect == "query_row_from_neighbour":
        bad = P.clone()
        bad[:, :, 127] = P[:, :, 128]
        return bad
    raise ValueError(defect)


DEFECTS = {  # defect -> the probe mode meant to catch it
    "rel_shift_off_by_one_in_one_band_block": "position",
    "last_key_dropped": "content",
    "masked_key_in_normaliser": "content",
    "v_tiles_swapped": "both",
    "query_row_from_neighbour": "both",
}


@pytest.mark.parametrize("defect", list(DEFECTS))
def test_checker_rejects_injected_defects(defect):
    ops, lens = self_test_case(DEFECTS[defect])
    P = ref_probs(*ops, lens, 0, SELF_TEST["T"])
    bad = inject(defect, ops, lens)
    res = checker_verdict(bad.bfloat16().double(), P, lens)
    assert not res["ok"] and res["n_bad"] > 0, res  # rejected by the element-wise comparison itself
    print(f"{defect}: rejected, {res['n_bad']} probes outside the bound, rows {res['bad_rows'][:8]}.., "
          f"keys {res['bad_keys'][:8]}..")


@pytest.mark.parametrize("mode", MODES)
def test_checker_accepts_kernel_rounding(mode):
    ops, lens = self_test_case(mode)
    T = SELF_TEST["T"]
    P = ref_probs(*ops, lens, 0, T)
    emu = emulate_kernel_rounding(scores(*ops, 0, T), lens)
    res = checker_verdict(emu, P, lens)
    assert res["ok"], res
    assert res["worst"] > 0.5  # the rounding is there and the bound is not loose by orders of magnitude
    print(f"kernel-rounding emulation, {mode}: worst |err|/bound {res['worst']:.4f} (margin {1 - res['worst']:.4f})")
