"""GPU: the TD3 kernels against float64 references -- the learner's five GEMM kernels through its own dispatch (launch(),
tests/cuda/td3_gemm_harness.cu), the generated policy-smoothing noise, the one-call update (plen_td3_train, a captured CUDA
graph) against the piecewise entry points and a float64 twin of the update rule, and the FP16 tensor-core actor against an
exact model of where it rounds."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest
import torch

import td3_gemm_util as hg
from td3_ref import (Td3Twin, actor_fp16_model, actor_noise, f16, graph_draw_seed, learner_noise, replay_rows,
                     train_seed)

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "td3_golden.npz")
DEV = torch.device("cuda:0")

S, A, SA, H = 26, 18, 44, 256
TOWER = H * SA + H + H * H + H + H + 1          # parameters of one critic tower (TOWER_N of plen_td3_learn.cu)
SPLIT_K_MIN_BATCH = 512
KERNELS = ("k_gemm<32,32>", "k_gemm<64,64>", "k_gemm_tc<fwd,BIAS_RELU>", "k_gemm_tc<bwd_data,RELUMASK>", "k_gemm_tc<dW,NONE>")


# ------------------------------------------------------------------------------------------------ the learner's products
# Python restatements of fwd / bwd_data / bwd_weight of plen_td3_learn.cu: strides in elements; *_off = element offset
# of the operand's first element in its buffer (a column sub-range such as the action columns of critic fc1)
def _fwd(name, ldx, xz, ldw, wz, ldc, cz, M, N, K, nz, epi, c_off=0, b_off=0):
    return dict(name=name, M=M, N=N, K=K, nz=nz, epi=epi, a=(xz, ldx, 1, 0), b=(wz, 1, ldw, b_off), c=(cz, ldc, c_off),
                bias=wz, aux=None, rowsum=None)


def _bwd_data(name, ldy, dyz, ldw, wz, ldx, dxz, M, Kin, Nout, nz, epi, ld_aux, aux_z, b_off=0, aux_off=0):
    return dict(name=name, M=M, N=Kin, K=Nout, nz=nz, epi=epi, a=(dyz, ldy, 1, 0), b=(wz, ldw, 1, b_off), c=(dxz, ldx, 0),
                bias=None, aux=(aux_z, ld_aux, aux_off), rowsum=None)


def _bwd_weight(name, ldy, dyz, ldx, xz, ldw, gz, Bt, Nout, Kin, nz):
    return dict(name=name, M=Nout, N=Kin, K=Bt, nz=nz, epi=hg.EPI_NONE, a=(dyz, 1, ldy, 0), b=(xz, ldx, 1, 0), c=(gz, ldw, 0),
                bias=None, aux=None, rowsum=gz)


def learner_products(B):
    """every distinct product of one TD3 update at minibatch B, with the arguments plen_td3_critic_grads /
    plen_td3_actor_grads give it, plus a forward product on the action columns of critic fc1 (rows not 16-byte aligned)"""
    E = hg
    BH = B * H
    return [
        _fwd("critic fc1|fc4", SA, 0, SA, TOWER, H, BH, B, H, SA, 2, E.EPI_BIAS_RELU),
        _fwd("critic fc2|fc5", H, BH, H, TOWER, H, BH, B, H, H, 2, E.EPI_BIAS_RELU),
        _fwd("critic fc3|fc6", H, BH, H, TOWER, 1, B, B, 1, H, 2, E.EPI_BIAS),
        _fwd("actor fc1", SA, 0, S, 0, H, 0, B, H, S, 1, E.EPI_BIAS_RELU),
        _fwd("actor fc2", H, 0, H, 0, H, 0, B, H, H, 1, E.EPI_BIAS_RELU),
        _fwd("actor fc3 (tanh)", H, 0, H, 0, SA, 0, B, A, H, 1, E.EPI_BIAS_TANH, c_off=S),
        _fwd("target actor fc3 (tanh + noise)", H, 0, H, 0, SA, 0, B, A, H, 1, E.EPI_BIAS_TANH_NOISE, c_off=S),
        _fwd("Q1(pi) fc3", H, 0, H, 0, 1, 0, B, 1, H, 1, E.EPI_BIAS),
        _bwd_weight("dW critic fc3|fc6", 1, B, H, BH, H, TOWER, B, 1, H, 2),
        _bwd_data("dX critic fc3|fc6", 1, B, H, TOWER, H, BH, B, H, 1, 2, E.EPI_RELUMASK, H, BH),
        _bwd_weight("dW critic fc2|fc5", H, BH, H, BH, H, TOWER, B, H, H, 2),
        _bwd_data("dX critic fc2|fc5", H, BH, H, TOWER, H, BH, B, H, H, 2, E.EPI_RELUMASK, H, BH),
        _bwd_weight("dW critic fc1|fc4", H, BH, SA, 0, SA, TOWER, B, H, SA, 2),
        _bwd_data("dX Q1 fc1 action columns (tanh grad)", H, 0, SA, 0, A, 0, B, A, H, 1, E.EPI_TANHGRAD, SA, 0, b_off=S, aux_off=S),
        _bwd_weight("dW actor fc3", A, 0, H, 0, H, 0, B, A, H, 1),
        _bwd_data("dX actor fc3", A, 0, H, 0, H, 0, B, H, A, 1, E.EPI_RELUMASK, H, 0),
        _bwd_weight("dW actor fc2", H, 0, H, 0, H, 0, B, H, H, 1),
        _bwd_weight("dW actor fc1", H, 0, SA, 0, S, 0, B, H, S, 1),
        _fwd("fwd on critic fc1 action columns (unaligned rows)", A, 0, SA, 0, H, 0, B, H, A, 1, E.EPI_BIAS_RELU, b_off=S),
    ]


def split_k(p):
    """(splits, k_chunk) of launch()"""
    K = p["K"]
    if p["epi"] == hg.EPI_NONE and p["rowsum"] is not None and K >= SPLIT_K_MIN_BATCH:
        s = min(K // 256, 16)
        chunk = ((K + s - 1) // s + 31) // 32 * 32
        return (K + chunk - 1) // chunk, chunk
    return 1, K


def expected_kernel(p, tc):
    """which of the five kernels launch() picks (its rules restated; test_dispatch_table_names_the_kernel_that_runs checks
    the statement against the kernel that actually runs)"""
    splits = split_k(p)[0]
    ak, bk = p["a"][2], p["b"][1]
    if tc and p["M"] >= 128 and p["N"] >= 16 and p["K"] >= 16:
        if ak == 1 and bk == 1 and p["epi"] == hg.EPI_BIAS_RELU:
            return KERNELS[2]
        if ak == 1 and bk != 1 and p["epi"] == hg.EPI_RELUMASK:
            return KERNELS[3]
        if ak != 1 and bk != 1 and p["epi"] == hg.EPI_NONE and splits > 1:
            return KERNELS[4]
    if -(-p["N"] // 64) * -(-p["M"] // 64) * p["nz"] * splits >= 148:
        return KERNELS[1]
    return KERNELS[0]


def accumulates(p):
    """the product adds into C / rowsum (split-K, on either kernel family): they must be zeroed first, as the learner does"""
    return split_k(p)[0] > 1


TABLE_B = (1, 31, 100, 127, 128, 129, 511, 512, 513, 1000, 4096, 4097, 65536)


def test_dispatch_table_reaches_every_kernel():
    seen = {expected_kernel(p, tc) for B in TABLE_B for tc in (False, True) for p in learner_products(B)}
    assert seen == set(KERNELS)
    # the boundaries of launch(): 16 splits, N rounded up to 16 on the tensor cores, a ragged one-row last tile
    assert split_k(learner_products(4096)[10])[0] == 16 and split_k(learner_products(511)[10])[0] == 1
    assert {p["N"] for p in learner_products(4097) if expected_kernel(p, True) == KERNELS[4]} >= {26, 44, 256}


class Case:
    """operand, output and reference buffers of one product; `kind` draws the operands: "int" = integers in {-2..2}
    (every partial sum exact in fp32 and in TF32 operands), "float" = standard normal"""

    def __init__(self, p, kind, gen, p_epi=(1.0, 0.2, 0.5), seed=12345):
        self.p, self.p_epi, self.seed = p, p_epi, seed
        nz, M, N, K = p["nz"], p["M"], p["N"], p["K"]

        def draw(n):
            if kind == "int":
                return torch.randint(-2, 3, (n,), device=DEV, generator=gen).to(torch.float32)
            return torch.randn(n, device=DEV, generator=gen)

        def operand(z, r, k, rows, cols, off):
            n = off + (nz - 1) * z + (rows - 1) * r + (cols - 1) * k + 1
            buf = draw(n)
            return buf, buf.double().as_strided((nz, rows, cols), (z, r, k), off)

        az, am, ak, _ = p["a"]
        bz, bk, bn, boff = p["b"]
        self.abuf, self.A = operand(az, am, ak, M, K, 0)
        self.bbuf, self.B = operand(bz, bk, bn, K, N, boff)
        self.b_off = boff
        self.bias = self.biasv = None
        if p["bias"] is not None:
            self.bias = draw((nz - 1) * p["bias"] + N)
            self.biasv = self.bias.double().as_strided((nz, 1, N), (p["bias"], 0, 1))
        self.aux = self.auxv = None
        if p["aux"] is not None:
            aux_z, ld_aux, aoff = p["aux"]
            n = aoff + (nz - 1) * aux_z + (M - 1) * ld_aux + N
            if p["epi"] == hg.EPI_TANHGRAD:      # max_action tanh(.) values
                self.aux = (torch.rand(n, device=DEV, generator=gen) * 2 - 1) * 0.999 * p_epi[0]
            else:                                # activations with exact zeros
                self.aux = torch.randint(-2, 3, (n,), device=DEV, generator=gen).to(torch.float32)
            self.aux_off = aoff
            self.auxv = self.aux.double().as_strided((nz, M, N), (aux_z, ld_aux, 1), aoff)
        cz, ldc, coff = p["c"]
        self.c_n = coff + (nz - 1) * cz + (M - 1) * ldc + N
        self.c_view = lambda t: t.as_strided((nz, M, N), (cz, ldc, 1), coff)
        if p["rowsum"] is not None:
            self.r_n = (nz - 1) * p["rowsum"] + M
            self.r_view = lambda t: t.as_strided((nz, M), (p["rowsum"], 1), 0)

    def reference(self):
        """float64 (C, rowsum) buffers as the product should leave them, unwritten entries = `fill`"""
        acc = self.A @ self.B
        e, (p0, p1, p2) = self.p["epi"], self.p_epi
        if e == hg.EPI_BIAS:
            acc = acc + self.biasv
        elif e == hg.EPI_BIAS_RELU:
            acc = torch.relu(acc + self.biasv)
        elif e == hg.EPI_BIAS_TANH:
            acc = p0 * torch.tanh(acc + self.biasv)
        elif e == hg.EPI_BIAS_TANH_NOISE:
            nz = torch.from_numpy(learner_noise(self.seed, self.p["M"], self.p["N"])).to(DEV)
            acc = (p0 * torch.tanh(acc + self.biasv) + (nz * p1).clamp(-p2, p2)).clamp(-p0, p0)
        elif e == hg.EPI_RELUMASK:
            acc = torch.where(torch.relu(self.auxv) > 0, acc, torch.zeros_like(acc))
        elif e == hg.EPI_TANHGRAD:
            t = self.auxv / p0
            acc = acc * p0 * (1 - t * t)
        return acc, (self.A.sum(-1) if self.p["rowsum"] is not None else None)

    def run(self, tc, fill):
        """launch the product with C / rowsum pre-filled with `fill`; -> (C buffer, rowsum buffer or None)"""
        p = self.p
        c = torch.full((self.c_n,), fill, device=DEV)
        rs = torch.full((self.r_n,), fill, device=DEV) if p["rowsum"] is not None else None
        az, am, ak, _ = p["a"]
        bz, bk, bn, _ = p["b"]
        cz, ldc, coff = p["c"]
        kw = {}
        if p["aux"] is not None:
            kw = dict(aux=self.aux.data_ptr() + 4 * self.aux_off, aux_z=p["aux"][0], ld_aux=p["aux"][1])
        hg.gemm(self.abuf, self.bbuf.data_ptr() + 4 * self.b_off, c.data_ptr() + 4 * coff, M=p["M"], N=p["N"], K=p["K"],
                az=az, am=am, ak=ak, bz=bz, bk=bk, bn=bn, cz=cz, ldc=ldc, nz=p["nz"], epi=p["epi"], bias=self.bias,
                bias_z=p["bias"] or 0, p=self.p_epi, seed=self.seed, rowsum=rs, rowsum_z=p["rowsum"] or 0, tc=tc, **kw)
        return c, rs


def _expected_buffer(n, view, val, fill):
    out = torch.full((n,), fill, device=DEV, dtype=torch.float64)
    view(out).copy_(val)
    return out


@pytest.mark.parametrize("tc", [False, True], ids=["fp32", "tc"])
@pytest.mark.parametrize("B", TABLE_B)
def test_learner_gemm_exact_with_integer_operands(B, tc):
    """Integer operands in {-2..2}: every partial sum (|.| < 2^19) is exact in fp32 under any summation order, split-K
    atomics included, and an integer below 2^11 has no TF32 low part -- so the FP32 kernels and all three 3xTF32 instances
    must equal the float64 product bit for bit: outputs, bias-gradient row sums, ReLU at exact zero, ReLU masks built by
    torch.relu.  The tanh epilogues then differ only by tanhf's rounding.  Entries outside the output (the state columns
    next to the action columns) must stay untouched."""
    gen = torch.Generator(device=DEV)
    gen.manual_seed(1000 + B)
    for p in learner_products(B):
        case = Case(p, "int", gen)
        acc = accumulates(p)
        fill = 0.0 if acc else -777.25
        c, rs = case.run(tc, fill)
        ref, rref = case.reference()
        exp = _expected_buffer(case.c_n, case.c_view, ref, fill)
        what = (B, tc, p["name"], expected_kernel(p, tc))
        if p["epi"] in (hg.EPI_BIAS_TANH, hg.EPI_BIAS_TANH_NOISE, hg.EPI_TANHGRAD):
            # tanhf / logf / cospif ulps; for the tanh gradient the float32 (1 - t^2) times the exact accumulator
            scale = case.p_epi[0] * (1.0 + case.A.abs() @ case.B.abs()) if p["epi"] == hg.EPI_TANHGRAD else 1.0 + ref.abs()
            assert bool(((case.c_view(c).double() - ref).abs() <= 1e-6 * scale).all()), what
            untouched = torch.ones(case.c_n, dtype=torch.bool, device=DEV)
            case.c_view(untouched).fill_(False)
            assert bool((c[untouched] == fill).all()), what
        else:
            assert torch.equal(c.double(), exp), what
        if rref is not None:
            assert torch.equal(rs.double(), _expected_buffer(case.r_n, case.r_view, rref, fill)), what
    torch.cuda.synchronize()
    assert hg.load_harness().harness_tc_timed_out() == 0


def test_dispatch_table_names_the_kernel_that_runs():
    """The kernel each table entry names is the one launch() runs (kernel names from the CUDA activity trace)."""
    from torch.profiler import ProfilerActivity, profile
    gen = torch.Generator(device=DEV)
    gen.manual_seed(7)
    runs = []
    for B in (100, 1000, 4097):
        for tc in (False, True):
            for p in learner_products(B):
                runs.append((Case(p, "int", gen), tc, expected_kernel(p, tc)))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for case, tc, _ in runs:
            case.run(tc, 0.0)
        torch.cuda.synchronize()
    names = [e.name for e in sorted(prof.events(), key=lambda e: e.time_range.start)
             if e.device_type == torch.autograd.DeviceType.CUDA and "k_gemm" in e.name]
    pattern = {KERNELS[0]: "k_gemm<32, 32", KERNELS[1]: "k_gemm<64, 64", KERNELS[2]: "k_gemm_tc<true, true",
               KERNELS[3]: "k_gemm_tc<true, false", KERNELS[4]: "k_gemm_tc<false, false"}
    assert len(names) == len(runs), (len(names), len(runs))
    for name, (case, tc, k) in zip(names, runs):
        assert pattern[k] in name, (case.p["name"], case.p["M"], tc, k, name)


# products that run on the tensor cores at a large minibatch, each kind with its epilogue
TC_PRODUCTS = ("critic fc1|fc4", "critic fc2|fc5", "actor fc1", "dX critic fc2|fc5", "dX actor fc3", "dW critic fc2|fc5",
               "dW critic fc1|fc4", "dW actor fc1", "fwd on critic fc1 action columns (unaligned rows)")
# Measured on a B200 (1000 W): the 3xTF32 error is 1.6-3.0x the FP32 kernel's on the forward and backward-data products
# and 5.0-6.0x on the split-K backward-weight products (the tensor cores' FP32 accumulation is coarser than the FP32 cores'
# round-to-nearest FMA chains), at most 9.6e-7 (x 2^11: 2.0e-3) relative to (|A| |B|)_mn.  Bounds: 10x, and 2^-19.
TC_ERR_FACTOR = 10.0
TF32_ONE_PASS = 2.0 ** -11           # relative size of a missing TF32 low part


@pytest.mark.parametrize("B", [1024, 4096])
def test_learner_gemm_rounding_3xtf32_vs_fp32(B):
    """Random normal operands: every entry of every product against float64, as error / (|A| |B| + |bias|)_mn -- not
    normalised by the largest entry, where cancellation in gradient sums would hide errors.  The 3xTF32 kernels stay within
    TC_ERR_FACTOR of the FP32 kernels' error on the same product and 256x below what one TF32 pass leaves (2^-11)."""
    gen = torch.Generator(device=DEV)
    gen.manual_seed(77 + B)
    for p in learner_products(B):
        if p["name"] not in TC_PRODUCTS:
            continue
        assert expected_kernel(p, True) in KERNELS[2:]
        case = Case(p, "float", gen)
        ref, rref = case.reference()
        mag = case.A.abs() @ case.B.abs()
        if case.biasv is not None:
            mag = mag + case.biasv.abs()
        err = {}
        for tc in (False, True):
            c, rs = case.run(tc, 0.0)
            e = ((case.c_view(c).double() - ref).abs() / mag.clamp_min(1e-30)).max().item()
            if rref is not None:
                rmag = case.A.abs().sum(-1)
                e = max(e, ((case.r_view(rs).double() - rref).abs() / rmag.clamp_min(1e-30)).max().item())
            err[tc] = e
        print("B %5d %-50s fp32 %.3e  3xtf32 %.3e  ratio %.2f  (x 2^11: %.1e)"
              % (B, p["name"], err[False], err[True], err[True] / err[False], err[True] / TF32_ONE_PASS))
        assert err[True] <= TC_ERR_FACTOR * max(err[False], 2.0 ** -24), (p["name"], err)
        assert err[True] <= TF32_ONE_PASS / 256, (p["name"], err)
    torch.cuda.synchronize()
    assert hg.load_harness().harness_tc_timed_out() == 0


@pytest.mark.parametrize("tc", [False, True], ids=["fp32", "tc"])
def test_learner_epilogues_noise_clip_and_max_action(tc):
    """EPI_BIAS_TANH_NOISE with the generator's own noise, value by value against the Python port (splitmix64 counters,
    float32 uniforms, Box-Muller): clipped at noise_clip and at max_action, both edges hit; EPI_BIAS_TANH and EPI_TANHGRAD
    with max_action = 2.  Dyadic operands keep the accumulator exact, so only logf / cospif / tanhf rounding remains."""
    gen = torch.Generator(device=DEV)
    gen.manual_seed(5)
    B = 4096
    prods = {p["name"]: p for p in learner_products(B)}
    for p_epi in ((1.0, 0.2, 0.5), (2.0, 0.3, 0.4), (2.0, 0.5, 1.5)):
        for name in ("target actor fc3 (tanh + noise)", "actor fc3 (tanh)", "dX Q1 fc1 action columns (tanh grad)"):
            case = Case(prods[name], "int", gen, p_epi=p_epi, seed=0xC0FFEE + int(10 * p_epi[1]))
            case.bbuf.mul_(1.0 / 64)                     # dyadic: |acc| stays small (tanh not saturated), still exact
            case.B = case.B / 64
            c, _ = case.run(tc, -777.25)
            ref, _ = case.reference()
            got = case.c_view(c).double()
            scale = p_epi[0] * (1.0 + case.A.abs() @ case.B.abs()) if name.startswith("dX") else p_epi[0]
            d = ((got - ref).abs() / scale).max().item()
            assert d < 1e-6, (p_epi, name, d)
            if "noise" in name:
                p0, p1, p2 = p_epi
                nz = torch.from_numpy(learner_noise(case.seed, B, A)).to(DEV) * p1
                pre = p0 * torch.tanh(case.A @ case.B + case.biasv)[0] + nz.clamp(-p2, p2)
                assert int((nz.abs() > p2).sum()) > 10                     # noise_clip reached
                assert int((pre.abs() > p0).sum()) > 10                    # max_action reached
                assert float(got.abs().max()) <= p0
                # the raw draws are standard normal
                z = learner_noise(case.seed, B, A)
                assert abs(z.mean()) < 0.02 and abs(z.std() - 1) < 0.02


# ------------------------------------------------------------------------------------------------ the one-call update
def _replay(n, dev, seed, max_action=1.0):
    from plen_ml_walk_b200.td3 import ReplayBuffer
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    st = torch.randn(n, 26, device=dev, generator=g)
    ac = (torch.rand(n, 18, device=dev, generator=g) * 2 - 1) * max_action
    s2 = st + 0.05 * torch.randn(n, 26, device=dev, generator=g)
    r = torch.randn(n, device=dev, generator=g)
    dn = torch.rand(n, device=dev, generator=g) < 0.05
    rb = ReplayBuffer(n, device=dev, seed=3)
    rb.add(st, ac, s2, r, dn)
    return rb


def _agent(seed=0, **kw):
    from plen_ml_walk_b200.td3 import TD3Agent
    torch.manual_seed(seed)
    return TD3Agent(device=DEV, seed=seed, **kw)


def _copy_agent(src, **kw):
    b = _agent(seed=src._seed, **kw)
    for k in ("actor", "actor_target", "critic", "critic_target"):
        b._flat[k].copy_(src._flat[k])
    return b


def test_one_call_update_equals_piecewise_entry_points_bitwise():
    """plen_td3_train (captured graph: minibatch drawn in k_sample_sa from the call seed, noise generated in the epilogue,
    Adam scalars read from device memory) against the piecewise entry points given the same draw seed, noise seed and Adam
    steps: below 512 rows in fp32 (no split-K atomics) 8 updates must agree bit for bit -- parameters, Adam moments and
    losses."""
    rb = _replay(5000, DEV, 1)
    for B in (100, 384):
        a = _agent(seed=9)
        b = _copy_agent(a)
        for it in range(8):
            al, cl = a.train(rb, B, return_losses=True)
            L, P, h = b._cuda_handles()
            b.total_it += 1
            b._draws += 1
            s = train_seed(b)
            assert s == train_seed(a)
            st = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
            policy = b.total_it % b.policy_freq == 0
            assert L.plen_td3_sample(b._learner, rb._rb, B, graph_draw_seed(s), st) == 0
            assert L.plen_td3_critic_grads(b._learner, C.byref(P), C.byref(h), None, s, C.c_void_p(b._losses.data_ptr() + 4), st) == 0
            b.critic_steps += 1
            assert L.plen_td3_adam(P.critic, P.critic_grad, P.critic_m, P.critic_v, 155138, b.critic_steps, C.byref(h), 0, st) == 0
            if policy:
                assert L.plen_td3_actor_grads(b._learner, C.byref(P), C.byref(h), C.c_void_p(b._losses.data_ptr()), st) == 0
                b.actor_steps += 1
                assert L.plen_td3_adam(P.actor, P.actor_grad, P.actor_m, P.actor_v, 77330, b.actor_steps, C.byref(h), 0, st) == 0
                assert L.plen_td3_soft_update(P.critic_target, P.critic, 155138, float(b.tau), 0, st) == 0
                assert L.plen_td3_soft_update(P.actor_target, P.actor, 77330, float(b.tau), 0, st) == 0
                assert torch.equal(al, b._losses[0]), (B, it)
            assert torch.equal(cl, b._losses[1]), (B, it)
            for k in ("actor", "critic", "actor_target", "critic_target"):
                assert torch.equal(a._flat[k], b._flat[k]), (B, it, k)
            for k in ("actor_m", "actor_v", "critic_m", "critic_v"):
                assert torch.equal(a._adam[k], b._adam[k]), (B, it, k)
        assert a.critic_steps == b.critic_steps == 8 and a.actor_steps == b.actor_steps == 4


def _resumed_agent(precision):
    """an agent loaded from a four-file checkpoint whose Adam states are at step 1e5 / 5e4"""
    a = _agent(seed=31, precision=precision)
    g = torch.Generator(device=DEV)
    g.manual_seed(32)
    for k in ("actor", "critic"):
        m = 1e-3 * torch.randn(a._adam[k + "_m"].shape, device=DEV, generator=g)
        a._adam[k + "_m"].copy_(m)
        a._adam[k + "_v"].copy_(m * m + 1e-7 * torch.rand(m.shape, device=DEV, generator=g))
    a.critic_steps, a.actor_steps = 100000, 50000
    with tempfile.TemporaryDirectory() as td:
        a.save(td + "/ck")
        b = _agent(seed=33, precision=precision)
        b.load(td + "/ck", sync_targets=True)
    assert b.critic_steps == 100000 and b.actor_steps == 50000
    return b


GRAPH_CASES = {
    "fp32-B100": (dict(), [100] * 6),
    "fp32-B37": (dict(), [37] * 6),
    "fp32-B1024": (dict(), [1024] * 6),
    "tf32-B1024": (dict(precision="tf32"), [1024] * 6),
    "tf32-B4096": (dict(precision="tf32"), [4096] * 6),
    "fp32-hyper": (dict(max_action=2.0, policy_noise=0.3, noise_clip=0.4, discount=0.9, policy_freq=3), [256] * 6),
    "tf32-resumed": ("resume", [1024] * 6),
    "tf32-batch-change": (dict(precision="tf32"), [1024, 1024, 100, 100, 1024, 1024]),
}
PARAM_MAX, PARAM_MEAN = 1e-4, 2e-6      # as the piecewise parity test of test_td3_gpu.py
ADAM_STEP_MAX = 3 * 3e-4                 # any parameter, per update: a few Adam steps of lr = 3e-4
# Share of a network's well-conditioned parameters allowed above PARAM_MAX: at a minibatch of 1024 a row whose
# pre-activation lies within rounding of zero can take the other side of a ReLU in one of the two runs, which puts one
# full term into a gradient sum, and the parameters it moves feed back into the next updates.  Measured on a B200: up to
# 12 of the critic's 155,138 parameters (7.7e-5, at most 2.9e-4 off) after 6 tf32 updates at B = 1024, none elsewhere.
MAX_OUTLIER_SHARE = 5e-4


@pytest.mark.parametrize("case", list(GRAPH_CASES))
def test_one_call_update_matches_float64_rule(case):
    """TD3Agent.train(replay, B) -- the one-call graph path of production runs and bench.py -- against the reference rule in
    float64 (autograd + torch.optim.Adam) on the same minibatch rows (plen_replay_sample with the graph's draw seed) and the
    same smoothing noise (the generator port), over 6 consecutive updates including policy updates.  After every update the
    parameters of the four networks agree within 1e-4 (a third of one Adam step) and 2e-6 on average.  The exception are
    parameters whose Adam step was ill-conditioned (sqrt(v_hat) below 1 % of the network's RMS at some update, see
    Td3Twin.adam_sensitive): there a gradient difference at the level of fp32 rounding -- which split-K atomics alone
    produce from run to run -- moves the step by up to 2 lr, so they are only held to a few Adam steps; and a share of
    at most MAX_OUTLIER_SHARE of the others may pass 1e-4 through a ReLU taken on the other side of zero."""
    kw, batches = GRAPH_CASES[case]
    agent = _resumed_agent("tf32") if kw == "resume" else _agent(seed=len(case), **kw)
    rb = _replay(20000, DEV, 2, agent.max_action)
    twin = Td3Twin(agent)
    worst = worst_sens = n_sens = 0.0
    outliers = 0
    for it, B in enumerate(batches):
        al, cl = agent.train(rb, B, return_losses=True)
        s = train_seed(agent)
        st, ac, s2, r, nd, _ = replay_rows(rb, B, graph_draw_seed(s))
        tal, tcl = twin.update((st, ac, s2, r, nd), torch.from_numpy(learner_noise(s, B)).to(DEV))
        assert abs(float(cl) - tcl) <= 1e-4 * max(1.0, abs(tcl)), (case, it, float(cl), tcl)
        assert (al is None) == (tal is None), (case, it)
        if tal is not None:
            assert abs(float(al) - tal) <= 1e-4 * max(1.0, abs(tal)), (case, it, float(al), tal)
        for k in ("actor", "critic", "actor_target", "critic_target"):
            d = (agent._flat[k].double() - twin.flat(k)).abs()
            sens = twin.adam_sensitive(k) if k in ("actor", "critic") else torch.zeros_like(d, dtype=torch.bool)
            dw = d[~sens]
            n_out = int((dw >= PARAM_MAX).sum())
            worst = max(worst, float(dw.max()))
            worst_sens = max(worst_sens, float(d[sens].max()) if bool(sens.any()) else 0.0)
            n_sens = max(n_sens, float(sens.double().mean()))
            outliers = max(outliers, n_out)
            assert n_out <= MAX_OUTLIER_SHARE * d.numel() and float(d.mean()) < PARAM_MEAN, (case, it, k, n_out, float(dw.max()), float(d.mean()))
            assert float(d.max()) < ADAM_STEP_MAX * (it + 1), (case, it, k, float(d.max()))
    for k in ("actor", "critic"):
        m, v = twin.moments(k)
        assert float((agent._adam[k + "_m"].double() - m).abs().max()) < 2e-2 * float(m.abs().max()), (case, k)
        assert float((agent._adam[k + "_v"].double() - v).abs().max()) < 2e-2 * float(v.abs().max()), (case, k)
    assert agent.actor_steps == twin.actor_optimizer.state[next(iter(twin.actor.parameters()))]["step"].item()
    torch.cuda.synchronize()
    from plen_ml_walk_b200 import _abi
    assert _abi.load_library().plen_td3_tc_timed_out() == 0
    print("graph vs float64, %s: worst parameter difference %.2e (%d above %.0e); Adam-sensitive parameters (<= %.2f %%) %.2e"
          % (case, worst, outliers, PARAM_MAX, 100 * n_sens, worst_sens))


# ------------------------------------------------------------------------------------------------ FP16 tensor-core actor
def _shipped_actor():
    from plen_ml_walk_b200.td3 import Actor
    g = np.load(GOLD)
    a = Actor().to(DEV)
    a.load_state_dict({k: torch.from_numpy(g["actor_" + k.replace(".", "_")]).to(DEV) for k in a.state_dict().keys()})
    return a


def _fresh_actor(max_action):
    from plen_ml_walk_b200.td3 import Actor
    torch.manual_seed(0)
    return Actor(max_action=max_action).to(DEV)


def _probe_rows(actor, scale):
    """26 one-hot rows (one observation feature set, the rest zero) and one row whose first hidden activation exceeds
    65504 (saturated to the largest FP16 by the kernel)"""
    eye = torch.eye(S, device=DEV) * scale
    w = actor.fc1.weight.detach()[0]
    big = (60000.0 * torch.sign(w)).reshape(1, S)
    pre = float(f16(big.double()) @ f16(w.double()) + actor.fc1.bias.detach()[0].double())
    assert pre > 65504.0
    return torch.cat([eye, big])


# residual of the FP16 actor against its exact rounding model: (median, 99.9th percentile, max).  Measured on a B200:
# shipped checkpoint 6.4e-14 / 4.8e-4 / 4.0e-2 (its large weights turn one FP16 rounding-boundary flip of a hidden
# activation into a visible action change where a tanh is steep), fresh network 4.7e-8 / 5.6e-5 / 1.9e-4.  Bounds: the
# measured values with a 2-4x margin (the medians rounded up to a decade).
FP16_BOUNDS = {"shipped": (1e-12, 1e-3, 8e-2), "fresh-max2": (1e-7, 2e-4, 5e-4)}


@pytest.mark.parametrize("which", ["shipped", "fresh-max2"])
def test_fp16_actor_matches_rounding_model(which):
    """plen_actor_forward_tc against a float64 model that rounds exactly where the kernel does (operands and both hidden
    layers to FP16, saturating at +-65504); what remains is the tensor cores' accumulation order and the rare FP16
    rounding-boundary flip it causes.  Ragged N, the persistent loop with more than one tile per CTA, one-hot probes (a
    dropped or misplaced observation column shows alone), a saturating row, max_action = 2."""
    from plen_ml_walk_b200 import _abi
    from plen_ml_walk_b200.td3 import actor_forward
    actor = _shipped_actor() if which == "shipped" else _fresh_actor(2.0)
    b_med, b_p999, b_max = FP16_BOUNDS[which]
    gen = torch.Generator(device=DEV)
    gen.manual_seed(3)
    res = []
    for n in (1, 127, 128, 129, 148 * 128, 148 * 128 + 1, 2 * 148 * 128 + 77):
        obs = torch.randn(n, S, device=DEV, generator=gen) * (0.5 if which == "shipped" else 1.0)
        if n == 2 * 148 * 128 + 77:
            obs[-S - 1:] = _probe_rows(actor, 1.0)
        got = actor_forward(actor, obs, precision="fp16").double()
        ref = actor_fp16_model(actor, obs)
        assert bool(torch.isfinite(got).all()), (which, n)
        res.append((got - ref).abs().reshape(-1))
    probes = _probe_rows(actor, 2.0)
    d = (actor_forward(actor, probes, precision="fp16").double() - actor_fp16_model(actor, probes)).abs()
    assert float(d.max()) < b_max, (which, "probes", d.max(dim=1).values.tolist())
    torch.cuda.synchronize()
    assert _abi.load_library().plen_actor_tc_timed_out() == 0
    r = torch.cat(res)
    med, p999, mx = float(r.median()), float(torch.quantile(r[:2 ** 24].float(), 0.999)), float(r.max())
    print("fp16 actor vs rounding model (%s): median %.2e  p99.9 %.2e  max %.2e  (%d actions)" % (which, med, p999, mx, r.numel()))
    assert med < b_med and p999 < b_p999 and mx < b_max, (which, med, p999, mx)


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_actor_exploration_noise_values(precision):
    """The exploration noise of both actor kernels, value by value: clip(clean + noise_std z, +-max_action) with z from the
    generator port (counter seed * FNV + 32 row + joint), on the shipped checkpoint and with max_action = 2."""
    from plen_ml_walk_b200.td3 import actor_forward
    gen = torch.Generator(device=DEV)
    gen.manual_seed(4)
    for actor in (_shipped_actor(), _fresh_actor(2.0)):
        ma = actor.max_action
        n, std, seed = 5000, 0.3 * ma, 0x1234567 + int(ma)
        obs = torch.randn(n, S, device=DEV, generator=gen)
        clean = actor_forward(actor, obs, precision=precision).double()
        noisy = actor_forward(actor, obs, noise_std=std, seed=seed, precision=precision).double()
        z = torch.from_numpy(actor_noise(seed, n)).to(DEV)
        pre = clean + std * z
        ref = pre.clamp(-ma, ma)
        d = float((noisy - ref).abs().max())
        assert d < 2e-6 * ma, (precision, ma, d)
        assert int((pre.abs() > ma).sum()) > 100 and int((pre.abs() < ma).sum()) > 1000     # both sides of the clip
