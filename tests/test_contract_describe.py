"""The full `contract_describe` string of every contraction path, for every dtype and every value of
SBB_CONTRACT_KERNEL (examined on the host; without a device the B200's 148 SMs are assumed).  Pins the
order in which the paths are tried (empty, tcgen05, dot, row, mma, simt), where a forced kernel that
cannot take a problem falls through to, and the parameters each path describes."""
import pytest

import superbblas_b200 as sb

D = sb.contract_desc
DTYPES = (sb.F32, sb.F64, sb.C64, sb.C128)
# values of SBB_CONTRACT_KERNEL: unset, each kernel, and a value that names no kernel
FORCES = (None, "simt", "mma", "tc", "row", "dot", "bogus")


def distillation(T, m, n, K):
    """cxyztn^H . cxyztm -> tnm after the planner merged c,x,y,z: K contiguous in both operands"""
    return D(T=[(T, K, K, 1)], M=[(m, K * T, 0, T)], N=[(n, 0, K * T, T * m)], K=[(K, 1, 1, 0)], conj0=True)


def skinny(m, n, k, b=32):
    """The reference's dist.cpp batched GEMMs: v0[m,k,b] v1[k,n,b] -> vr[m,n,b] (column major)"""
    return D(T=[(b, m * k, k * n, m * n)], M=[(m, 1, 0, 1)], N=[(n, 0, k, m)], K=[(k, m, 1, 0)])


def mma(shape, split, smem, kfast):
    """The mma kernel's description for F32, F64, C64 and C128; `smem` lists their bytes in that order"""
    return {dt: "mma f64%s tile=64x64x8 stages=4 %s %s smem=%d %s loader=cp.async"
            % (" (float operands)" if dt in (sb.F32, sb.C64) else "", shape, split, s, kfast)
            for dt, s in zip(DTYPES, smem)}


# shared memory of the mma kernel by operand layout (F32, F64, C64, C128)
KK = (24576, 49152, 49152, 98304), "a_kfast=1 b_kfast=1"
RK = (21504, 41984, 41984, 82944), "a_kfast=0 b_kfast=1"
RR = (18432, 34816, 34816, 67584), "a_kfast=0 b_kfast=0"
TC = "tcgen05 tf32x3 tile=64x64x32 (complex) %s %s promote=4 smem=230656 loader=tma"

# name: (descriptor, description of each path it can take, path for each value in FORCES, the same for
# complex float where it differs)
PROBLEMS = {
    "headline": (
        distillation(64, 64, 64, 3 * 32 ** 3),
        dict(mma=mma("T=64 M=64 N=64 K=98304", "ksplit=37 ctas=2368", *KK),
             tc=TC % ("T=64 M=64 N=64 K=98304", "ksplit=9 ctas=576"),
             simt="simt T=64 M=64 N=64 K=98304"),
        "mma simt mma mma mma mma mma", "tc simt mma tc mma mma mma"),
    "configs3": (
        distillation(24, 128, 128, 3 * 48 * 48 * 24),
        dict(mma=mma("T=24 M=128 N=128 K=165888", "ksplit=37 ctas=3552", *KK),
             tc=TC % ("T=24 M=128 N=128 K=165888", "ksplit=3 ctas=288"),
             simt="simt T=24 M=128 N=128 K=165888"),
        "mma simt mma mma mma mma mma", "tc simt mma tc mma mma mma"),
    "short_k": (  # too short for tcgen05
        distillation(64, 64, 64, 128),
        dict(mma=mma("T=64 M=64 N=64 K=128", "ksplit=1 ctas=64", *KK), simt="simt T=64 M=64 N=64 K=128"),
        "mma simt mma mma mma mma mma", None),
    "strided_k": (  # K not contiguous: no tcgen05
        D(T=[(8, 64 * 4096, 64 * 4096, 1)], M=[(64, 1, 0, 8)], N=[(64, 0, 1, 512)], K=[(4096, 64, 64, 0)]),
        dict(mma=mma("T=8 M=64 N=64 K=4096", "ksplit=16 ctas=128", *RR), simt="simt T=8 M=64 N=64 K=4096"),
        "mma simt mma mma mma mma mma", None),
    "tile_12x64": (  # M under 16: no tcgen05
        distillation(8, 12, 64, 4096),
        dict(mma=mma("T=8 M=12 N=64 K=4096", "ksplit=16 ctas=128", *KK), simt="simt T=8 M=12 N=64 K=4096"),
        "mma simt mma mma mma mma mma", None),
    "dot_1x1": (
        skinny(1, 1, 49152),
        dict(dot="dot T=32 M=1 N=1 K=49152 slices=8192 blocks=1x1",
             mma=mma("T=32 M=1 N=1 K=49152", "ksplit=74 ctas=2368", *KK), simt="simt T=32 M=1 N=1 K=49152"),
        "dot simt mma mma mma dot mma", None),
    "dot_4x4": (
        skinny(4, 4, 49152),
        dict(dot="dot T=32 M=4 N=4 K=49152 slices=8192 blocks=1x1",
             mma=mma("T=32 M=4 N=4 K=49152", "ksplit=74 ctas=2368", *RK), simt="simt T=32 M=4 N=4 K=49152"),
        "dot simt mma mma mma dot mma", None),
    "dot_12x12": (
        skinny(12, 12, 49152),
        dict(dot="dot T=32 M=12 N=12 K=49152 slices=1024 blocks=3x3",
             mma=mma("T=32 M=12 N=12 K=49152", "ksplit=74 ctas=2368", *RK), simt="simt T=32 M=12 N=12 K=49152"),
        "dot simt mma mma mma dot mma", None),
    "dot_short_k": (  # K under 1024: the dot kernel only when forced
        skinny(4, 4, 256),
        dict(dot="dot T=32 M=4 N=4 K=256 slices=256 blocks=1x1",
             mma=mma("T=32 M=4 N=4 K=256", "ksplit=1 ctas=32", *RK), simt="simt T=32 M=4 N=4 K=256"),
        "simt simt mma simt simt dot simt", None),
    "dot_over_bound": (  # too many threads for the dot kernel's workspace
        distillation(4096, 16, 16, 1024),
        dict(mma=mma("T=4096 M=16 N=16 K=1024", "ksplit=1 ctas=4096", *KK),
             tc=TC % ("T=4096 M=16 N=16 K=1024", "ksplit=1 ctas=4096"),
             simt="simt T=4096 M=16 N=16 K=1024"),
        "mma simt mma mma mma mma mma", "tc simt mma tc mma mma mma"),
    "row_1": (
        skinny(49152, 1, 1),
        dict(row="row rows=1572864 small=1 K=1 big_operand=v0",
             mma=mma("T=32 M=49152 N=1 K=1", "ksplit=1 ctas=24576", *RR), simt="simt T=32 M=49152 N=1 K=1"),
        "row simt mma simt row simt simt", None),
    "row_3": (
        skinny(49152, 3, 3),
        dict(row="row rows=1572864 small=3 K=3 big_operand=v0",
             mma=mma("T=32 M=49152 N=3 K=3", "ksplit=1 ctas=24576", *RK), simt="simt T=32 M=49152 N=3 K=3"),
        "row simt mma simt row simt simt", None),
    "row_12": (
        skinny(49152, 12, 12),
        dict(row="row rows=1572864 small=12 K=12 big_operand=v0",
             mma=mma("T=32 M=49152 N=12 K=12", "ksplit=1 ctas=24576", *RK), simt="simt T=32 M=49152 N=12 K=12"),
        "row simt mma simt row simt simt", None),
    "row_16": (
        skinny(49152, 16, 16),
        dict(row="row rows=1572864 small=16 K=16 big_operand=v0",
             mma=mma("T=32 M=49152 N=16 K=16", "ksplit=1 ctas=24576", *RK), simt="simt T=32 M=49152 N=16 K=16"),
        "row simt mma simt row simt simt", None),
    "row_16_k64": (  # the mma kernel's shape: the row kernel only when forced
        skinny(49152, 16, 64),
        dict(row="row rows=1572864 small=16 K=64 big_operand=v0",
             mma=mma("T=32 M=49152 N=16 K=64", "ksplit=1 ctas=24576", *RK), simt="simt T=32 M=49152 N=16 K=64"),
        "mma simt mma mma row mma mma", None),
    "k0": (  # an empty contracted range: vr = beta * vr
        D(T=[(4, 1, 1, 1)], M=[(8, 4, 0, 4)], N=[(8, 0, 4, 32)], K=[(0, 1, 1, 0)]),
        dict(simt="simt T=4 M=8 N=8 K=0"),
        "simt simt simt simt simt simt simt", None),
    "empty": (
        D(T=[(0, 1, 1, 1)], K=[(4, 1, 1, 0)]),
        dict(empty="empty"),
        "empty empty empty empty empty empty empty", None),
}


@pytest.fixture(autouse=True)
def no_tc_overrides(monkeypatch):
    monkeypatch.delenv("SBB_TC_KSPLIT", raising=False)
    monkeypatch.delenv("SBB_TC_PROMOTE", raising=False)


@pytest.mark.parametrize("force", FORCES, ids=[str(f) for f in FORCES])
@pytest.mark.parametrize("name", list(PROBLEMS))
def test_contract_describe(monkeypatch, name, force):
    desc, text, route, route_c64 = PROBLEMS[name]
    if force is None:
        monkeypatch.delenv("SBB_CONTRACT_KERNEL", raising=False)
    else:
        monkeypatch.setenv("SBB_CONTRACT_KERNEL", force)
    for dt in DTYPES:
        path = (route_c64 if dt == sb.C64 and route_c64 else route).split()[FORCES.index(force)]
        want = text[path] if isinstance(text[path], str) else text[path][dt]
        assert sb.contract_describe(desc, dt) == want, (dt, path)
