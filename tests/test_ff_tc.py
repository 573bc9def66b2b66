"""Tensor-core Montgomery reduction (zk-email-verify_b200/csrc/ff_tc.cuh) without a GPU:
  * the host table builder (constant matrix in mma fragment order, Barrett reciprocal) against Python integers;
  * a lane-level model of the device routine - ldmatrix / mma.m16n8k32.u8 fragment index maps, column folding,
    stmatrix hand-over, 14-bit Barrett tail - against a*b/2^256 mod p for both BN254 fields, including the bounds
    the device code relies on (column sums < 2^21, r' < 2^268, r' - q p < 2p).
The device routine itself is checked on the GPU against the integer product (scripts/tc_product.cu, 2 M products) and
through the bit-exact proof test test_tensor_core_reduction_h_msm_bit_exact."""
import os
import random
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "zk-email-verify_b200", "csrc")
FQ = 21888242871839275222246405745257275088696311157297823662689037894645226208583
FR = 21888242871839275222246405745257275088548364400416034343698204186575808495617
R = 1 << 256


def _consts(p):
    rinv = pow(R, -1, p)
    return [(pow(2, 8 * j, p) * rinv) % p for j in range(32)], (1 << 285) // p


def _byte_of_column(nt, col):          # column `col` of n-tile `nt` carries this byte of C_j (ff_tc.cuh: tc_build_table)
    return 8 * (col >> 1) + 2 * nt + (col & 1)


def _expected_bfrag(p):
    C, _ = _consts(p)
    out = []
    for lane in range(32):
        g, t = lane >> 2, lane & 3
        row = []
        for nt in range(4):
            byte = _byte_of_column(nt, g)
            for half in range(2):
                w = 0
                for i in range(4):
                    w |= ((C[16 * half + 4 * t + i] >> (8 * byte)) & 0xff) << (8 * i)
                row.append(w)
        out.append(row)
    return out


@pytest.fixture(scope="module")
def dump_binary(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("tc") / "tc_table_dump")
    nvcc = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    subprocess.check_call([nvcc, "-O1", "-I", CSRC, "-o", exe, os.path.join(ROOT, "tests", "tc_table_dump.cu")])
    return exe


@pytest.mark.parametrize("p", [FQ, FR])
def test_table_builder_matches_python(dump_binary, p):
    limbs = ["%08x" % ((p >> (32 * i)) & 0xffffffff) for i in range(8)]
    lines = subprocess.check_output([dump_binary] + limbs, text=True).split("\n")
    assert int(lines[0], 16) == (1 << 285) // p
    got = [[int(x, 16) for x in lines[1 + lane].split()] for lane in range(32)]
    assert got == _expected_bfrag(p)


def _model(p, a_list, b_list):
    """32 lanes, one product each, following redc_n<1> step by step."""
    C, mu = _consts(p)
    nmod = R - p
    T = [a * b for a, b in zip(a_list, b_list)]
    rows = {lane: [((T[lane] & (R - 1)) >> (8 * j)) & 0xff for j in range(32)] for lane in range(32)}     # STS.128 x 2
    planes = [[[0] * 4 for _ in range(32)] for _ in range(3)]        # [p][element][t]: the stmatrix hand-over rows
    for lane in range(32):
        g, t = lane >> 2, lane & 3
        for mt in range(2):
            # ldmatrix.x4: a0 = row g bytes 4t.., a1 = row g + 8, a2 = row g bytes 16 + 4t.., a3 = row g + 8 (rows of tile mt)
            def dot(row, nt, col):
                byte = _byte_of_column(nt, col)
                return sum(rows[16 * mt + row][k] * ((C[k] >> (8 * byte)) & 0xff) for k in range(32))
            for h in range(2):
                s = [dot(g + 8 * h, b >> 1, 2 * t + (b & 1)) for b in range(8)]     # d[nt][2h + c]: row g + 8h, column 2t + c
                assert max(s) < 1 << 21
                y = [s[2 * c] + (s[2 * c + 1] << 8) for c in range(4)]
                assert max(y) < 1 << 30
                lo, mid, hi = (y[1] << 16) & 0xffffffff, ((y[1] >> 16) | (y[3] << 16)) & 0xffffffff, y[3] >> 16
                w0 = y[0] + lo
                w1 = y[2] + mid + (w0 >> 32)
                w2 = hi + (w1 >> 32)
                k = 2 * mt + h                                   # slot k <-> element of lane 8k + g
                planes[0][8 * k + g][t], planes[1][8 * k + g][t], planes[2][8 * k + g][t] = w0 & 0xffffffff, w1 & 0xffffffff, w2
    res = []
    for lane in range(32):
        val = sum((planes[0][lane][t] | (planes[1][lane][t] << 32) | (planes[2][lane][t] << 64)) << (64 * t) for t in range(4))
        rp = val + (T[lane] >> 256)
        assert rp < 1 << 268
        x = rp >> 240
        q = (x * mu) >> 45
        r = ((rp & (R - 1)) + q * nmod) & (R - 1)
        assert r < 2 * p
        res.append(r - p if r >= p else r)
    return res


@pytest.mark.parametrize("p", [FQ, FR])
def test_lane_model_equals_montgomery_product(p):
    rng = random.Random(7)
    rinv = pow(R, -1, p)
    for trial in range(6):
        a = [rng.randrange(p) for _ in range(32)]
        b = [rng.randrange(p) for _ in range(32)]
        if trial == 0:
            a[0] = b[0] = p - 1
            a[1] = 0
            a[2] = b[2] = 1
            a[3] = b[3] = R - 1                                  # unreduced operands: still the right residue
        assert _model(p, a, b) == [(x * y * rinv) % p for x, y in zip(a, b)]
