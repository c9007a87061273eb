"""Which copy kernel variant a box takes, examined on the host (`sbk_permute_describe` plans and never
launches, so no device is needed).  Pins the classification (zero / raw move / typed), the widening of
the element, the tile budget of every path and the describe strings themselves, byte for byte."""
import pytest

import superbblas_b200 as sb

D = sb.box_desc
# reversed strides over nine extent-2 dims: nothing merges, so the copy needs more than one launch
NINE = ([2] * 9, [2 ** k for k in range(9)], [2 ** (8 - k) for k in range(9)])

CASES = [
    # (box, dtype_src, dtype_dst, alpha, add, description)
    (D([8, 8, 4], [0, 0, 0], [1, 8, 64]), sb.C128, sb.C128, 0, False,
     "zero es=16 tile=256 ntiles=1"),
    (D([6, 5], [0, 0], [1, 6]), sb.C64, sb.C64, 0, False,
     "zero es=16 tile=15 ntiles=1"),
    (D([6, 5], [0, 0], [1, 6]), sb.C64, sb.C64, 0, True,   # adding zero: nothing to do
     ""),
    (D([64, 48], [1, 64], [48, 1]), sb.F64, sb.F64, 2j, False,  # a real type ignores the imaginary part
     "zero es=16 tile=1536 ntiles=1"),
    (D([64, 32], [1, 64], [1, 64]), sb.F32, sb.F32, 1, False,
     "move direct es=16 tile=512 ntiles=1 run_dst=8192B run_src=8192B nd=1"),
    (D([6, 32], [1, 6], [1, 8]), sb.F64, sb.F64, 1, False,
     "move direct es=16 tile=96 ntiles=1 run_dst=48B run_src=1536B nd=2"),
    (D([2, 64, 64], [1, 2, 128], [1, 128, 2]), sb.C64, sb.C64, 1, False,  # complex float widened to 16 B
     "move tiled es=16 tile=2048 ntiles=2 run_dst=512B run_src=32768B nd=2"),
    (D([8, 8, 8, 16, 4, 3], [1, 8, 64, 512, 8192, 32768], [16384, 2048, 256, 16, 4, 1]), sb.C128, sb.C128,
     1, False, "move tiled es=16 tile=1536 ntiles=64 run_dst=48B run_src=8192B nd=6"),
    (D([256, 256], [1, 256], [256, 1]), sb.F32, sb.F32, 1, False,  # 16 slots per thread
     "move tiled es=4 tile=4096 ntiles=16 run_dst=128B run_src=512B nd=2"),
    (D([256, 256], [1, 256], [256, 1]), sb.F64, sb.F64, 1, False,
     "move tiled es=8 tile=4096 ntiles=16 run_dst=512B run_src=512B nd=2"),
    (D([64, 48], [1, 64], [48, 1]), sb.I32, sb.I32, 1, False,
     "move tiled es=4 tile=3072 ntiles=1 run_dst=12288B run_src=12288B nd=2"),
    (D([64, 48], [1, 64], [48, 1]), sb.F64, sb.F64, 1 + 2j, False,
     "move tiled es=8 tile=3072 ntiles=1 run_dst=24576B run_src=24576B nd=2"),
    (D([32, 16, 4], [1, 32, 512], [1, 32, 512], rot=1), sb.C128, sb.C128, 1, False,
     "move direct es=16 tile=2048 ntiles=1 run_dst=512B run_src=512B nd=2"),
    (D([32, 16, 4], [1, 32, 512], [1, 32, 512], rot=3), sb.F32, sb.F32, 1, False,  # rot 3: no widening
     "move direct es=4 tile=2048 ntiles=1 run_dst=128B run_src=128B nd=2"),
    (D([64, 32], [1, 64], [1, 64]), sb.C128, sb.C64, 2, True,
     "typed direct es=16->8 tile=2048 ntiles=1 scale=1 add=1"),
    (D([64, 32], [1, 64], [1, 64]), sb.F32, sb.F64, 1, False,
     "typed direct es=4->8 tile=2048 ntiles=1 scale=0 add=0"),
    (D([64, 48], [1, 64], [48, 1]), sb.C64, sb.C128, 0.5 - 1j, True,
     "typed tiled es=8->16 tile=1536 ntiles=2 scale=1 add=1"),
    (D([64, 48], [1, 64], [48, 1]), sb.F64, sb.F64, -1, False,
     "typed tiled es=8->8 tile=1536 ntiles=2 scale=1 add=0"),
    (D([64, 48], [1, 64], [48, 1]), sb.C64, sb.C64, 2j, False,  # a complex type does not
     "typed tiled es=8->8 tile=1536 ntiles=2 scale=1 add=0"),
    (D(*NINE), sb.F64, sb.F64, 1, False,
     "move tiled es=8 tile=64 ntiles=4 run_dst=512B run_src=8B nd=8"),
    (D(*NINE), sb.F64, sb.F32, 3, True,
     "typed tiled es=8->4 tile=64 ntiles=4 scale=1 add=1"),
    (D([0, 4], [1, 0], [1, 0]), sb.F64, sb.F64, 1, False,
     "empty"),
]


@pytest.mark.parametrize("box,dt0,dt1,alpha,add,want", CASES, ids=[str(i) for i in range(len(CASES))])
def test_permute_describe(box, dt0, dt1, alpha, add, want):
    assert sb.permute_describe(box, dt0, dt1, alpha, add) == want
