"""The case matrix of the segmentation conv conformance suite (test_conv_conformance_gpu.py runs it on the device,
test_conv_conformance_cases.py checks on the host that each case lands on the plan, issuer and epilogue it exists for).

Every case names the branch of the kernel it is there for.  The issuer and epilogue a plan takes are restated from the
kernel (issuer() / epi_variant() below), so a planner change that silently moves a case onto another branch fails on a
machine without a GPU."""
from dataclasses import dataclass, field

# ops.FLAG_* and the planner's private A/B flags (api_conv.cu:23-30)
FLAG_FORCE_KD1 = 4
FLAG_NO_FAST_PATH = 8
FLAG_WIDE_N = 16
FLAG_WIDE_ROWS = 32
FLAG_ONE_KH_ROW = 64
FLAG_NO_PING_PONG = 128
KH_SHARED = 256              # kConvFlagKhShared (conv_api.h)
AB_FLAGS = FLAG_FORCE_KD1 | FLAG_NO_FAST_PATH | FLAG_WIDE_N | FLAG_WIDE_ROWS | FLAG_ONE_KH_ROW | FLAG_NO_PING_PONG

# conv_igemm.cuh: enum of ConvIgemmParams::mode
ROW_SHARED, PER_TAP, POINTWISE, UP2, KH_SHARED_MODE = 0, 1, 2, 3, 4
MODE_NAMES = {ROW_SHARED: "row-shared", PER_TAP: "per-tap", POINTWISE: "pointwise", UP2: "k2s2",
              KH_SHARED_MODE: "kh-shared"}

ISSUERS = ("fast<3,4,4>", "fast<3,2,4,nkh=3>", "fast<3,2,4>", "fast<1,4,4>", "fast<1,4,2>", "fast<1,4,1>",
           "lo8<3,4,4>", "lo8<1,4,4>", "general")
EPI_VARIANTS = tuple(range(12))


@dataclass(frozen=True)
class Case:
    name: str
    why: str               # the branch / mode / epilogue variant / shape the case exists for
    D: int
    H: int
    W: int
    c0: int
    c1: int = 0
    cout: int = 64
    kind: int = 0          # 0: 3x3x3 p1, 1: 1x1x1, 2: ConvTranspose3d(k2, s2) (D, H, W: the input grid)
    terms: int = 1
    fmt: int = 0           # 0 fp16, 1 bf16
    out: str = "plain"     # "plain" | "split" ([hi | lo] output) | "lo8" (e4m3 lo plane beside the 16-bit output)
    relu: bool = True
    NT: int = 1
    flags: int = 0
    api: str = "ex"        # "ex": ops.conv3d_igemm_ex | "convt2": ops.convt2_igemm | "obase": ops.conv3d_igemm
    region: tuple = None   # {d_lo, d_cnt, h_lo, h_cnt} (k2s2: on the input grid)
    expect: dict = field(default_factory=dict)   # plan fields (ops.conv_plan_ex keys) the case must land on

    @property
    def ab(self):
        """A/B-flag case: exists only for a debug / comparison flag of the planner."""
        return bool(self.flags & AB_FLAGS)

    @property
    def id(self):
        return self.name


def C(name, why, D, H, W, c0, **kw):
    return Case(name, why, D, H, W, c0, **kw)


# ---------------------------------------------------------------------------------------------------- layer cases
CASES = [
    # ---- issuers (conv_igemm.cu:706-718), reached through real shapes
    C("rs344_fp16", "fast<3,4,4>, row-shared, epilogue 1 (fp16 plain relu)", 5, 4, 128, 64,
      expect=dict(mode=ROW_SHARED, R=5, nchunks=1, row_bytes=128)),
    C("rs344_bf16_relu0", "fast<3,4,4>, row-shared, epilogue 6 (bf16 plain, no relu)", 5, 4, 128, 64, fmt=1,
      relu=False, expect=dict(mode=ROW_SHARED)),
    C("rs_w256_split_relu0", "row-shared at W = 256: two M tiles per row; epilogue 2 (fp16 split, no relu)", 3, 2,
      256, 64, out="split", relu=False, expect=dict(mode=ROW_SHARED, R=3)),
    C("ec1_nkh3", "fast<3,2,4,nkh=3>: ec1's 32-channel three-row stage, 64-byte rows", 5, 4, 128, 32,
      expect=dict(mode=ROW_SHARED, row_bytes=64, nchunks=1)),
    C("ec1_nkh3_bf16_split_relu0", "fast<3,2,4,nkh=3>, epilogue 8 (bf16 split, no relu)", 5, 4, 128, 32, fmt=1,
      out="split", relu=False, expect=dict(mode=ROW_SHARED, row_bytes=64)),
    C("c24_rs324", "fast<3,2,4>: a 24-channel source (k16 = 2, 128-byte rows, TMA zero fill of channels 24-63)",
      5, 4, 128, 24, expect=dict(mode=ROW_SHARED, row_bytes=128, nchunks=1)),
    C("pt144", "fast<1,4,4>, per-tap with kd stacked in threes", 5, 8, 16, 64,
      expect=dict(mode=PER_TAP, kd_per_block=3, nhalf=1, cout_per_half=64)),
    C("pt142_cout128", "fast<1,4,2>: per-tap, 128 output channels in one N split", 5, 8, 16, 64, cout=128,
      expect=dict(mode=PER_TAP, kd_per_block=3, nhalf=1, cout_per_half=128, R=4)),
    C("pw141_cout256", "fast<1,4,1>: pointwise 1x1x1 with a 256-wide N tile", 4, 8, 16, 64, cout=256, kind=1,
      expect=dict(mode=POINTWISE, nhalf=1, cout_per_half=256, R=2)),
    C("pw_bf16_lo8out_relu0", "pointwise, epilogue 10 (bf16 e4m3 lo plane, no relu)", 4, 8, 16, 64, kind=1, fmt=1,
      out="lo8", relu=False, expect=dict(mode=POINTWISE)),
    C("c16_general", "general issuer: a 16-channel source (k16 = 1)", 5, 4, 128, 16,
      expect=dict(mode=ROW_SHARED, row_bytes=128, nchunks=1)),
    C("c8_general", "general issuer, 8-channel source: one 64-channel box, 56 channels of TMA zero fill", 5, 8, 16, 8,
      expect=dict(mode=PER_TAP, nchunks=1)),
    C("cout32_general", "general issuer: cout 32 (per = 8), row-shared", 5, 4, 128, 64, cout=32,
      expect=dict(mode=ROW_SHARED, cout_per_half=32, R=5)),
    C("lo8_rs344", "lo8<3,4,4>: terms 7 row-shared, epilogue 3", 5, 4, 128, 64, terms=7, out="split",
      expect=dict(mode=ROW_SHARED, nchunks=2)),
    C("lo8_pt144_bf16", "lo8<1,4,4>: terms 7 per-tap in bf16 (S = 8), epilogue 7", 5, 8, 16, 64, terms=7, fmt=1,
      expect=dict(mode=PER_TAP, nchunks=2)),
    C("lo8_pt_cout128_general", "general issuer for lo8: per-tap with 128 output channels per half", 5, 8, 16, 64,
      cout=128, terms=7, expect=dict(mode=PER_TAP, cout_per_half=128, R=3)),
    # ---- A/B-flag cases: exist only for the planner's comparison flags
    C("ab_no_fast_path", "A/B kFlagNoFastPath: general issuer on a row-shared layer", 5, 4, 128, 64,
      flags=FLAG_NO_FAST_PATH, expect=dict(mode=ROW_SHARED)),
    C("ab_force_kd1", "A/B kFlagForceKd1: per-tap with one kd per block", 5, 8, 16, 64, flags=FLAG_FORCE_KD1,
      expect=dict(mode=PER_TAP, kd_per_block=1, nblk=27)),
    C("ab_wide_n", "A/B kFlagWideN: 3x3x3 with a 256-wide N tile, one kd per block (fast<1,4,1>)", 3, 8, 16, 64,
      cout=256, flags=FLAG_WIDE_N, expect=dict(mode=PER_TAP, kd_per_block=1, nhalf=1, cout_per_half=256, R=2)),
    C("ab_one_kh_row", "A/B kFlagOneKhRow: ec1 with one kh row per stage (fast<3,2,4>)", 5, 4, 128, 32,
      flags=FLAG_ONE_KH_ROW, expect=dict(mode=ROW_SHARED, row_bytes=64)),
    C("ab_wide_rows", "A/B kFlagWideRows: ec1 with 128-byte zero-filled rows (fast<3,2,4>)", 5, 4, 128, 32,
      flags=FLAG_WIDE_ROWS, expect=dict(mode=ROW_SHARED, row_bytes=128)),
    C("ab_no_ping_pong", "A/B kFlagNoPingPong: k2s2 units on every TMEM column (R = 8)", 2, 8, 16, 64, kind=2,
      flags=FLAG_NO_PING_PONG, expect=dict(mode=UP2, R=8, kd_per_block=1)),
    # ---- modes
    C("up_dc3", "k2s2 at dc3's channels: ping-pong, stationary weights, fast<1,4,2>", 4, 8, 16, 128, cout=128,
      kind=2, expect=dict(mode=UP2, R=2, kd_per_block=4, nblk=2)),
    C("up_dc6", "k2s2 at dc6's channels: ping-pong with R = 1, stationary weights, fast<1,4,1>", 2, 4, 32, 256,
      cout=256, kind=2, expect=dict(mode=UP2, R=1, kd_per_block=8, nblk=4)),
    C("up_bf16_split_relu0", "k2s2, epilogue 8 (bf16 split, no relu)", 2, 8, 16, 64, kind=2, fmt=1, out="split",
      relu=False, expect=dict(mode=UP2, R=4)),
    C("up_convt2_api", "k2s2 through oai_convt2_igemm, 3 tiles", 2, 8, 16, 64, kind=2, NT=3, api="convt2",
      expect=dict(mode=UP2)),
    C("kh32", "kh-shared at tile width 32 (W = 64, 2 x 2 tiles)", 5, 8, 64, 64, flags=KH_SHARED,
      expect=dict(mode=KH_SHARED_MODE, nblk=3)),
    C("kh16", "kh-shared at tile width 16 (W = 16)", 5, 16, 16, 64, flags=KH_SHARED, expect=dict(mode=KH_SHARED_MODE)),
    C("kh8_bf16", "kh-shared at tile width 8 (W = 8), bf16, epilogue 9", 5, 16, 8, 64, flags=KH_SHARED, fmt=1,
      out="split", expect=dict(mode=KH_SHARED_MODE)),
    C("kh_t2", "kh-shared on a split 32-channel source (terms 2: 64 virtual channels)", 4, 8, 64, 32, terms=2,
      flags=KH_SHARED, expect=dict(mode=KH_SHARED_MODE, row_bytes=128, nchunks=1)),
    C("kh_t4_relu0", "kh-shared, terms 4 on two sources, epilogue 0 (fp16 plain, no relu)", 4, 8, 32, 64, c1=64,
      terms=4, relu=False, flags=KH_SHARED, expect=dict(mode=KH_SHARED_MODE, nchunks=3)),
    C("kh_t6_lo8out", "kh-shared, terms 6 (dc2's pattern), epilogue 5 (fp16 e4m3 lo plane)", 4, 8, 32, 128, c1=64,
      terms=6, out="lo8", flags=KH_SHARED, expect=dict(mode=KH_SHARED_MODE, nchunks=4)),
    C("kh_t5_bf16", "kh-shared, terms 5 in bf16 (the first source split)", 4, 8, 32, 64, c1=64, terms=5, fmt=1,
      flags=KH_SHARED, expect=dict(mode=KH_SHARED_MODE, nchunks=3)),
    # ---- term codes 1-7, both formats, one and two sources
    C("t1_2src_fp16", "terms 1 on two sources (the K loop runs over src0 then src1)", 5, 8, 16, 64, c1=64,
      expect=dict(mode=PER_TAP, nchunks=2)),
    C("t1_2src_bf16", "terms 1 on two sources, bf16", 5, 8, 16, 128, c1=256, fmt=1, expect=dict(nchunks=6)),
    C("t2_1src_fp16", "terms 2, one split 32-channel source ([hi | lo] = one 64-channel chunk)", 5, 4, 128, 32,
      terms=2, expect=dict(mode=ROW_SHARED, nchunks=1, row_bytes=128)),
    C("t2_1src_bf16", "terms 2, one split source, bf16, epilogue 9", 5, 8, 16, 64, terms=2, fmt=1, out="split",
      expect=dict(nchunks=2)),
    C("t2_2src_fp16", "terms 2, two split sources", 5, 8, 16, 64, c1=64, terms=2, out="split",
      expect=dict(nchunks=4)),
    C("t2_2src_bf16_relu0", "terms 2, two split sources, bf16, epilogue 6", 5, 8, 16, 64, c1=128, terms=2, fmt=1,
      relu=False, expect=dict(nchunks=6)),
    C("t3_1src_fp16", "terms 3, one source: hi*w_hi + lo*w_hi + hi*w_lo", 5, 8, 16, 32, terms=3, out="split",
      expect=dict(nchunks=2)),
    C("t3_1src_bf16", "terms 3, one source, bf16", 5, 8, 16, 32, terms=3, fmt=1, out="split",
      expect=dict(nchunks=2)),
    C("t3_2src_fp16", "terms 3, two sources", 3, 8, 16, 64, c1=64, terms=3, expect=dict(nchunks=6)),
    C("t3_2src_bf16_relu0", "terms 3, two sources, bf16, epilogue 8", 3, 8, 16, 64, c1=64, terms=3, fmt=1,
      out="split", relu=False, expect=dict(nchunks=6)),
    C("t4_fp16", "terms 4: only the skip source split", 5, 8, 16, 64, c1=128, terms=4, out="split",
      expect=dict(nchunks=5)),
    C("t4_bf16", "terms 4, bf16", 5, 8, 16, 64, c1=128, terms=4, fmt=1, expect=dict(nchunks=5)),
    C("t5_fp16", "terms 5: only the first source split", 5, 8, 16, 128, c1=64, terms=5, out="split",
      expect=dict(nchunks=5)),
    C("t5_bf16_relu0", "terms 5, bf16, no relu", 5, 8, 16, 128, c1=64, terms=5, fmt=1, relu=False,
      expect=dict(nchunks=5)),
    C("t6_dc2_fp16", "terms 6 at dc2's channels (128 + 64, the skip source with an e4m3 lo plane), row-shared",
      5, 4, 128, 128, c1=64, terms=6, out="split", expect=dict(mode=ROW_SHARED, nchunks=4)),
    C("t6_bf16", "terms 6 in bf16 (S = 8), two lo8 chunks, epilogue 11 (bf16 lo8 out)", 5, 8, 16, 64, c1=128,
      terms=6, fmt=1, out="lo8", expect=dict(mode=PER_TAP, nchunks=5)),
    C("t6_bf16_relu0", "terms 6 in bf16, epilogue 6", 5, 4, 128, 128, c1=64, terms=6, fmt=1, relu=False,
      expect=dict(mode=ROW_SHARED, nchunks=4)),
    C("t7_fp16_lo8out_relu0", "terms 7, epilogue 4 (fp16 e4m3 lo plane, no relu)", 5, 8, 16, 64, terms=7,
      out="lo8", relu=False, expect=dict(nchunks=2)),
    C("t7_c512", "terms 7 on a 512-channel source (8 + 8 chunks), 4 N splits", 3, 4, 32, 512, cout=512, terms=7,
      expect=dict(mode=PER_TAP, nhalf=4, cout_per_half=128, nchunks=16)),
    # ---- shapes the planner accepts but the network never launches
    C("c40", "c0 = 40: one chunk, channels 40-63 zero filled (fast<1,4,4>)", 5, 8, 16, 40, expect=dict(nchunks=1)),
    C("c96_bf16", "c0 = 96: second chunk partial (channels 96-127 zero filled)", 5, 8, 16, 96, fmt=1,
      expect=dict(nchunks=2)),
    C("cout96", "cout 96: 96 columns per N split (not a power of two), per = 2", 5, 8, 16, 64, cout=96,
      expect=dict(mode=PER_TAP, nhalf=1, cout_per_half=96, R=5)),
    C("cout192", "cout 192: two N splits of 96", 3, 8, 16, 64, cout=192,
      expect=dict(mode=PER_TAP, nhalf=2, cout_per_half=96)),
    C("cout256", "cout 256: two N splits of 128", 3, 8, 16, 64, cout=256, expect=dict(nhalf=2, cout_per_half=128)),
    C("cout384_bf16", "cout 384: three N splits", 3, 8, 16, 64, cout=384, fmt=1,
      expect=dict(nhalf=3, cout_per_half=128)),
    C("cout512", "cout 512: four N splits (ec7's width)", 3, 8, 16, 64, cout=512,
      expect=dict(nhalf=4, cout_per_half=128)),
    C("nt3", "three tiles per launch", 3, 8, 16, 64, NT=3, out="split"),
    C("d1", "D = 1: one partial accumulator group", 1, 8, 16, 64, expect=dict(R=1)),
    C("d9", "D = 9: R = 8 then a partial group of 1", 9, 4, 128, 64, expect=dict(R=8)),
    C("d18_lo8", "D = 18, terms 7: lo8's equal d groups 6 + 6 + 6", 18, 4, 128, 64, terms=7, expect=dict(R=6)),
    C("obase_slice", "oai_conv3d_igemm writing channels 64-127 of a 192-channel tensor (obase, osW > cout)",
      3, 8, 16, 64, api="obase"),
]

# ---------------------------------------------------------------------------------------------------- region cases
REGION_CASES = [
    C("reg_dc4", "per-tap with TH = 2 at dc4's production grid: rows 6 and 57 outside the region are written", 16, 64,
      64, 128, cout=128, region=(3, 10, 7, 50), expect=dict(mode=PER_TAP)),
    C("reg_row_shared", "row-shared region", 5, 8, 128, 64, region=(1, 3, 2, 5), out="split",
      expect=dict(mode=ROW_SHARED)),
    C("reg_k2s2", "k2s2 region on the input grid (written set: its 2x image)", 4, 8, 16, 128, cout=128, kind=2,
      region=(1, 2, 3, 4), expect=dict(mode=UP2)),
    C("reg_kh_shared", "kh-shared region whose last tile is clamped into the grid (tiles at rows 9 and 12, TH = 4)",
      5, 16, 64, 64, flags=KH_SHARED, region=(0, 5, 9, 6), expect=dict(mode=KH_SHARED_MODE)),
    C("reg_kh_shared_low", "kh-shared region starting at row 0 whose rows end before the tile does", 5, 16, 64, 64,
      flags=KH_SHARED, region=(1, 3, 0, 5), out="split"),
    C("reg_h1", "h_cnt = 1", 5, 8, 16, 64, region=(2, 1, 5, 1)),
    C("reg_far_edges", "a region touching the grid's far d and h edges (TH = 4)", 5, 8, 32, 64, region=(3, 2, 5, 3)),
    C("reg_lo8_bf16", "terms 7 bf16 region with an e4m3 lo output plane", 6, 8, 16, 64, terms=7, fmt=1, out="lo8",
      region=(1, 4, 2, 3)),
]

# ---------------------------------------------------------------------------------------------------- w-box cases
# oai_conv3d_igemm_box: region = (d_lo, d_cnt, h_lo, h_cnt, w_lo, w_cnt) on a kh-shared layer; 32-wide tiles over the
# largest multiple of 32 columns, then an 8-wide strip ending at w_lo + w_cnt (api_conv.cu: conv_run_w_box)
BOX_CASES = [
    C("box_dc2_98", "dc2's 98-column box (96 + an overlapping 8-wide strip), terms 6, e4m3 lo output", 3, 16, 128, 128,
      c1=64, terms=6, out="lo8", flags=KH_SHARED, region=(0, 3, 2, 12, 15, 98), api="box"),
    C("box_dc1_96", "dc1's 96-column box, terms 7", 3, 16, 128, 64, terms=7, flags=KH_SHARED,
      region=(1, 2, 3, 11, 16, 96), api="box"),
    C("box_w1", "w_cnt = 1: the strip alone, one column", 3, 16, 64, 64, flags=KH_SHARED, region=(0, 3, 4, 5, 5, 1),
      api="box"),
    C("box_w7", "w_cnt = 7", 3, 16, 64, 64, flags=KH_SHARED, fmt=1, region=(0, 2, 0, 16, 20, 7), api="box"),
    C("box_w8", "w_cnt = 8: one 8-wide strip", 3, 16, 64, 64, flags=KH_SHARED, region=(1, 2, 6, 7, 3, 8), api="box"),
    C("box_w33", "w_cnt = 33: 32 columns and a strip overlapping 7 of them", 3, 16, 64, 64, flags=KH_SHARED,
      out="split", region=(0, 3, 1, 9, 10, 33), api="box"),
    C("box_w40_end", "w_cnt = 40 ending at W: 32 columns and an 8-wide strip on the grid's last columns", 3, 16, 64,
      64, flags=KH_SHARED, region=(0, 3, 5, 11, 24, 40), api="box"),
]

ALL_CASES = CASES + REGION_CASES + BOX_CASES


def kh_tile_width(H, W, h_cnt, w_cnt):
    """api_conv.cu: kh_tile_width -- the width with the fewest M tiles over the box, the widest on a tie."""
    tw, best = 32, 0
    for t in (32, 16, 8):
        if t > W or 128 // t > H:
            continue
        n = -(-w_cnt // t) * -(-h_cnt // (128 // t))
        if best == 0 or n < best:
            best, tw = n, t
    return tw


def region_rows(case):
    """Rows (on the output grid) a region launch writes: whole M tiles (include/oai_b200.h, oai_conv3d_igemm_region)."""
    _, _, h_lo, h_cnt = case.region[:4]
    if case.flags & KH_SHARED:
        TH = 128 // kh_tile_width(case.H, case.W, h_cnt, case.W)
        return min(h_lo, case.H - TH), min(h_lo + -(-h_cnt // TH) * TH, case.H)
    TH = 128 // min(case.W, 128)
    up = 2 if case.kind == 2 else 1
    return up * (h_lo // TH * TH), up * min(-(-(h_lo + h_cnt) // TH) * TH, case.H)


# ---------------------------------------------------------------------------------------------------- production replay
# Mirror of the segmentation network's conv layers (oai_analysis_2_b200/csrc/seg_net.cu:41-48, kLayers; ec0 runs in
# the stem kernel, dc0 in dc1's fused head): name, kind ('c' conv, 't' transposed k3 = conv, 'u' k2s2), cin, cout,
# level of the INPUT grid, channels of the first source of a concatenating layer; then the packed weight size in 16-byte
# units at the production tile under the mixed plan (seg_layer_terms(1)), checked by test_conv_conformance_cases.py.
PROD_TILE = (32, 128, 128)      # z, y, x
PROD_OVERLAP = (8, 16, 16)
PROD_NT = 2
SEG_LAYERS = [
    ("ec1", "c", 32, 64, 0, 0, 6912), ("ec2", "c", 64, 64, 1, 0, 13824), ("ec3", "c", 64, 128, 1, 0, 27648),
    ("ec4", "c", 128, 128, 2, 0, 55296), ("ec5", "c", 128, 256, 2, 0, 110592), ("ec6", "c", 256, 256, 3, 0, 221184),
    ("ec7", "c", 256, 512, 3, 0, 442368), ("dc9", "u", 512, 512, 3, 0, 262144), ("dc8", "t", 768, 256, 2, 512, 663552),
    ("dc7", "t", 256, 256, 2, 0, 221184), ("dc6", "u", 256, 256, 2, 0, 65536), ("dc5", "t", 384, 128, 1, 256, 165888),
    ("dc4", "t", 128, 128, 1, 0, 55296), ("dc3", "u", 128, 128, 1, 0, 16384), ("dc2", "t", 192, 64, 0, 128, 55297),
    ("dc1", "t", 64, 64, 0, 0, 27649),
]
KH_SHARED_LAYERS = ("dc2", "dc1")   # seg_net.cu: dc2 and dc1 run kh-shared over their needed (h, w) box
FIRST_REGION_LAYER = "dc9"          # seg_net.cu: layers from dc9 on compute only their needed region


def production_cases(terms17, fmt, regions):
    """The tcgen05 launches of oai_seg_forward at the production tile as cases: terms17 = seg_layer_terms(...) (index
    0 is the stem), regions = ops.seg_needed_regions(PROD_TILE, PROD_OVERLAP) (inclusive lo z,y,x, hi z,y,x per layer
    ec0..dc1).  Storage follows seg_net.cu's tensor plan for these plans: a tensor read by a terms 6 / 7 layer carries an
    e4m3 lo plane (ec1's output, the skip of dc2, and dc2's output), every other one is plain."""
    names = [L[0] for L in SEG_LAYERS]
    out = []
    for i, (name, kind, cin, cout, level, c_first, _) in enumerate(SEG_LAYERS):
        D, H, W = (t >> level for t in PROD_TILE)
        c0 = c_first or cin
        terms = terms17[i + 1]
        consumers = {"ec1": "dc2", "dc2": "dc1"}   # the lo8-capable tensors and the layer reading them
        lo8_out = name in consumers and terms17[names.index(consumers[name]) + 1] in (6, 7)
        lo, hi = regions[i + 1][:3], regions[i + 1][3:]
        region = None
        api = "ex"
        flags = 0
        if names.index(name) >= names.index(FIRST_REGION_LAYER):
            region = (int(lo[0]), int(hi[0] - lo[0] + 1), int(lo[1]), int(hi[1] - lo[1] + 1))
        if name in KH_SHARED_LAYERS:
            flags = KH_SHARED
            api = "box"
            region = region + (int(lo[2]), int(hi[2] - lo[2] + 1))
        out.append(Case(f"prod_{name}_t{terms}_f{fmt}", f"oai_seg_forward's {name} launch", D, H, W, c0,
                        c1=cin - c0, cout=cout, kind=2 if kind == "u" else 0, terms=terms, fmt=fmt,
                        out="lo8" if lo8_out else "plain", NT=PROD_NT, flags=flags, api=api, region=region))
    return out


# ---------------------------------------------------------------------------------------------------- restatements
def split_src(terms, src):
    """api_conv.cu:53-55: sources a term code reads as [hi | lo] planes."""
    return terms in (2, 3) or (terms == 4 and src == 1) or (terms == 5 and src == 0)


def k16_steps(case):
    """api_conv.cu (make_plan): K=16 steps per chunk."""
    c0v = 2 * case.c0 if split_src(case.terms, 0) else case.c0
    return (1 if c0v <= 16 else 2) if (case.c1 == 0 and c0v <= 32) else 4


def kh_rows(case, plan):
    """api_conv.cu (make_plan): kh rows per A stage (3: ec1's three-row stage)."""
    off = FLAG_ONE_KH_ROW | FLAG_NO_FAST_PATH | 2
    return 3 if (plan["mode"] == ROW_SHARED and plan["row_bytes"] == 64 and plan["nchunks"] == 1
                 and not case.flags & off) else 1


def issuer(case, plan):
    """conv_igemm.cu:696-718: the MMA issuer specialisation a launch of this plan takes."""
    if case.flags & (FLAG_NO_FAST_PATH | 2):
        return "general"
    nkw = 3 if plan["mode"] in (ROW_SHARED, KH_SHARED_MODE) else 1
    k16 = k16_steps(case)
    per = max(1, 256 // plan["cout_per_half"])
    if case.terms in (6, 7):
        if k16 == 4 and per == 4:
            return f"lo8<{nkw},4,4>"
        return "general"
    if nkw == 3 and k16 == 4 and per == 4:
        return "fast<3,4,4>"
    if nkw == 3 and k16 == 2 and per == 4:
        return "fast<3,2,4,nkh=3>" if kh_rows(case, plan) == 3 else "fast<3,2,4>"
    if nkw == 1 and k16 == 4 and per in (4, 2, 1):
        return f"fast<1,4,{per}>"
    return "general"


def epi_variant(case):
    """conv_igemm.cu:726: the compiled epilogue variant."""
    return (6 if case.fmt else 0) + (4 if case.out == "lo8" else 2 if case.out == "split" else 0) + int(case.relu)


def plan_of(ops, case):
    return ops.conv_plan_ex(case.D, case.H, case.W, case.c0, case.c1, case.cout, case.kind, case.terms, case.flags)
