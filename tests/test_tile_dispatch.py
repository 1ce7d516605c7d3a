"""Workspace queries and tile-path choice of the forward and training entry points.

Callers size buffers with the workspace queries, some of them baked into CUDA graphs, so their values are API.
The CPU part evaluates ncf_forward_workspace_bytes, ncf_train_workspace_bytes, ncf_eval_workspace_bytes and
ncf_recommend_workspace_bytes over GRID and compares them with WORKSPACE. The queries read only the model struct
and the environment: they run without a GPU on a struct of fake 256-byte-aligned pointers, and the SM count
falls back to 148, the B200's.

The GPU part runs ncf_forward and ncf_train_step_grads at each cheap grid point B, and at the grid point below
it, with a workspace of exactly the size queried for B followed by a guard band. It checks ncf_last_tile_path()
against PATHS, that the guard band is intact, and that a training call with one byte less is refused.

Both tables were recorded from a build of commit 5aa5552, the last commit before the tile-path choice moved into
one function: `python tests/test_tile_dispatch.py` prints WORKSPACE and, on a B200, `... --paths` prints PATHS.
A row is listed only where it differs from the row it falls back to (see _expected).
"""
import ctypes
import os
import sys
from pathlib import Path

import pytest

gpu = pytest.mark.gpu

MODELS = {"GMF": 0, "MLP": 1, "NeuMF": 2}
FS = (5, 8, 16, 32, 64, 128)
LS = (1, 2, 3, 4)
BS = (1, 256, 2048, 2049, 8191, 8192, 65536, 300_000)
GRID = [(mt, f, L) for mt in MODELS for f in FS for L in LS]
# variant -> (environment, byte offset of every tower weight from its 256-byte-aligned address)
VARIANTS = {
    "base": ({}, 0),
    "misaligned": ({}, 4),   # neither the thread-per-sample nor the layer-per-launch kernel takes the model
    "umma_off": ({"NCF_UMMA_DISABLE": "1"}, 0),
    "umma_min_b1": ({"NCF_UMMA_MIN_B": "1"}, 0),
}
QUERIES = ("fwd", "train", "eval", "rec")
EVAL_C = 100            # eval query: n = max(1, B // 100) users of 100 candidates
REC_ITEMS, REC_K = 999, 10   # recommend query: max(1, B // 999) users of a 999-item catalog (user_div = 999)
NCF_ERR_WORKSPACE = -3

WORKSPACE = """
base GMF 5 1 fwd 0 0 0 0 0 0 0 0
base GMF 5 1 train 256 256 256 256 256 256 256 256
base GMF 5 1 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 5 1 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 5 2 fwd 0 0 0 0 0 0 0 0
base GMF 5 2 train 256 256 256 256 256 256 256 256
base GMF 5 2 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 5 2 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 5 3 fwd 0 0 0 0 0 0 0 0
base GMF 5 3 train 256 256 256 256 256 256 256 256
base GMF 5 3 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 5 3 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 5 4 fwd 0 0 0 0 0 0 0 0
base GMF 5 4 train 256 256 256 256 256 256 256 256
base GMF 5 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 5 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 8 1 fwd 0 0 0 0 0 0 0 0
base GMF 8 1 train 256 256 256 256 256 256 256 256
base GMF 8 1 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 8 1 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 8 2 fwd 0 0 0 0 0 0 0 0
base GMF 8 2 train 256 256 256 256 256 256 256 256
base GMF 8 2 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 8 2 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 8 3 fwd 0 0 0 0 0 0 0 0
base GMF 8 3 train 256 256 256 256 256 256 256 256
base GMF 8 3 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 8 3 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 8 4 fwd 0 0 0 0 0 0 0 0
base GMF 8 4 train 256 256 256 256 256 256 256 256
base GMF 8 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 8 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 16 1 fwd 0 0 0 0 0 0 0 0
base GMF 16 1 train 256 256 256 256 256 256 256 256
base GMF 16 1 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 16 1 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 16 2 fwd 0 0 0 0 0 0 0 0
base GMF 16 2 train 256 256 256 256 256 256 256 256
base GMF 16 2 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 16 2 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 16 3 fwd 0 0 0 0 0 0 0 0
base GMF 16 3 train 256 256 256 256 256 256 256 256
base GMF 16 3 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 16 3 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 16 4 fwd 0 0 0 0 0 0 0 0
base GMF 16 4 train 256 256 256 256 256 256 256 256
base GMF 16 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 16 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 32 1 fwd 0 0 0 0 0 0 0 0
base GMF 32 1 train 256 256 256 256 256 256 256 256
base GMF 32 1 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 32 1 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 32 2 fwd 0 0 0 0 0 0 0 0
base GMF 32 2 train 256 256 256 256 256 256 256 256
base GMF 32 2 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 32 2 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 32 3 fwd 0 0 0 0 0 0 0 0
base GMF 32 3 train 256 256 256 256 256 256 256 256
base GMF 32 3 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 32 3 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 32 4 fwd 0 0 0 0 0 0 0 0
base GMF 32 4 train 256 256 256 256 256 256 256 256
base GMF 32 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 32 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 64 1 fwd 0 0 0 0 0 0 0 0
base GMF 64 1 train 256 256 256 256 256 256 256 256
base GMF 64 1 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 64 1 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 64 2 fwd 0 0 0 0 0 0 0 0
base GMF 64 2 train 256 256 256 256 256 256 256 256
base GMF 64 2 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 64 2 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 64 3 fwd 0 0 0 0 0 0 0 0
base GMF 64 3 train 256 256 256 256 256 256 256 256
base GMF 64 3 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 64 3 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 64 4 fwd 0 0 0 0 0 0 0 0
base GMF 64 4 train 256 256 256 256 256 256 256 256
base GMF 64 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 64 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 128 1 fwd 0 0 0 0 0 0 0 0
base GMF 128 1 train 256 256 256 256 256 256 256 256
base GMF 128 1 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 128 1 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 128 2 fwd 0 0 0 0 0 0 0 0
base GMF 128 2 train 256 256 256 256 256 256 256 256
base GMF 128 2 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 128 2 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 128 3 fwd 0 0 0 0 0 0 0 0
base GMF 128 3 train 256 256 256 256 256 256 256 256
base GMF 128 3 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 128 3 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base GMF 128 4 fwd 0 0 0 0 0 0 0 0
base GMF 128 4 train 256 256 256 256 256 256 256 256
base GMF 128 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
base GMF 128 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base NeuMF 5 1 fwd 0 0 0 0 0 0 0 0
base NeuMF 5 1 train 512 5376 41216 41472 164096 164096 1310976 6000384
base NeuMF 5 1 eval 768 1280 8448 8448 32768 32768 262400 1200384
base NeuMF 5 1 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base NeuMF 5 2 fwd 0 0 0 0 0 0 0 0
base NeuMF 5 2 train 512 25856 205056 205312 819456 819456 6553856 30000384
base NeuMF 5 2 eval 768 1280 8448 8448 32768 32768 262400 1200384
base NeuMF 5 2 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base NeuMF 5 3 fwd 0 0 0 0 0 0 0 0
base NeuMF 5 3 train 768 66816 532736 533248 2129920 2130176 17039616 78000384
base NeuMF 5 3 eval 768 1280 8448 8448 32768 32768 262400 1200384
base NeuMF 5 3 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base NeuMF 5 4 fwd 0 0 0 0 0 0 0 0
base NeuMF 5 4 train 1024 148736 1188096 1188864 4751104 4751616 38011136 174000384
base NeuMF 5 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
base NeuMF 5 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
base NeuMF 8 1 fwd 2048 2048 2048 2048 2048 2048 2048 2048
base NeuMF 8 1 train 2304 2304 2304 2304 2304 2304 2304 2304
base NeuMF 8 1 eval 2816 3328 10496 10496 34816 34816 264448 1202432
base NeuMF 8 1 rec 14592 14592 26624 26624 98304 98304 781824 3598848
base NeuMF 8 2 fwd 10240 10240 10240 10240 10240 10240 10240 10240
base NeuMF 8 2 train 10496 10496 10496 10496 10496 10496 10496 10496
base NeuMF 8 2 eval 11008 11520 18688 18688 43008 43008 272640 1210624
base NeuMF 8 2 rec 22784 22784 34816 34816 106496 106496 790016 3607040
base NeuMF 8 3 fwd 43008 43008 43008 43008 43008 43008 43008 43008
base NeuMF 8 3 train 43264 43264 43264 43264 43264 43264 43264 43264
base NeuMF 8 3 eval 43776 44288 51456 51456 75776 75776 305408 1243392
base NeuMF 8 3 rec 55552 55552 67584 67584 139264 139264 822784 3639808
base NeuMF 8 4 fwd 174080 174080 174080 174080 174080 174080 174080 174080
base NeuMF 8 4 train 174336 174336 174336 174336 174336 174336 174336 174336
base NeuMF 8 4 eval 174848 175360 182528 182528 206848 206848 436480 1374464
base NeuMF 8 4 rec 186624 186624 198656 198656 270336 270336 953856 3770880
base NeuMF 16 1 fwd 8192 16384 131072 131072 131072 131072 131072 131072
base NeuMF 16 1 train 8448 8448 8448 8448 8448 8448 8448 8448
base NeuMF 16 1 eval 8960 14080 136448 136448 163840 163840 393472 1331456
base NeuMF 16 1 rec 76544 76544 152576 152576 227328 227328 910848 3727872
base NeuMF 16 2 fwd 40960 49152 393216 393216 393216 393216 393216 393216
base NeuMF 16 2 train 41216 41216 41216 41216 41216 41216 41216 41216
base NeuMF 16 2 eval 41728 42240 392448 392448 425984 425984 655616 1593600
base NeuMF 16 2 rec 204544 204544 408320 408320 489472 489472 1172992 3990016
base NeuMF 16 3 fwd 172032 172032 917504 917504 917504 917504 917504 917504
base NeuMF 16 3 train 172288 172288 172288 172288 172288 172288 172288 172288
base NeuMF 16 3 eval 172800 173312 904448 904448 950272 950272 1179904 2117888
base NeuMF 16 3 rec 460288 460288 919808 919808 1013760 1013760 1697280 4514304
base NeuMF 16 4 fwd 696320 696320 1966080 1966080 1966080 1966080 1966080 1966080
base NeuMF 16 4 train 696576 696576 696576 696576 696576 696576 696576 696576
base NeuMF 16 4 eval 697088 697600 1928448 1928448 1998848 1998848 2228480 3166464
base NeuMF 16 4 rec 971776 971776 1942784 1942784 2062336 2062336 2745856 5562880
base NeuMF 32 1 fwd 32768 32768 262144 262144 262144 262144 262144 262144
base NeuMF 32 1 train 33024 33024 33024 33024 33024 1081856 8421888 38433280
base NeuMF 32 1 eval 33536 34048 264448 264448 294912 294912 524544 1462528
base NeuMF 32 1 rec 140544 140544 280320 280320 358400 358400 1041920 3858944
base NeuMF 32 2 fwd 163840 163840 786432 786432 786432 2261504 16941568 67273216
base NeuMF 32 2 train 164096 164096 164096 164096 164096 5407232 42107392 192164352
base NeuMF 32 2 eval 164608 165120 776448 776448 819200 819200 17194752 68473600
base NeuMF 32 2 rec 396288 396288 791808 791808 882688 882688 17567488 70766080
base NeuMF 32 3 fwd 688128 688128 1835008 1835008 1835008 6980096 51020288 202015232
base NeuMF 32 3 train 688384 688384 688384 688384 688384 14320128 109740544 499888640
base NeuMF 32 3 eval 688896 689408 1800448 1800448 1867776 1867776 51255040 203215616
base NeuMF 32 3 rec 907776 907776 1814784 1814784 1931264 1931264 51338496 205300224
base NeuMF 32 4 fwd 2785280 2785280 3932160 3932160 3932160 17465856 120226304 472547840
base NeuMF 32 4 train 2785536 2785536 2785536 2785536 2785536 33194496 246055424 1116385792
base NeuMF 32 4 eval 2786048 2786560 3848448 3848448 3964928 3964928 120424192 473748224
base NeuMF 32 4 rec 2797824 2797824 3860736 3860736 4028416 4028416 119929088 475417088
base NeuMF 64 1 fwd 131072 131072 524288 524288 524288 524288 524288 524288
base NeuMF 64 1 train 131328 131328 131328 131328 131328 2228736 16908800 76931584
base NeuMF 64 1 eval 131840 132352 520448 520448 557056 557056 786688 1724672
base NeuMF 64 1 rec 268288 268288 536064 536064 620544 620544 1304064 4121088
base NeuMF 64 2 fwd 655360 655360 1572864 1572864 1572864 4850176 34210304 134873600
base NeuMF 64 2 train 655616 655616 655616 655616 655616 11141632 84541952 384655872
base NeuMF 64 2 eval 656128 656640 1544448 1544448 1605632 1605632 34454272 136073984
base NeuMF 64 2 rec 779776 779776 1559040 1559040 1669120 1669120 34682368 138262528
base NeuMF 64 3 fwd 2752512 2752512 3670016 3670016 3670016 15335936 103416320 405406208
base NeuMF 64 3 train 2752768 2752768 2752768 2752768 2752768 30016000 220856832 1001153024
base NeuMF 64 3 eval 2753280 2753792 3592448 3592448 3702784 3702784 103623424 406606592
base NeuMF 64 3 rec 2765056 2765056 3604992 3604992 3766272 3766272 103272960 408379392
base NeuMF 64 4 fwd 3840 983040 7864320 7864320 7864320 7864320 7864320 7864320
base NeuMF 64 4 train 7680 1900800 15204608 15212032 60810240 60817664 486539520 2227200256
base NeuMF 64 4 eval 384768 769280 7688448 7688448 7897088 7897088 8126720 9064704
base NeuMF 64 4 rec 3848704 3848704 7696896 7696896 7960576 7960576 8644096 11461120
base NeuMF 128 1 fwd 524288 524288 1048576 1048576 1048576 1048576 1048576 1048576
base NeuMF 128 1 train 524544 524544 524544 524544 524544 4719104 34079232 154124800
base NeuMF 128 1 eval 525056 525568 1032448 1032448 1081344 1081344 1310976 2248960
base NeuMF 128 1 rec 536832 536832 1047552 1047552 1144832 1144832 1828352 4645376
base NeuMF 128 2 fwd 2621440 2621440 3145728 3145728 3145728 11010560 69730816 271057408
base NeuMF 128 2 train 2621696 2621696 2621696 2621696 2621696 23593472 170394112 770621952
base NeuMF 128 2 eval 2622208 2622720 3080448 3080448 3178496 3178496 69956352 272257792
base NeuMF 128 2 rec 2633984 2633984 3093504 3093504 3241984 3241984 69895168 274238464
base NeuMF 128 3 fwd 3584 917504 7340032 7340032 7340032 7340032 7340032 7340032
base NeuMF 128 3 train 6912 1704192 13631744 13638400 54519552 54526208 436207872 1996800256
base NeuMF 128 3 eval 359168 718080 7176448 7176448 7372800 7372800 7602432 8540416
base NeuMF 128 3 rec 3592960 3592960 7185408 7185408 7436288 7436288 8119808 10936832
base NeuMF 128 4 fwd 7680 1966080 15728640 15728640 15728640 15728640 15728640 15728640
base NeuMF 128 4 train 15104 3801344 30408960 30423808 121620224 121635072 973078784 4454400256
base NeuMF 128 4 eval 768768 1537280 15368448 15368448 15761408 15761408 15991040 16929024
base NeuMF 128 4 rec 7684864 7684864 15369216 15369216 15824896 15824896 16508416 19325440
misaligned NeuMF 16 1 fwd 8192 8192 8192 8192 8192 8192 8192 8192
misaligned NeuMF 16 1 eval 8960 9472 16640 16640 40960 40960 270592 1208576
misaligned NeuMF 16 1 rec 20736 20736 32768 32768 104448 104448 787968 3604992
misaligned NeuMF 16 2 fwd 40960 40960 40960 40960 40960 40960 40960 40960
misaligned NeuMF 16 2 eval 41728 42240 49408 49408 73728 73728 303360 1241344
misaligned NeuMF 16 2 rec 53504 53504 65536 65536 137216 137216 820736 3637760
misaligned NeuMF 16 3 fwd 172032 172032 172032 172032 172032 172032 172032 172032
misaligned NeuMF 16 3 eval 172800 173312 180480 180480 204800 204800 434432 1372416
misaligned NeuMF 16 3 rec 184576 184576 196608 196608 268288 268288 951808 3768832
misaligned NeuMF 16 4 fwd 696320 696320 696320 696320 696320 696320 696320 696320
misaligned NeuMF 16 4 eval 697088 697600 704768 704768 729088 729088 958720 1896704
misaligned NeuMF 16 4 rec 708864 708864 720896 720896 792576 792576 1476096 4293120
misaligned NeuMF 32 1 fwd 32768 32768 32768 32768 32768 33280 33280 33280
misaligned NeuMF 32 1 eval 33536 34048 41216 41216 65536 65536 295680 1233664
misaligned NeuMF 32 1 rec 45312 45312 57344 57344 129024 129024 813056 3630080
misaligned NeuMF 32 2 fwd 163840 163840 163840 163840 163840 2261504 16941568 67273216
misaligned NeuMF 32 2 eval 164608 165120 172288 172288 196608 196608 17194752 68473600
misaligned NeuMF 32 2 rec 176384 176384 188416 188416 260096 260096 17567488 70766080
misaligned NeuMF 32 3 fwd 688128 688128 688128 688128 688128 6980096 51020288 202015232
misaligned NeuMF 32 3 eval 688896 689408 696576 696576 720896 720896 51255040 203215616
misaligned NeuMF 32 3 rec 700672 700672 712704 712704 784384 784384 51338496 205300224
misaligned NeuMF 32 4 fwd 2785280 2785280 2785280 2785280 2785280 17465856 120226304 472547840
misaligned NeuMF 32 4 eval 2786048 2786560 2793728 2793728 2818048 2818048 120424192 473748224
misaligned NeuMF 32 4 rec 2797824 2797824 2809856 2809856 2881536 2881536 119929088 475417088
misaligned NeuMF 64 1 fwd 131072 131072 131072 131072 131072 131584 131584 131584
misaligned NeuMF 64 1 eval 131840 132352 139520 139520 163840 163840 393984 1331968
misaligned NeuMF 64 1 rec 143616 143616 155648 155648 227328 227328 911360 3728384
misaligned NeuMF 64 2 fwd 655360 655360 655360 655360 655360 4850176 34210304 134873600
misaligned NeuMF 64 2 eval 656128 656640 663808 663808 688128 688128 34454272 136073984
misaligned NeuMF 64 2 rec 667904 667904 679936 679936 751616 751616 34682368 138262528
misaligned NeuMF 64 3 fwd 2752512 2752512 2752512 2752512 2752512 15335936 103416320 405406208
misaligned NeuMF 64 3 eval 2753280 2753792 2760960 2760960 2785280 2785280 103623424 406606592
misaligned NeuMF 64 3 rec 2765056 2765056 2777088 2777088 2848768 2848768 103272960 408379392
misaligned NeuMF 64 4 fwd 0 0 0 0 0 0 0 0
misaligned NeuMF 64 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
misaligned NeuMF 64 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
misaligned NeuMF 128 1 fwd 524288 524288 524288 524288 524288 524800 524800 524800
misaligned NeuMF 128 1 eval 525056 525568 532736 532736 557056 557056 787200 1725184
misaligned NeuMF 128 1 rec 536832 536832 548864 548864 620544 620544 1304576 4121600
misaligned NeuMF 128 2 fwd 2621440 2621440 2621440 2621440 2621440 11010560 69730816 271057408
misaligned NeuMF 128 2 eval 2622208 2622720 2629888 2629888 2654208 2654208 69956352 272257792
misaligned NeuMF 128 2 rec 2633984 2633984 2646016 2646016 2717696 2717696 69895168 274238464
misaligned NeuMF 128 3 fwd 0 0 0 0 0 0 0 0
misaligned NeuMF 128 3 eval 768 1280 8448 8448 32768 32768 262400 1200384
misaligned NeuMF 128 3 rec 12544 12544 24576 24576 96256 96256 779776 3596800
misaligned NeuMF 128 4 fwd 0 0 0 0 0 0 0 0
misaligned NeuMF 128 4 eval 768 1280 8448 8448 32768 32768 262400 1200384
misaligned NeuMF 128 4 rec 12544 12544 24576 24576 96256 96256 779776 3596800
umma_off NeuMF 32 1 train 33024 33024 33024 33024 33024 33024 33024 33024
umma_off NeuMF 32 2 fwd 163840 163840 786432 786432 786432 786432 786432 786432
umma_off NeuMF 32 2 train 164096 164096 164096 164096 164096 164096 164096 164096
umma_off NeuMF 32 2 eval 164608 165120 776448 776448 819200 819200 1048832 1986816
umma_off NeuMF 32 2 rec 396288 396288 791808 791808 882688 882688 1566208 4383232
umma_off NeuMF 32 3 fwd 688128 688128 1835008 1835008 1835008 1835008 1835008 1835008
umma_off NeuMF 32 3 train 688384 688384 688384 688384 688384 688384 688384 688384
umma_off NeuMF 32 3 eval 688896 689408 1800448 1800448 1867776 1867776 2097408 3035392
umma_off NeuMF 32 3 rec 907776 907776 1814784 1814784 1931264 1931264 2614784 5431808
umma_off NeuMF 32 4 fwd 2785280 2785280 3932160 3932160 3932160 3932160 3932160 3932160
umma_off NeuMF 32 4 train 2785536 2785536 2785536 2785536 2785536 2785536 2785536 2785536
umma_off NeuMF 32 4 eval 2786048 2786560 3848448 3848448 3964928 3964928 4194560 5132544
umma_off NeuMF 32 4 rec 2797824 2797824 3860736 3860736 4028416 4028416 4711936 7528960
umma_off NeuMF 64 1 train 131328 131328 131328 131328 131328 131328 131328 131328
umma_off NeuMF 64 2 fwd 655360 655360 1572864 1572864 1572864 1572864 1572864 1572864
umma_off NeuMF 64 2 train 655616 655616 655616 655616 655616 655616 655616 655616
umma_off NeuMF 64 2 eval 656128 656640 1544448 1544448 1605632 1605632 1835264 2773248
umma_off NeuMF 64 2 rec 779776 779776 1559040 1559040 1669120 1669120 2352640 5169664
umma_off NeuMF 64 3 fwd 2752512 2752512 3670016 3670016 3670016 3670016 3670016 3670016
umma_off NeuMF 64 3 train 2752768 2752768 2752768 2752768 2752768 2752768 2752768 2752768
umma_off NeuMF 64 3 eval 2753280 2753792 3592448 3592448 3702784 3702784 3932416 4870400
umma_off NeuMF 64 3 rec 2765056 2765056 3604992 3604992 3766272 3766272 4449792 7266816
umma_off NeuMF 128 1 train 524544 524544 524544 524544 524544 524544 524544 524544
umma_off NeuMF 128 2 fwd 2621440 2621440 3145728 3145728 3145728 3145728 3145728 3145728
umma_off NeuMF 128 2 train 2621696 2621696 2621696 2621696 2621696 2621696 2621696 2621696
umma_off NeuMF 128 2 eval 2622208 2622720 3080448 3080448 3178496 3178496 3408128 4346112
umma_off NeuMF 128 2 rec 2633984 2633984 3093504 3093504 3241984 3241984 3925504 6742528
umma_min_b1 NeuMF 32 1 fwd 33280 33280 262144 262144 262144 262144 262144 262144
umma_min_b1 NeuMF 32 1 train 33536 66048 295424 295680 1081856 1081856 8421888 38433280
umma_min_b1 NeuMF 32 1 eval 34048 34560 264448 264448 294912 294912 524544 1462528
umma_min_b1 NeuMF 32 2 fwd 164608 229888 786432 786432 2261248 2261504 16941568 67273216
umma_min_b1 NeuMF 32 2 train 165120 328192 1475072 1475840 5406720 5407232 42107392 192164352
umma_min_b1 NeuMF 32 2 eval 190720 216832 776448 776448 2270720 2270720 17194752 68473600
umma_min_b1 NeuMF 32 2 rec 432640 432640 791808 791808 2306560 2306560 17567488 70766080
umma_min_b1 NeuMF 32 3 fwd 689408 885248 2261504 2262272 6979328 6980096 51020288 202015232
umma_min_b1 NeuMF 32 3 train 690432 1114624 4096512 4098304 14318592 14320128 109740544 499888640
umma_min_b1 NeuMF 32 3 eval 766208 843520 2233088 2233088 6942208 6942208 51255040 203215616
umma_min_b1 NeuMF 32 3 rec 1468416 1468416 2247680 2247680 6922752 6922752 51338496 205300224
umma_min_b1 NeuMF 32 4 fwd 2787584 3244544 6455808 6457600 17464064 17465856 120226304 472547840
umma_min_b1 NeuMF 32 4 train 2789632 3736064 10387968 10391808 33190912 33194496 246055424 1116385792
umma_min_b1 NeuMF 32 4 eval 2965760 3145472 6378240 6378240 17333760 17333760 120424192 473748224
umma_min_b1 NeuMF 32 4 rec 4588544 4588544 6390784 6390784 17203712 17203712 119929088 475417088
umma_min_b1 NeuMF 64 1 fwd 131584 131584 524288 524288 524288 524288 524288 524288
umma_min_b1 NeuMF 64 1 train 131840 197120 655872 656128 2228480 2228736 16908800 76931584
umma_min_b1 NeuMF 64 1 eval 132352 132864 520448 520448 557056 557056 786688 1724672
umma_min_b1 NeuMF 64 2 fwd 656384 786944 1704448 1704960 4849664 4850176 34210304 134873600
umma_min_b1 NeuMF 64 2 train 657152 983552 3277312 3278592 11140352 11141632 84541952 384655872
umma_min_b1 NeuMF 64 2 eval 707840 759552 1688320 1688320 4835840 4835840 34454272 136073984
umma_min_b1 NeuMF 64 2 rec 1179904 1179904 1703424 1703424 4844032 4844032 34682368 138262528
umma_min_b1 NeuMF 64 3 fwd 2754560 3146240 5898752 5900288 15334400 15335936 103416320 405406208
umma_min_b1 NeuMF 64 3 train 2756352 3604992 9568768 9572096 30012672 30016000 220856832 1001153024
umma_min_b1 NeuMF 64 3 eval 2907392 3061504 5833472 5833472 15227392 15227392 103623424 406606592
umma_min_b1 NeuMF 64 3 rec 4300032 4300032 5846528 5846528 15124992 15124992 103272960 408379392
umma_min_b1 NeuMF 128 1 fwd 524800 524800 1048576 1048576 1048576 1048576 1048576 1048576
umma_min_b1 NeuMF 128 1 train 525312 655872 1573376 1573888 4718592 4719104 34079232 154124800
umma_min_b1 NeuMF 128 1 eval 525568 526080 1032448 1032448 1081344 1081344 1310976 2248960
umma_min_b1 NeuMF 128 1 rec 537344 537344 1047552 1047552 1144832 1144832 1828352 4645376
umma_min_b1 NeuMF 128 2 fwd 2622976 2884096 4719104 4720128 11009536 11010560 69730816 271057408
umma_min_b1 NeuMF 128 2 train 2624512 3277312 7864832 7867392 23590912 23593472 170394112 770621952
umma_min_b1 NeuMF 128 2 eval 2725120 2828032 4678400 4678400 10949120 10949120 69956352 272257792
umma_min_b1 NeuMF 128 2 rec 3657472 3657472 4692480 4692480 10902016 10902016 69895168 274238464
"""

PATHS = """
base GMF 5 1 fwd 1 1 1 1 1 1 1 1
base GMF 5 1 train 1 1 1 1 1 1 1 1
base GMF 5 2 fwd 1 1 1 1 1 1 1 1
base GMF 5 2 train 1 1 1 1 1 1 1 1
base GMF 5 3 fwd 1 1 1 1 1 1 1 1
base GMF 5 3 train 1 1 1 1 1 1 1 1
base GMF 5 4 fwd 1 1 1 1 1 1 1 1
base GMF 5 4 train 1 1 1 1 1 1 1 1
base GMF 8 1 fwd 1 1 1 1 1 1 1 1
base GMF 8 1 train 1 1 1 1 1 1 1 1
base GMF 8 2 fwd 1 1 1 1 1 1 1 1
base GMF 8 2 train 1 1 1 1 1 1 1 1
base GMF 8 3 fwd 1 1 1 1 1 1 1 1
base GMF 8 3 train 1 1 1 1 1 1 1 1
base GMF 8 4 fwd 1 1 1 1 1 1 1 1
base GMF 8 4 train 1 1 1 1 1 1 1 1
base GMF 16 1 fwd 1 1 1 1 1 1 1 1
base GMF 16 1 train 1 1 1 1 1 1 1 1
base GMF 16 2 fwd 1 1 1 1 1 1 1 1
base GMF 16 2 train 1 1 1 1 1 1 1 1
base GMF 16 3 fwd 1 1 1 1 1 1 1 1
base GMF 16 3 train 1 1 1 1 1 1 1 1
base GMF 16 4 fwd 1 1 1 1 1 1 1 1
base GMF 16 4 train 1 1 1 1 1 1 1 1
base GMF 32 1 fwd 1 1 1 1 1 1 1 1
base GMF 32 1 train 1 1 1 1 1 1 1 1
base GMF 32 2 fwd 1 1 1 1 1 1 1 1
base GMF 32 2 train 1 1 1 1 1 1 1 1
base GMF 32 3 fwd 1 1 1 1 1 1 1 1
base GMF 32 3 train 1 1 1 1 1 1 1 1
base GMF 32 4 fwd 1 1 1 1 1 1 1 1
base GMF 32 4 train 1 1 1 1 1 1 1 1
base GMF 64 1 fwd 1 1 1 1 1 1 1 1
base GMF 64 1 train 1 1 1 1 1 1 1 1
base GMF 64 2 fwd 1 1 1 1 1 1 1 1
base GMF 64 2 train 1 1 1 1 1 1 1 1
base GMF 64 3 fwd 1 1 1 1 1 1 1 1
base GMF 64 3 train 1 1 1 1 1 1 1 1
base GMF 64 4 fwd 1 1 1 1 1 1 1 .
base GMF 64 4 train 1 1 1 1 1 1 1 .
base GMF 128 1 fwd 1 1 1 1 1 1 1 1
base GMF 128 1 train 1 1 1 1 1 1 1 1
base GMF 128 2 fwd 1 1 1 1 1 1 1 1
base GMF 128 2 train 1 1 1 1 1 1 1 1
base GMF 128 3 fwd 1 1 1 1 1 1 1 .
base GMF 128 3 train 1 1 1 1 1 1 1 .
base GMF 128 4 fwd 1 1 1 1 1 1 . .
base GMF 128 4 train 1 1 1 1 1 1 . .
base NeuMF 5 1 fwd 1 1 1 1 1 1 1 1
base NeuMF 5 1 train 1 1 1 1 1 1 1 1
base NeuMF 5 2 fwd 1 1 1 1 1 1 1 1
base NeuMF 5 2 train 1 1 1 1 1 1 1 1
base NeuMF 5 3 fwd 1 1 1 1 1 1 1 1
base NeuMF 5 3 train 1 1 1 1 1 1 1 1
base NeuMF 5 4 fwd 1 1 1 1 1 1 1 1
base NeuMF 5 4 train 1 1 1 1 1 1 1 1
base NeuMF 8 1 fwd 4 4 4 4 4 4 4 4
base NeuMF 8 1 train 4 4 4 4 4 4 4 4
base NeuMF 8 2 fwd 4 4 4 4 4 4 4 4
base NeuMF 8 2 train 4 4 4 4 4 4 4 4
base NeuMF 8 3 fwd 4 4 4 4 4 4 4 4
base NeuMF 8 3 train 4 4 4 4 4 4 4 4
base NeuMF 8 4 fwd 2 2 2 2 2 2 2 2
base NeuMF 8 4 train 2 2 2 2 2 2 2 2
base NeuMF 16 1 fwd 5 5 5 2 2 2 2 2
base NeuMF 16 1 train 2 2 2 2 2 2 2 2
base NeuMF 16 2 fwd 5 5 5 2 2 2 2 2
base NeuMF 16 2 train 2 2 2 2 2 2 2 2
base NeuMF 16 3 fwd 5 5 5 2 2 2 2 2
base NeuMF 16 3 train 2 2 2 2 2 2 2 2
base NeuMF 16 4 fwd 5 5 5 2 2 2 2 2
base NeuMF 16 4 train 2 2 2 2 2 2 2 2
base NeuMF 32 1 fwd 5 5 5 2 2 3 3 3
base NeuMF 32 1 train 2 2 2 2 2 3 3 3
base NeuMF 32 2 fwd 5 5 5 2 2 3 3 3
base NeuMF 32 2 train 2 2 2 2 2 3 3 3
base NeuMF 32 3 fwd 5 5 5 2 2 3 3 3
base NeuMF 32 3 train 2 2 2 2 2 3 3 3
base NeuMF 32 4 fwd 5 5 5 2 2 3 3 3
base NeuMF 32 4 train 2 2 2 2 2 3 3 3
base NeuMF 64 1 fwd 5 5 5 2 2 3 3 3
base NeuMF 64 1 train 2 2 2 2 2 3 3 3
base NeuMF 64 2 fwd 5 5 5 2 2 3 3 3
base NeuMF 64 2 train 2 2 2 2 2 3 3 3
base NeuMF 64 3 fwd 5 5 5 2 2 3 3 3
base NeuMF 64 3 train 2 2 2 2 2 3 3 3
base NeuMF 64 4 fwd 5 5 5 1 1 1 1 .
base NeuMF 64 4 train 1 1 1 1 1 1 1 .
base NeuMF 128 1 fwd 5 5 5 2 2 3 3 3
base NeuMF 128 1 train 2 2 2 2 2 3 3 3
base NeuMF 128 2 fwd 5 5 5 2 2 3 3 3
base NeuMF 128 2 train 2 2 2 2 2 3 3 3
base NeuMF 128 3 fwd 5 5 5 1 1 1 1 .
base NeuMF 128 3 train 1 1 1 1 1 1 1 .
base NeuMF 128 4 fwd 5 5 5 1 1 1 . .
base NeuMF 128 4 train 1 1 1 1 1 1 . .
misaligned NeuMF 8 1 fwd 2 2 2 2 2 2 2 2
misaligned NeuMF 8 1 train 2 2 2 2 2 2 2 2
misaligned NeuMF 8 2 fwd 2 2 2 2 2 2 2 2
misaligned NeuMF 8 2 train 2 2 2 2 2 2 2 2
misaligned NeuMF 8 3 fwd 2 2 2 2 2 2 2 2
misaligned NeuMF 8 3 train 2 2 2 2 2 2 2 2
misaligned NeuMF 16 1 fwd 2 2 2 2 2 2 2 2
misaligned NeuMF 16 2 fwd 2 2 2 2 2 2 2 2
misaligned NeuMF 16 3 fwd 2 2 2 2 2 2 2 2
misaligned NeuMF 16 4 fwd 2 2 2 2 2 2 2 2
misaligned NeuMF 32 1 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 32 2 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 32 3 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 32 4 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 64 1 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 64 2 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 64 3 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 64 4 fwd 1 1 1 1 1 1 1 .
misaligned NeuMF 128 1 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 128 2 fwd 2 2 2 2 2 3 3 3
misaligned NeuMF 128 3 fwd 1 1 1 1 1 1 1 .
misaligned NeuMF 128 4 fwd 1 1 1 1 1 1 . .
umma_off NeuMF 32 1 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 32 1 train 2 2 2 2 2 2 2 2
umma_off NeuMF 32 2 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 32 2 train 2 2 2 2 2 2 2 2
umma_off NeuMF 32 3 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 32 3 train 2 2 2 2 2 2 2 2
umma_off NeuMF 32 4 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 32 4 train 2 2 2 2 2 2 2 2
umma_off NeuMF 64 1 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 64 1 train 2 2 2 2 2 2 2 2
umma_off NeuMF 64 2 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 64 2 train 2 2 2 2 2 2 2 2
umma_off NeuMF 64 3 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 64 3 train 2 2 2 2 2 2 2 2
umma_off NeuMF 128 1 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 128 1 train 2 2 2 2 2 2 2 2
umma_off NeuMF 128 2 fwd 5 5 5 2 2 2 2 2
umma_off NeuMF 128 2 train 2 2 2 2 2 2 2 2
umma_min_b1 NeuMF 32 1 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 32 1 train 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 32 2 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 32 2 train 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 32 3 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 32 3 train 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 32 4 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 32 4 train 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 64 1 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 64 1 train 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 64 2 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 64 2 train 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 64 3 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 64 3 train 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 128 1 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 128 1 train 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 128 2 fwd 3 3 3 3 3 3 3 3
umma_min_b1 NeuMF 128 2 train 3 3 3 3 3 3 3 3
"""


def _parse(text):
    table = {}
    for line in text.strip().splitlines():
        variant, mt, f, L, what, *vals = line.split()
        table[variant, mt, int(f), int(L), what] = [v if v == "." else int(v) for v in vals]
    return table


def _expected(table, variant, mt, f, L, what):
    """The row of (variant, model), else of the same model in the base variant. An MLP model has the tower
    widths of a NeuMF model of the same f and L, so an MLP row falls back to the NeuMF row first."""
    models = (mt, "NeuMF") if mt == "MLP" else (mt,)
    for key in [(v, m, f, L, what) for v in dict.fromkeys((variant, "base")) for m in models]:
        if key in table:
            return table[key]
    return None


def _fake_model(mt, f, L, offset):
    from ncf_b200 import _lib
    m = _lib.NcfModel()
    m.model_type, m.factor_num, m.num_layers, m.mlp_dim = MODELS[mt], f, L, f << (L - 1)
    m.user_num, m.item_num = 64, REC_ITEMS
    addr = iter(range(1 << 30, 1 << 31, 1 << 20))
    m.embed_user_gmf, m.embed_item_gmf, m.embed_user_mlp, m.embed_item_mlp = (next(addr) for _ in range(4))
    for k in range(L):
        m.mlp_w[k] = next(addr) + offset
        m.mlp_b[k] = next(addr)
    m.predict_w, m.predict_b = next(addr), next(addr)
    return m


def _queries(lib, m, B):
    r = ctypes.byref(m)
    return {"fwd": lib.ncf_forward_workspace_bytes(r, B), "train": lib.ncf_train_workspace_bytes(r, B),
            "eval": lib.ncf_eval_workspace_bytes(r, max(1, B // EVAL_C), EVAL_C),
            "rec": lib.ncf_recommend_workspace_bytes(r, max(1, B // REC_ITEMS), REC_K)}


def _workspace_rows(lib, variant):
    env, offset = VARIANTS[variant]
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        rows = {}
        for mt, f, L in GRID:
            per_b = [_queries(lib, _fake_model(mt, f, L, offset), B) for B in BS]
            for q in QUERIES:
                rows[variant, mt, f, L, q] = [v[q] for v in per_b]
        return rows
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v


@pytest.mark.parametrize("variant", VARIANTS)
def test_workspace_queries_keep_their_values(variant, monkeypatch):
    from ncf_b200 import _lib
    for var in ("NCF_UMMA_MIN_B", "NCF_UMMA_DISABLE", "NCF_UMMA_FUSED"):
        monkeypatch.delenv(var, raising=False)
    table = _parse(WORKSPACE)
    got = _workspace_rows(_lib.load(), variant)
    for (_, mt, f, L, q), vals in got.items():
        assert vals == _expected(table, variant, mt, f, L, q), f"{variant} {mt} f={f} L={L} {q}: {vals}"


# ---- GPU: the path each grid point runs on, and that the queried workspace suffices ---------------------------
def _tower_macs(f, L):
    return sum((f << (L - k)) * (f << (L - k - 1)) for k in range(L))


def _cheap(f, L, B):
    return B * _tower_macs(f, L) <= 10 ** 11


def _gpu_grid(variant):
    return [g for g in GRID if variant == "base" or g[0] == "NeuMF"]


def _device_model(mt, f, L, offset, gen):
    """64-row tables; with offset 4 every tower weight starts 4 bytes past a 256-byte-aligned address"""
    import torch
    from ncf_b200 import ops
    dev = torch.device("cuda")
    rnd = lambda *s: (torch.rand(*s, generator=gen, device=dev) - 0.5) * 0.2
    d = f << (L - 1)
    tables = (rnd(64, f), rnd(64, f), rnd(64, d), rnd(64, d))
    linears = []
    for k in range(L):
        n_in, n_out = f << (L - k), f << (L - k - 1)
        w = torch.empty(n_in * n_out + offset // 4, device=dev)[offset // 4:].view(n_out, n_in)
        w.copy_(rnd(n_out, n_in))
        linears.append((w, rnd(n_out)))
    predict = (rnd(2 * f if mt == "NeuMF" else f), rnd(1))
    bufs = (tables, linears, predict)
    return ops.model_struct(MODELS[mt], f, L, 64, 64, tables, linears, predict), bufs


GUARD = 4096


def _guarded(nbytes):
    import torch
    return torch.full((nbytes + GUARD,), 0xA5, dtype=torch.uint8, device="cuda")


def _guard_intact(ws, nbytes):
    return bool((ws[nbytes:] == 0xA5).all())


def _run_paths(lib, variant, mt, f, L):
    """(forward paths, training paths) over BS, "." where the point is not cheap; asserts that the workspace
    queried for B serves B and the grid point below it without writing past its end"""
    import torch
    from ncf_b200 import ops
    from ncf_b200._lib import current_stream, ptr
    gen = torch.Generator(device="cuda").manual_seed(f * 10 + L)
    m, _bufs = _device_model(mt, f, L, VARIANTS[variant][1], gen)
    r = ctypes.byref(m)
    bmax = max(B for B in BS if _cheap(f, L, B))
    user = torch.randint(0, 64, (bmax,), generator=gen, device="cuda")
    item = torch.randint(0, 64, (bmax,), generator=gen, device="cuda")
    label = (torch.rand(bmax, generator=gen, device="cuda") < 0.5).float()
    logits = torch.empty(bmax, device="cuda")
    loss = torch.zeros(1, dtype=torch.float64, device="cuda")
    grads = ops.GradBuffers.allocate(MODELS[mt], f, L, 64, 64, 64, torch.device("cuda"))
    g = grads.struct()
    st = current_stream()

    def forward(B, ws, nbytes):
        assert lib.ncf_forward(r, ptr(user), ptr(item), B, ptr(logits), ptr(ws), nbytes, st) == 0, \
            lib.ncf_last_error()
        return lib.ncf_last_tile_path()

    def train(B, ws, nbytes):
        for t in (grads.flat, grads.user_flag, grads.item_flag, grads.touched_count):
            t.zero_()
        rc = lib.ncf_train_step_grads(r, ctypes.byref(g), ptr(user), ptr(item), ptr(label), None, 1.0, B,
                                      ptr(loss), ptr(logits), ptr(ws), nbytes, st)
        return rc if rc != 0 else lib.ncf_last_tile_path()

    fwd, trn = [], []
    for i, B in enumerate(BS):
        if not _cheap(f, L, B):
            fwd.append(".")
            trn.append(".")
            continue
        Bs = BS[i - 1] if i > 0 else B
        for run, query, out in ((forward, lib.ncf_forward_workspace_bytes, fwd),
                                (train, lib.ncf_train_workspace_bytes, trn)):
            nbytes = query(r, B)
            ws = _guarded(nbytes)
            path = run(B, ws, nbytes)
            assert path > 0, f"{variant} {mt} f={f} L={L} B={B}: {path}, {lib.ncf_last_error()}"
            small_path = run(Bs, ws, nbytes)
            assert small_path > 0, f"{variant} {mt} f={f} L={L} B={Bs} in the workspace of B={B}: {small_path}"
            torch.cuda.synchronize()
            assert _guard_intact(ws, nbytes), f"{variant} {mt} f={f} L={L} B={B}: wrote past the workspace"
            out.append(path)
        nbytes = lib.ncf_train_workspace_bytes(r, B)
        ws = _guarded(nbytes)
        assert train(B, ws, nbytes - 1) == NCF_ERR_WORKSPACE, f"{variant} {mt} f={f} L={L} B={B}"
    torch.cuda.synchronize()
    return fwd, trn


@gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_tile_paths_and_queried_workspace_on_device(variant, monkeypatch):
    from ncf_b200 import _lib
    for var in ("NCF_UMMA_MIN_B", "NCF_UMMA_DISABLE", "NCF_UMMA_FUSED"):
        monkeypatch.delenv(var, raising=False)
    for k, v in VARIANTS[variant][0].items():
        monkeypatch.setenv(k, v)
    lib = _lib.load()
    table = _parse(PATHS)
    for mt, f, L in _gpu_grid(variant):
        fwd, trn = _run_paths(lib, variant, mt, f, L)
        assert fwd == _expected(table, variant, mt, f, L, "fwd"), f"{variant} {mt} f={f} L={L} forward: {fwd}"
        assert trn == _expected(table, variant, mt, f, L, "train"), f"{variant} {mt} f={f} L={L} train: {trn}"


def _print_table(rows):
    """the rows that differ from what _expected would fall back to"""
    listed = {}
    for key in sorted(rows, key=lambda k: (k[0] != "base", k[1] == "MLP")):
        if rows[key] != _expected(listed, *key):
            listed[key] = rows[key]
            print(" ".join(map(str, key + tuple(rows[key]))))


if __name__ == "__main__":
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    from ncf_b200 import _lib
    lib = _lib.load()
    rows = {}
    if "--paths" in sys.argv:
        for variant, (env, _) in VARIANTS.items():
            os.environ.update(env)
            for mt, f, L in _gpu_grid(variant):
                rows[variant, mt, f, L, "fwd"], rows[variant, mt, f, L, "train"] = _run_paths(lib, variant, mt, f, L)
            for k in env:
                os.environ.pop(k)
    else:
        for variant in VARIANTS:
            rows.update(_workspace_rows(lib, variant))
    _print_table(rows)
