"""Host-side logic without a GPU: the C-ABI library loads and exports every symbol include/hdrvae.h
declares, struct layouts match the ctypes mirror, the node surface equals the reference's, error paths
fail loudly (no CPU fallback), multi-GPU host logic on gloo with world_size 2."""
import ctypes as C
import os
import re
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle.ref_loader import reference_available

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from vae_decode_hdr_b200 import _native
    if not os.path.isfile(_native.LIB_PATH):
        _native.build_library()
    return _native.load_library()


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "hdrvae.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hdrvae_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib):
    from vae_decode_hdr_b200 import _native
    names = _declared_symbols()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"libhdrvae.so lacks {n} declared in include/hdrvae.h"
        assert n in _native.SIGNATURES, f"{n} has no ctypes signature in _native.py"
    assert sorted(_native.SIGNATURES) == names


def test_abi_version_and_argument_counts_match_header(lib):
    """The library, the ctypes binding and include/hdrvae.h agree on HDRVAE_ABI_VERSION, and every ctypes signature takes
    as many arguments as the header's prototype (a stale binding would pass garbage for a new trailing argument)."""
    from vae_decode_hdr_b200 import _native
    src = open(os.path.join(ROOT, "include", "hdrvae.h")).read()
    version = int(re.search(r"#define HDRVAE_ABI_VERSION (\d+)", src).group(1))
    assert lib.hdrvae_abi_version() == _native.ABI_VERSION == version
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = dict(re.findall(r"\b(hdrvae_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", src))
    assert sorted(protos) == sorted(_native.SIGNATURES)
    for name, params in protos.items():
        n = 0 if params.strip() in ("", "void") else params.count(",") + 1
        assert len(_native.SIGNATURES[name][1]) == n, f"{name}: header declares {n} arguments"


def test_struct_layouts_match_header():
    from vae_decode_hdr_b200 import _native as N
    assert C.sizeof(N.HdrvaeStats) == 200           # static_assert'ed in csrc/api.cu
    assert C.sizeof(N.HdrvaeRawStats) == 96
    assert C.sizeof(N.HdrvaeWeightDesc) == 56
    assert C.sizeof(N.HdrvaeConvExtra) == 64 and N.HdrvaeConvExtra.y2.offset == 16 and N.HdrvaeConvExtra.act.offset == 60
    assert N.HdrvaeStats.norm_function.offset == 184 and N.HdrvaeStats.hdr_pixels.offset == 144


def test_sass_is_blackwell_native():
    """The product kernels must be tcgen05/TMA code, not recompiled mma.sync: UTCHMMA / UTMALDG / LDTM in SASS."""
    import shutil
    import subprocess
    from vae_decode_hdr_b200 import _native
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", _native.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic
    assert "HMMA." not in sass.replace("UTCHMMA", "")


def test_no_cpu_fallback(lib):
    """Without a CUDA device the product path must raise, never compute on the CPU."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS
    from vae_decode_hdr_b200.synthetic import SyntheticVAE
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        HdrVaeEngine({}, "cuda")
    ctx = C.c_void_p()
    assert lib.hdrvae_create(C.byref(ctx), 0) != 0 and lib.hdrvae_last_error()
    node = NODE_CLASS_MAPPINGS["HDRVAEDecode"]()
    with pytest.raises(RuntimeError):
        node.simple_hdr_decode({"samples": torch.zeros(1, 16, 4, 4)}, SyntheticVAE({}, device="cpu"))


def test_product_package_never_imports_oracle():
    for fn in os.listdir(os.path.join(ROOT, "vae_decode_hdr_b200")):
        if fn.endswith(".py"):
            src = open(os.path.join(ROOT, "vae_decode_hdr_b200", fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn


def test_node_surface_equals_reference():
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS, NODE_DISPLAY_NAME_MAPPINGS
    cls = NODE_CLASS_MAPPINGS["HDRVAEDecode"]
    assert NODE_DISPLAY_NAME_MAPPINGS == {"HDRVAEDecode": "HDR VAE Decode", "LinearEXRExport": "Linear EXR Export",
                                          "HDRUpscaleWithModel": "HDR Upscale with Model"}
    assert list(NODE_CLASS_MAPPINGS) == ["HDRVAEDecode", "LinearEXRExport", "HDRUpscaleWithModel"]     # __init__.py:43-47
    assert (cls.RETURN_TYPES, cls.RETURN_NAMES, cls.FUNCTION, cls.CATEGORY) == (("IMAGE",), ("image",), "simple_hdr_decode", "latent")


@pytest.mark.skipif(not reference_available(), reason="unmodified reference source not present (HDRVAE_REFERENCE_ROOT)")
def test_node_surface_equals_reference_tree():
    """The same node surface against the unmodified reference class itself."""
    import inspect
    from oracle.ref_loader import load_reference_module
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS
    cls = NODE_CLASS_MAPPINGS["HDRVAEDecode"]
    ref = load_reference_module().HDRVAEDecode
    assert cls.INPUT_TYPES() == ref.INPUT_TYPES()
    assert (cls.RETURN_TYPES, cls.RETURN_NAMES, cls.FUNCTION, cls.CATEGORY) == \
        (ref.RETURN_TYPES, ref.RETURN_NAMES, ref.FUNCTION, ref.CATEGORY)
    mine = inspect.signature(cls.simple_hdr_decode).parameters
    # same named parameters in the same order; the only addition is a **kwargs sink for the README-era inputs
    assert [n for n, p in mine.items() if p.kind is not inspect.Parameter.VAR_KEYWORD] == \
        list(inspect.signature(ref.simple_hdr_decode).parameters)
    assert NODE_CLASS_MAPPINGS.keys() == load_reference_package_mappings().keys()


def load_reference_package_mappings():
    """NODE_CLASS_MAPPINGS keys of the unmodified reference __init__.py (read as text: importing it needs ComfyUI)."""
    from oracle.ref_loader import REFERENCE_ROOT
    src = open(os.path.join(REFERENCE_ROOT, "__init__.py")).read()
    block = src[src.index("NODE_CLASS_MAPPINGS = {"):]
    block = block[:block.index("}")]
    return {k: None for k in re.findall(r'"(\w+)":', block)}


def test_legacy_readme_inputs_are_tolerated_and_unknown_ones_rejected():
    """README.md:143-145 / workflow_examples/HDR_VAE_DECODE.json:499-504: max_range, scale_factor, enable_negatives no
    longer exist in the reference code; prompts that still carry them must not fail on the argument list."""
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS
    from vae_decode_hdr_b200.synthetic import SyntheticVAE
    node = NODE_CLASS_MAPPINGS["HDRVAEDecode"]()
    z = {"samples": torch.zeros(1, 16, 4, 4)}
    with pytest.raises(TypeError, match="bogus"):
        node.simple_hdr_decode(z, SyntheticVAE({}, device="cpu"), bogus=1)
    if not torch.cuda.is_available():
        # the legacy names pass the argument check; what fails afterwards is the missing GPU, not the call signature
        with pytest.raises(RuntimeError, match="CUDA"):
            node.simple_hdr_decode(z, SyntheticVAE({}, device="cpu"), hdr_mode="conservative", max_range=50,
                                   scale_factor=1, enable_negatives=False)


def test_mode_resolution_and_synthetic_weights():
    from vae_decode_hdr_b200.engine import resolve_mode
    from vae_decode_hdr_b200.synthetic import decoder_param_shapes, random_decoder_state_dict
    from oracle.flux_decoder import build_decoder
    assert resolve_mode("conservative") == (0, 1.0) and resolve_mode("exposure") == (1, 1.0)
    assert resolve_mode("adaptive_recovery") == (2, 1.0) and resolve_mode("mathematical_recovery") == (3, 1.0)
    assert resolve_mode("Moderate") == (0, 3.0) and resolve_mode("aggressive") == (3, 1.0)
    with pytest.raises(ValueError):
        resolve_mode("bypass")
    ref = build_decoder(0).state_dict()
    assert {k: tuple(v.shape) for k, v in ref.items()} == dict(decoder_param_shapes())
    sd = random_decoder_state_dict(0)
    assert sum(v.numel() for v in sd.values()) == 49_545_475


def test_shard_bounds():
    from vae_decode_hdr_b200.sharding import shard_bounds
    assert shard_bounds(32, 8) == [(4 * i, 4 * i + 4) for i in range(8)]
    assert shard_bounds(5, 2) == [(0, 3), (3, 5)]
    assert shard_bounds(1, 4) == [(0, 1), (1, 1), (1, 1), (1, 1)]
    assert shard_bounds(0, 2) == [(0, 0), (0, 0)]
    with pytest.raises(ValueError):
        shard_bounds(4, 0)


def _gloo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from oracle import hdr_oracle as ho
    from vae_decode_hdr_b200.sharding import allreduce_raw_stats, shard_bounds
    g = torch.Generator().manual_seed(0)
    pre = torch.randn(4, 128, 8, 8, generator=g) * 0.7
    w = torch.randn(3, 128, 3, 3, generator=g) * 0.05
    b = torch.zeros(3)
    s, e = shard_bounds(4, world)[rank]

    def raw(x):     # the hdrvae_raw_stats block of a slice, computed by the oracle (CPU stand-in for phase A)
        an = ho.analyze(x, w, b)
        p3 = ho.channel_maxpool3(x)
        st, co = an["standard"], an["conv_only"]
        vmin = torch.tensor([x.min(), st.min(), co.min(), p3.min()])
        vmax = torch.tensor([x.max(), st.max(), co.max(), p3.max()])
        vsum = torch.tensor([x.double().sum(), (x.double() ** 2).sum(), st.double().sum(), (st.double() ** 2).sum(),
                             co.double().sum(), x.numel(), st.numel(), float((p3 > 1).sum())], dtype=torch.float64)
        return vmin, vmax, vsum
    vmin, vmax, vsum = raw(pre[s:e])
    allreduce_raw_stats(vmin, vmax, vsum)
    fmin, fmax, fsum = raw(pre)
    ok = torch.equal(vmin, fmin) and torch.equal(vmax, fmax) and torch.allclose(vsum, fsum, rtol=1e-12)
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def _gloo_block_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from vae_decode_hdr_b200.sharding import exchange_raw_stats_block, identity_raw_block
    # rank 2 holds an EMPTY shard (batch 2 over 3 ranks): it contributes the neutral block
    if rank == 2:
        blk = identity_raw_block("cpu")
    else:
        blk = torch.zeros(96, dtype=torch.uint8)
        blk[0:16].view(torch.float32).copy_(torch.tensor([1.0, -2.0, 0.5, 3.0]) + rank)
        blk[16:32].view(torch.float32).copy_(torch.tensor([5.0, 6.0, 7.0, 8.0]) - rank)
        blk[32:96].view(torch.float64).copy_(torch.arange(8, dtype=torch.float64) * (rank + 1))
    exchange_raw_stats_block(blk, group=None)
    ok = torch.equal(blk[0:16].view(torch.float32), torch.tensor([1.0, -2.0, 0.5, 3.0]))
    ok &= torch.equal(blk[16:32].view(torch.float32), torch.tensor([5.0, 6.0, 7.0, 8.0]))
    ok &= torch.equal(blk[32:96].view(torch.float64), torch.arange(8, dtype=torch.float64) * 3)
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_raw_stats_single_collective_exchange_with_empty_shard_gloo_world3():
    """The batch-sharded exchange step (ONE all-gather + rank-order merge) on 3 CPU ranks, one of which holds an empty
    shard and contributes the neutral block: every rank ends with the statistics of the two non-empty shards."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_block_worker, args=(r, 3, port, q)) for r in range(3)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True), (2, True)]


def test_batch_sharded_stats_allreduce_gloo_world2():
    """N>1 host logic on CPU: sharded raw statistics + MIN/MAX/SUM all-reduce == whole-batch statistics."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def _rows_exchange_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from vae_decode_hdr_b200 import _native as N
    from vae_decode_hdr_b200.sharding import _exchange_nccl
    # a miniature workspace: one slab of 4 interior rows of 16 bytes with a halo row each side at offset 64,
    # 5 float64 sums at 256, a 3-rank gather region of 8 bytes per rank at 320, a raw statistics block at 384
    ws = torch.zeros(512, dtype=torch.uint8)
    row = 16
    slab = ws[64:64 + 6 * row].view(6, row)
    slab[1:5] = torch.arange(4, dtype=torch.uint8)[:, None] + 10 * (rank + 1)
    ws[256:296].view(torch.float64).copy_(torch.arange(5, dtype=torch.float64) + rank)
    ws[320 + 8 * rank:328 + 8 * rank] = rank + 1
    vmin, vmax = ws[384:400].view(torch.float32), ws[400:416].view(torch.float32)
    vsum = ws[416:480].view(torch.float64)
    vmin.fill_(float(rank)); vmax.fill_(float(rank)); vsum.fill_(float(rank + 1))
    ex = N.HdrvaeExchange()
    ex.kind = N.EX_HALO | N.EX_ALLREDUCE_F64
    ex.n_halo = 1
    ex.halo_row_bytes[0] = row
    ex.halo_top_off[0] = 64
    ex.halo_first_row_off[0] = 64 + row
    ex.halo_last_row_off[0] = 64 + 4 * row
    ex.halo_bottom_off[0] = 64 + 5 * row
    ex.allreduce_off, ex.allreduce_count = 256, 5
    _exchange_nccl(ex, ws, rank, world)
    ok = True
    top = 0 if rank == 0 else 10 * rank + 3                   # the neighbour's last interior row (or untouched)
    bot = 0 if rank == world - 1 else 10 * (rank + 2)          # the neighbour's first interior row
    ok &= bool((slab[0] == top).all()) and bool((slab[5] == bot).all())
    ok &= bool((slab[1:5] == torch.arange(4, dtype=torch.uint8)[:, None] + 10 * (rank + 1)).all())
    ok &= torch.equal(ws[256:296].view(torch.float64), world * torch.arange(5, dtype=torch.float64) + sum(range(world)))
    ex2 = N.HdrvaeExchange()
    ex2.kind = N.EX_ALLGATHER | N.EX_RAW_STATS
    ex2.n_gather = 1
    ex2.gather_off[0], ex2.gather_bytes_per_rank[0] = 320, 8
    ex2.raw_stats_off = 384
    _exchange_nccl(ex2, ws, rank, world)
    ok &= torch.equal(ws[320:320 + 8 * world], torch.arange(1, world + 1, dtype=torch.uint8).repeat_interleave(8))
    ok &= bool((vmin == 0).all()) and bool((vmax == world - 1).all()) and bool((vsum == world * (world + 1) / 2).all())
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_row_tiling_exchange_executor_gloo_world3():
    """The executor of the row-tiled decode's exchange descriptors (halo send/recv with both neighbours, float64
    sum all-reduce, all-gather in rank order, MIN/MAX/SUM of the raw statistics block) on 3 CPU ranks."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_rows_exchange_worker, args=(r, 3, port, q)) for r in range(3)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True), (2, True)]


def test_upscaler_node_surface_equals_reference():
    """HDRUpscaleWithModel: RETURN_TYPES / FUNCTION / CATEGORY of the reference class (hdr_upscale_with_model.py:50-71,148),
    and no CPU fallback."""
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS
    cls = NODE_CLASS_MAPPINGS["HDRUpscaleWithModel"]
    assert (cls.RETURN_TYPES, cls.FUNCTION, cls.CATEGORY) == (("IMAGE",), "upscale", "HDR/Upscale")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cls._compute_device(torch.zeros(1, 4, 4, 3))


@pytest.mark.skipif(not reference_available(), reason="unmodified reference source not present (HDRVAE_REFERENCE_ROOT)")
def test_upscaler_node_surface_equals_reference_tree():
    """Same INPUT_TYPES / RETURN_TYPES / FUNCTION / CATEGORY / upscale() parameters as the unmodified reference class."""
    import inspect
    from oracle import upscaler_oracle as uo
    from oracle.ref_loader import load_reference_upscaler
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS
    cls = NODE_CLASS_MAPPINGS["HDRUpscaleWithModel"]
    ref = type(load_reference_upscaler(uo.FakeDescriptor(torch.nn.Identity())))
    want, got = ref.INPUT_TYPES()["required"], cls.INPUT_TYPES()["required"]
    assert list(want) == list(got)
    for k in want:
        if k != "model_name":                 # the file list comes from ComfyUI's folder_paths
            assert want[k] == got[k], k
    assert (cls.RETURN_TYPES, cls.FUNCTION, cls.CATEGORY) == (ref.RETURN_TYPES, ref.FUNCTION, ref.CATEGORY)
    assert list(inspect.signature(cls.upscale).parameters) == list(inspect.signature(ref.upscale).parameters)


def test_groupnorm_partial_capacity_covers_both_conv_tilings(lib):
    """Host logic, no GPU: the GroupNorm partial-chunk capacity the library reports for an H x W conv output must cover
    both ways the tensor-core kernel may tile it (the best 128-pixel patch, and the 8 x 16 tiles of the slab form) —
    the conv epilogue writes one partial per tile."""
    import itertools
    for H, W in itertools.chain([(1, 1), (5, 9), (16, 8), (40, 72), (128, 128), (1024, 1024), (4096, 4096), (17, 1000)],
                                [(h, w) for h in (3, 24, 100) for w in (7, 64, 257)]):
        cap = lib.hdrvae_conv2d_stats_chunks(H, W, 0)
        slab = -(-W // 8) * -(-H // 16)
        best = min(-(-W // (1 << lg)) * -(-H // (128 >> lg)) for lg in range(8))
        assert cap >= slab and cap >= best, (H, W, cap, slab, best)
        assert lib.hdrvae_conv2d_stats_chunks(H, W, 1) == 4 * cap          # upsample convs: 4 phases


def test_public_header_is_plain_c():
    """The drop-in boundary is a C ABI: include/hdrvae.h must compile as C99 (no C++ or torch types in the signatures)."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    hdr = os.path.join(ROOT, "include", "hdrvae.h")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-fsyntax-only", "-x", "c", hdr], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_environment_is_read_only_by_the_switch_table():
    """The library reads its environment switches in one place, switches() in csrc/api.cu, and DESIGN.md §6 lists exactly
    the switches read there: no getenv elsewhere in csrc/, every getenv there names its variable literally."""
    csrc = os.path.join(ROOT, "vae_decode_hdr_b200", "csrc")
    api = open(os.path.join(csrc, "api.cu")).read()
    m = re.search(r"^const Switches& switches\(\) \{\n.*?^\}\n", api, flags=re.S | re.M)
    assert m, "switches() not found in csrc/api.cu"
    table = m.group(0)
    for fn in sorted(os.listdir(csrc)):
        if fn.endswith((".cu", ".cuh", ".h")):
            src = open(os.path.join(csrc, fn)).read()
            if fn == "api.cu":
                src = src.replace(table, "")
            assert "getenv" not in src, f"csrc/{fn} reads the environment outside switches()"
    names = re.findall(r"getenv\(\"(HDRVAE_[A-Z0-9_]+)\"\)", table)
    assert len(names) == table.count("getenv(") and len(set(names)) == len(names), table
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    sec = re.search(r"^## 6\..*?(?=^## 7\.)", design, flags=re.S | re.M)
    assert sec, "DESIGN.md has no section 6"
    para = re.search(r"^\*\*Switches\*\*.*?(?=\n\n)", sec.group(0), flags=re.S | re.M)
    assert para, "DESIGN.md §6 has no **Switches** paragraph"
    assert sorted(set(re.findall(r"HDRVAE_[A-Z0-9_]+", para.group(0)))) == sorted(names)
