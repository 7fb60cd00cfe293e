"""CPU tests (-m "not gpu"): the C-ABI library loads and exports every symbol include/cfb.h declares, the host-side
mirror of the reference interface (constructor surface, errors, state_dict layout, config selection), and the
length-bucketed sharding logic incl. a world_size-2 gloo run."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

import conformer_nemo_b200 as cn
from conformer_nemo_b200 import _lib
from oracle import conformer_oracle as oc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def lib():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge

    ge.build()
    return _lib.load_library()


def test_library_exports_every_declared_symbol(lib):
    header = open(os.path.join(ROOT, "include", "cfb.h")).read()
    declared = set(re.findall(r"CFB_API\s+[\w\s\*]+?\b(cfb_\w+)\s*\(", header))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (cfb_\w+)", out))
    assert declared <= exported
    # the library must not need libcuda at load time (driver entry points are resolved through the runtime)
    ldd = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "libcuda.so" not in ldd and "libtorch" not in ldd


def test_integration_notes_name_every_entry_point():
    """INTEGRATION.md is the maintainer-facing map of the C ABI: every exported entry point is named there."""
    header = open(os.path.join(ROOT, "include", "cfb.h")).read()
    declared = set(re.findall(r"CFB_API\s+[\w\s\*]+?\b(cfb_\w+)\s*\(", header))
    notes = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    missing = sorted(n for n in declared if n not in notes)
    assert not missing, missing


def test_hot_kernels_keep_index_registers_out_of_the_tile_loops(lib):
    """ptxas rematerialises special-register reads (S2R SR_TID.X, SR_CgaCtaId: tens of cycles each) wherever it is short of
    registers; in the attention kernels that was several reads per key tile (DESIGN.md section 4).  The fixes route the
    values through a shuffle / a volatile mov; this pins the count so that a refactor does not silently bring them back."""
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    if not sass:
        pytest.skip("cuobjdump unavailable")
    counts, fn = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = m.group(1)
        elif fn and ("SR_TID" in line or "SR_CgaCtaId" in line):
            counts[fn] = counts.get(fn, 0) + 1
    attn = {k: v for k, v in counts.items() if "rel_attn_tc" in k}
    assert attn, "attention kernels not found in the library"
    for name, n in attn.items():
        assert n <= 6, (name, n)  # set-up and tear-down reads only (was 25 + 14 in the persistent kernel)
    # and no local-memory frames in the tensor-core kernels (run-time indexed counters were LDL in front of mbarrier waits)
    res = subprocess.run(["cuobjdump", "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    fn = None
    for line in res.splitlines():
        m = re.search(r"Function (\S+?):", line)
        if m:
            fn = m.group(1)
        m = re.search(r"STACK:(\d+)", line)
        if m and fn and any(k in fn for k in ("rel_attn_tc", "gemm_tc", "dw_pw_kernel")):
            assert int(m.group(1)) == 0, (fn, line.strip())


def test_sass_contains_blackwell_tensor_core_and_tma_instructions(lib):
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    if not sass:
        pytest.skip("cuobjdump unavailable")
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic
    assert "HMMA.16816" not in sass  # no legacy mma.sync tensor path


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_create_fails_loudly_without_a_gpu(lib):
    cfg = _lib.CfbConfig(feat_in=80, n_layers=1, d_model=64, feat_out=-1, subsampling_factor=4,
                         subsampling_conv_channels=-1, ff_expansion_factor=4, n_heads=4, conv_kernel_size=31,
                         xscaling=1, precision=0)
    handle = ctypes.c_void_p()
    rc = lib.cfb_create(ctypes.byref(cfg), 0, ctypes.byref(handle))
    assert rc != 0 and not handle.value
    assert "no CPU fallback" in _lib.last_error(None)
    with pytest.raises(RuntimeError):
        _lib.check(rc, None, "cfb_create")


def test_unsupported_config_is_rejected_by_the_library(lib):
    cfg = _lib.CfbConfig(feat_in=80, n_layers=1, d_model=64, feat_out=-1, subsampling_factor=8,
                         subsampling_conv_channels=-1, ff_expansion_factor=4, n_heads=4, conv_kernel_size=31,
                         xscaling=1, precision=0)
    handle = ctypes.c_void_p()
    assert lib.cfb_create(ctypes.byref(cfg), 0, ctypes.byref(handle)) == 2  # CFB_ERR_UNSUPPORTED
    cfg.subsampling_factor = 4
    cfg.d_model = 60
    assert lib.cfb_create(ctypes.byref(cfg), 0, ctypes.byref(handle)) in (1, 2)
    assert lib.cfb_create(None, 0, ctypes.byref(handle)) == 1


def test_constructor_surface_and_errors():
    # the reference raises ValueError for these (conformer_encoder.py:190-191, subsampling.py:63-64,149)
    with pytest.raises(ValueError):
        cn.ConformerEncoder(feat_in=80, n_layers=1, d_model=64, self_attention_model="bogus")
    with pytest.raises(ValueError):
        cn.ConformerEncoder(feat_in=80, n_layers=1, d_model=64, subsampling="nope")
    with pytest.raises(ValueError):
        cn.ConformerEncoder(feat_in=80, n_layers=1, d_model=64, subsampling_factor=3)
    # supported by the reference, not built here: explicit NotImplementedError, never a silent fallback
    for kw in (dict(self_attention_model="abs_pos"), dict(subsampling="vggnet"), dict(conv_norm_type="layer_norm"),
               dict(att_context_size=[10, 10]), dict(subsampling_factor=8)):
        with pytest.raises(NotImplementedError):
            cn.ConformerEncoder(feat_in=80, n_layers=1, d_model=64, **kw)
    enc = cn.ConformerEncoder(feat_in=80, n_layers=2, d_model=64, n_heads=4, feat_out=48)
    assert enc._feat_in == 80 and enc._feat_out == 48 and enc.d_model == 64
    assert list(enc.input_types) == ["audio_signal", "length"] and list(enc.output_types) == ["outputs", "encoded_lengths"]
    with pytest.raises(RuntimeError, match="no CPU path"):
        enc(audio_signal=torch.randn(1, 80, 40), length=torch.tensor([40]))
    with pytest.raises(TypeError):
        enc(audio_signal=torch.randn(1, 79, 40))
    enc.unfreeze()
    assert enc.training and all(p.requires_grad for p in enc.parameters())
    enc.freeze()
    assert not enc.training and not any(p.requires_grad for p in enc.parameters())


@pytest.mark.parametrize("kw", [dict(feat_in=80, n_layers=2, d_model=64, n_heads=4),
                                dict(feat_in=80, n_layers=1, d_model=176, n_heads=4, feat_out=96),
                                dict(feat_in=64, n_layers=1, d_model=128, n_heads=8, subsampling_conv_channels=32)])
def test_state_dict_layout_matches_reference(kw):
    enc = cn.ConformerEncoder(**kw)
    cfg = oc.EncoderConfig(**kw)
    want = oc.expected_state_shapes(cfg)
    got = {k: tuple(v.shape) for k, v in enc.state_dict().items() if not k.endswith("num_batches_tracked")}
    assert got == want
    sd = oc.random_state_dict(cfg, 3)
    missing, unexpected = enc.load_state_dict(sd, strict=False)
    assert not unexpected and all(m.endswith("num_batches_tracked") for m in missing)
    assert enc._dirty


def test_untied_biases_false_shares_one_parameter_pair():
    enc = cn.ConformerEncoder(feat_in=80, n_layers=3, d_model=64, n_heads=4, untie_biases=False)
    us = {id(l.self_attn.pos_bias_u) for l in enc.layers}
    assert len(us) == 1
    assert "layers.2.self_attn.pos_bias_u" in enc.state_dict()


def test_recipe_selection_from_reference_yaml(tmp_path):
    doc = """
model:
  preprocessor: {features: 80}
  encoder:
    _target_: nemo.collections.asr.modules.ConformerEncoder
    feat_in: ${model.preprocessor.features}
    feat_out: -1
    n_layers: 2
    d_model: 64
    subsampling: striding
    subsampling_factor: 4
    subsampling_conv_channels: -1
    ff_expansion_factor: 4
    self_attention_model: rel_pos
    n_heads: 4
    att_context_size: [-1, -1]
    xscaling: true
    untie_biases: true
    pos_emb_max_len: 5000
    conv_kernel_size: 31
    conv_norm_type: 'batch_norm'
    dropout: 0.1
    dropout_emb: 0.0
    dropout_att: 0.1
  decoder: {feat_in: "${model.encoder.d_model}"}
"""
    p = tmp_path / "recipe.yaml"
    p.write_text(doc)
    cfg = cn.load_encoder_config(str(p))
    assert cfg["feat_in"] == 80 and cfg["_target_"].endswith("ConformerEncoder")
    enc = cn.instantiate_encoder(cfg)
    assert isinstance(enc, cn.ConformerEncoder) and len(enc.layers) == 2
    cfg["_target_"] = "conformer_nemo_b200.ConformerEncoder"
    assert isinstance(cn.instantiate_encoder(cfg), cn.ConformerEncoder)
    from oracle import reference_loader as rl

    # every recipe resolves and is accepted by the constructor: the stored encoder blocks (tests/golden/recipes), plus the
    # shipped recipes themselves when the reference tree is reachable
    stored = os.path.join(ROOT, "tests", "golden", "recipes")
    want = {"conformer_ctc_bpe.yaml": (512, 18, 8), "conformer_transducer_bpe.yaml": (512, 17, 8),
            "conformer_ctc_char.yaml": (256, 16, 8)}
    assert sorted(os.listdir(stored)) == sorted(want)
    for name, (d, layers, heads) in want.items():
        c = cn.load_encoder_config(os.path.join(stored, name))
        assert (c["feat_in"], c["d_model"], c["n_layers"], c["n_heads"]) == (80, d, layers, heads), name
    ref_recipes = os.path.join(rl.REFERENCE_ROOT, "configs")
    paths = [os.path.join(stored, n) for n in sorted(want)]
    if os.path.isdir(ref_recipes):
        paths += [os.path.join(ref_recipes, n) for n in sorted(os.listdir(ref_recipes))]
    for path in paths:
        c = cn.load_encoder_config(path, overrides=dict(n_layers=1))
        assert isinstance(cn.instantiate_encoder(c), cn.ConformerEncoder), path


def test_plan_shards_properties():
    import random

    rnd = random.Random(1234)
    lengths = [rnd.randint(200, 3000) for _ in range(64)]
    for n in (1, 2, 4, 8):
        plan = cn.plan_shards(lengths, n, max_batch=16, bucket_frames=256)
        seen = sorted(i for r in range(n) for i in plan.rank_indices(r))
        assert seen == list(range(64))  # a partition
        assert max(plan.cost) / (sum(plan.cost) / n) < 1.10  # balanced within 10 %
        for r in range(n):
            for sub in plan.batches[r]:
                ls = [lengths[i] for i in sub]
                assert len(sub) <= 16 and max(ls) - min(ls) <= 256
    assert cn.plan_shards(lengths, 4).batches == cn.plan_shards(list(lengths), 4).batches  # deterministic
    empty = cn.plan_shards([], 2)
    assert empty.batches == [[], []]
    ragged = cn.plan_shards([5], 4)
    assert sum(len(b) for b in ragged.batches) == 1


def _oracle_encode(sd, cfg):
    def encode(batch, length):
        return oc.encoder_forward(sd, cfg, batch, length)

    return encode


def test_forward_sharded_matches_unsharded_on_cpu_oracle():
    cfg = oc.EncoderConfig(feat_in=80, n_layers=1, d_model=64, n_heads=4)
    sd = oc.random_state_dict(cfg, 2)
    g = torch.Generator().manual_seed(0)
    lens = [97, 40, 64, 33, 120, 5]
    feats = [torch.randn(80, n, generator=g) for n in lens]
    plan = cn.plan_shards(lens, 2, max_batch=2, bucket_frames=64)
    merged = {}
    for r in range(2):
        merged.update(cn.forward_sharded(_oracle_encode(sd, cfg), feats, plan, r))
    assert sorted(merged) == list(range(len(lens)))
    # Reference semantics: the strided convolutions run over the padded batch, so the last valid frames of a short
    # row see relu(bias) of the padded region (subsampling.py:172-175) -- results depend on the padded extent of the
    # sub-batch an utterance lands in.  The expectation is therefore the oracle on exactly the planned sub-batches.
    for r in range(2):
        for sub in plan.batches[r]:
            t_max = max(lens[i] for i in sub)
            batch = torch.zeros(len(sub), 80, t_max)
            for row, i in enumerate(sub):
                batch[row, :, : lens[i]] = feats[i]
            want, wl = oc.encoder_forward(sd, cfg, batch, torch.tensor([lens[i] for i in sub]))
            for row, i in enumerate(sub):
                got, gl = merged[i]
                assert gl == int(wl[row])
                torch.testing.assert_close(got, want[row, :, :gl], atol=1e-6, rtol=0)
    # a row that is the longest of its sub-batch is unaffected by padding: equal to running it alone
    heads = [sub[0] for r in range(2) for sub in plan.batches[r]]
    for i in heads:
        want, wl = oc.encoder_forward(sd, cfg, feats[i].unsqueeze(0), torch.tensor([lens[i]]))
        got, gl = merged[i]
        assert gl == int(wl[0])


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    cfg = oc.EncoderConfig(feat_in=80, n_layers=1, d_model=64, n_heads=4)
    sd = oc.random_state_dict(cfg, 2)
    g = torch.Generator().manual_seed(0)
    lens = [97, 40, 64, 33, 120, 5, 77]
    feats = [torch.randn(80, n, generator=g) for n in lens]
    plan = cn.plan_shards(lens, world, max_batch=3, bucket_frames=64)
    mine = cn.forward_sharded(_oracle_encode(sd, cfg), feats, plan, rank)
    # no data-path collective: the only exchange is the test's own bookkeeping gather of (index, frames, checksum)
    summary = [(i, n, float(t.double().sum())) for i, (t, n) in sorted(mine.items())]
    gathered = [None] * world
    dist.all_gather_object(gathered, summary)
    dist.barrier()
    if rank == 0:
        q.put(gathered)
    dist.destroy_process_group()


def test_world_size_2_gloo_shards_cover_the_batch():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    gathered = q.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    flat = sorted(x for part in gathered for x in part)
    assert [i for i, _, _ in flat] == list(range(7))
    assert not (set(i for i, _, _ in gathered[0]) & set(i for i, _, _ in gathered[1]))
    # same numbers as a single-process run
    cfg = oc.EncoderConfig(feat_in=80, n_layers=1, d_model=64, n_heads=4)
    sd = oc.random_state_dict(cfg, 2)
    g = torch.Generator().manual_seed(0)
    lens = [97, 40, 64, 33, 120, 5, 77]
    feats = [torch.randn(80, n, generator=g) for n in lens]
    plan = cn.plan_shards(lens, 2, max_batch=3, bucket_frames=64)
    single = {}
    for r in range(2):
        single.update(cn.forward_sharded(_oracle_encode(sd, cfg), feats, plan, r))
    for i, n, checksum in flat:
        assert n == single[i][1]
        assert checksum == pytest.approx(float(single[i][0].double().sum()), abs=1e-3)  # thread-count dependent rounding


def test_plan_shards_auto_bucket_width_trades_padding_against_launch_overhead():
    """bucket_frames="auto": covers every utterance once, is never worse than the fixed widths under the plan's own
    cost model, and uses fewer sub-batches than narrow buckets on a wide length distribution (cfg3)."""
    import random

    from conformer_nemo_b200.sharding import plan_cost, plan_shards

    rnd = random.Random(1234)
    lengths = [rnd.randint(200, 3000) for _ in range(64)]
    for n in (1, 2, 4, 8):
        auto = plan_shards(lengths, n, 64, "auto")
        assert sorted(i for r in range(n) for i in auto.rank_indices(r)) == list(range(64))
        for width in (128, 256, 1024):
            fixed = plan_shards(lengths, n, 64, width)
            assert plan_cost(lengths, auto) <= plan_cost(lengths, fixed) + 1e-6
        assert sum(len(b) for b in auto.batches) < sum(len(b) for b in plan_shards(lengths, n, 64, 128).batches)


def test_packed_layout_host_arithmetic_and_dispatch_rule():
    """Host side of the packed forward (no GPU): the slot arithmetic the wrapper uses to decide and to size things must
    be the one of csrc/common.cuh (slot = T'_b + 15 rows rounded up to 8; T1 = (len + 1) >> 1, T' = (T1 + 1) >> 1 with
    lengths clipped to [0, T]), and the dispatch rule: packed only with host lengths, bf16, no out_proj, >= 15 % saved."""
    enc = cn.ConformerEncoder(feat_in=80, n_layers=1, d_model=64, n_heads=4)

    def model(lens, t):
        rows = 0
        for n in lens:
            n = min(max(n, 0), t)
            t2 = (((n + 1) // 2) + 1) // 2
            rows += -(-(t2 + 15) // 8) * 8
        return rows

    for lens, t in (([1000, 37, 640, 333, 5, 999, 2, 1, 0], 1000), ([2965, 271], 2965), ([400] * 7, 400), ([5000, -3], 1200)):
        assert enc.packed_rows(lens, t) == model(lens, t)
    assert enc.packed_rows([1000], 1000) == 272 and enc.packed_rows([0], 8) == 16
    # a tensor of int32 T' values agrees with calc_length (subsampling.py:272-282) on the same lengths
    lens = [1, 2, 3, 4, 5, 17, 333, 640, 900, 1000, 2001]
    t2 = [(((n + 1) // 2) + 1) // 2 for n in lens]
    assert t2 == oc.subsampled_lengths(torch.tensor(lens), 2).tolist()
    assert enc._want_packed((1000, 100), 2, 1000, 250) and not enc._want_packed((1000, 990), 2, 1000, 250)
    assert not enc._want_packed(None, 2, 1000, 250)
    enc.packed = False
    assert not enc._want_packed((1000, 100), 2, 1000, 250)
    enc.packed = True
    assert enc._want_packed((1000, 990), 2, 1000, 250)
    assert not cn.ConformerEncoder(feat_in=80, n_layers=1, d_model=64, n_heads=4, precision="fp32_validate")._want_packed(
        (1000, 100), 2, 1000, 250)
    assert not cn.ConformerEncoder(feat_in=80, n_layers=1, d_model=64, n_heads=4, feat_out=32)._want_packed(
        (1000, 100), 2, 1000, 250)
    # graph identity: a packed capture is keyed by its lengths, a dense one is not
    k1 = enc.graph_key(2, 1000, torch.float32, True, torch.float32, 0, (1000, 100))
    k2 = enc.graph_key(2, 1000, torch.float32, True, torch.float32, 0, (1000, 200))
    assert k1 != k2 and enc.graph_key(2, 1000, torch.float32, True, torch.float32, 0, None) not in (k1, k2)


def test_one_sub_batch_per_rank_when_buckets_are_unbounded():
    """With the packed forward padding costs nothing, so bench.py / INTEGRATION.md plan with an unbounded bucket width:
    every rank then gets exactly one sub-batch (one launch set) and the LPT balance is untouched."""
    import random

    rnd = random.Random(1234)
    lengths = [rnd.randint(200, 3000) for _ in range(64)]
    for world in (1, 2, 4, 8):
        plan = cn.plan_shards(lengths, world, bucket_frames=1 << 30)
        assert [len(b) for b in plan.batches] == [1] * world
        assert sorted(i for b in plan.batches for s in b for i in s) == list(range(64))
        costs = plan.cost
        assert max(costs) / min(costs) < 1.01
        for b in plan.batches:  # descending lengths inside a share: the interleaved groups of the engine are balanced
            ls = [lengths[i] for i in b[0]]
            assert ls == sorted(ls, reverse=True)
