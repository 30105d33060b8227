"""CPU-only tests of the host layer: the C-ABI library loads and exports every symbol include/pnp_b200.h declares
(no compute calls -- there is no GPU here), the TF-style variable registry reproduces the reference's checkpoint
naming contract, entry-point configuration mirrors train_gan.py, error behaviour of the layers.py surface, arena layout,
and the world_size-2 data-parallel path over gloo."""
import ctypes
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import pnp_b200
    from pnp_b200 import _C
    hdr = open(os.path.join(ROOT, "include", "pnp_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(pnp_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 40
    lib = ctypes.CDLL(_C.LIB_PATH)
    missing = [n for n in declared if not hasattr(lib, n)]
    assert not missing, missing
    # the ctypes table mirrors the header one to one
    bound = set(_C.SIGNATURES) | {"pnp_error_string", "pnp_version", "pnp_tc_available", "pnp_tc_last_config", "pnp_tc_last_pair"}
    assert set(declared) == bound, (set(declared) ^ bound)
    assert _C.lib.pnp_version() >= 100
    assert _C.lib.pnp_error_string(100002).decode().startswith("pnp: unsupported")
    # the tcgen05 path reports itself available exactly on a Blackwell (compute capability 10.x) device
    on_sm100 = torch.cuda.is_available() and torch.cuda.get_device_capability()[0] == 10
    assert _C.lib.pnp_tc_available() == int(on_sm100)


def test_no_cpu_fallback_product_does_not_import_oracle():
    """the product path must never route through the oracle (or any CPU fallback)"""
    pkg = os.path.join(ROOT, "medical-cross-modality-domain-adaptation_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), fn
            assert "oracle." not in src, fn


def test_variable_names_follow_reference_checkpoint_contract():
    import pnp_b200
    from pnp_b200 import runtime as rt, source_segmenter as seg, adversarial as adv
    from pnp_b200.train_gan import configure
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_var_names.json")))
    net = seg.Full_DRN(channels=3, n_class=5, batch_size=2, cost_kwargs={"cross_flag": True, "miu_cross": 1.0, "miu_dice": 1.0})
    names = set(rt.graph.order)
    assert set(gold["old_bn_list"]) <= names
    assert len(names) == 33 + 120
    # L2 list quirk of source_segmenter.py:132-135: wr4_4 twice, wr4_3 never
    v = rt.graph.vars
    assert sum(1 for w in net.conv_weights if w is v["group_4/Variable_3"]) == 2
    assert sum(1 for w in net.conv_weights if w is v["group_4/Variable_2"]) == 0
    ck, nc, tc = configure("train-gan")
    anet = adv.Full_DRN(channels=3, n_class=5, batch_size=2, cost_kwargs=ck, network_config=nc)
    names = set(rt.graph.order)
    for key in ("half_zip_mri_vars", "half_zip_ct_vars"):
        assert not [n for n in gold[key] if n not in names], key
    leafs = set(n.split("/", 1)[1] for n in names if "/" in n)
    assert not [n for n in gold["pred_bn_list"] if n not in leafs]
    # adversarial.py:478-501: membership by name substring
    assert all("cls" in x.pnp_name for x in anet.cls_vars) and len(anet.cls_vars) == 26 + 24 * 4
    assert all("adapt" in x.pnp_name for x in anet.adapt_vars) and len(anet.adapt_vars) == 21 + 20 * 4
    assert len(anet.cls_weights) == 2 * len(anet.cls_weights_unique)     # appended on both create_classifier calls
    tr = adv.Trainer(anet, num_cls=5, batch_size=2, opt_kwargs={"learning_rate": 3e-4}, train_config=tc)
    # clip_op: exactly the cls vars whose name contains "Variable"
    clipped = [x.pnp_name for x, c in zip(tr.d_vars, tr.dis_optimizer.seg_clip.tolist()) if c > 0]
    assert clipped and all("Variable" in n for n in clipped) and len(clipped) == 26
    assert all(abs(c - 0.03) < 1e-9 for c in tr.dis_optimizer.seg_clip.tolist() if c > 0)
    # arena: every variable is a view of the flat arena, 1024-float aligned
    for x, (o, n) in zip(tr.d_vars, tr.d_arena.offsets):
        assert o % 1024 == 0 and x.data_ptr() == tr.d_arena.theta.data_ptr() + 4 * o and x.grad.data_ptr() == tr.d_arena.grad.data_ptr() + 4 * o
    # weight decay = gradient of dis_reg / dis_sub_iter (critic weights counted twice), lambda-scaled for the mask critic
    wd = dict(zip([x.pnp_name for x in tr.d_vars], tr.dis_optimizer.seg_wd.tolist()))
    base = 1e-4 * 0.002 * 2 / tc["dis_sub_iter"]
    assert abs(wd["cls_scope/cls_1/Variable"] - base) < 1e-12 and abs(wd["mask_cls_scope/mask_cls_1/Variable"] - 0.3 * base) < 1e-12
    assert wd["cls_scope/cls_1/cls_1_1/gamma"] == 0.0


def test_scope_registry_semantics():
    import pnp_b200
    from pnp_b200 import runtime as rt, layers as L
    rt.reset_default_graph()
    with rt.variable_scope("group_1"):
        a = L.weight_variable([3, 3, 3, 16])
        b = L.weight_variable([3, 3, 16, 16])
        c = L.sharable_weight_variable([3, 3, 16, 16], name="Variable_7")
        c2 = L.sharable_weight_variable([3, 3, 16, 16], name="Variable_7")
    assert (a.pnp_name, b.pnp_name, c.pnp_name) == ("group_1/Variable", "group_1/Variable_1", "group_1/Variable_7") and c is c2
    bn1 = L.bn_variables(None, 8)
    bn2 = L.bn_variables(None, 8)
    assert bn1.gamma.pnp_name == "BatchNorm/gamma" and bn2.gamma.pnp_name == "BatchNorm_1/gamma"
    assert float(bn1.gamma.sum()) == 8 and float(bn1.moving_var.sum()) == 8 and float(bn1.beta.abs().sum()) == 0
    w = L.weight_variable([1000], stddev=0.01)
    assert float(w.abs().max()) <= 0.02 + 1e-7        # truncated normal: |z| <= 2 sigma
    assert float(L.bias_variable([4]).sum()) == pytest.approx(0.4)


def test_train_gan_phase_configuration():
    from pnp_b200.train_gan import configure
    ck, nc, tc = configure("pre-train")
    assert ck["lambda_mask_loss"] == 0 and nc["ct_front_trainable"] is False and tc["gen_interval"] == 0 and tc["dis_sub_iter"] == 1
    assert tc["restore_from_baseline"] and tc["training_iters"] == 201 and tc["epochs"] == 100
    ck, nc, tc = configure("train-gan")
    assert ck["lambda_mask_loss"] == 0.3 and nc["ct_front_trainable"] is True and tc["dis_sub_iter"] == 20 and tc["gen_sub_iter"] == 1
    assert tc["iter_upd_interval"] == 300 and tc["dis_sub_iter_inc"] == 1 and tc["lr_decay_factor"] == 0.98
    ck, nc, tc = configure("fine-tune")
    assert tc["dis_sub_iter"] == 30 and tc["lr_update"] is False
    with pytest.raises(Exception, match="Please set a training phase!"):
        configure(None)


def test_layers_error_behaviour_without_a_gpu():
    import pnp_b200
    from pnp_b200 import layers as L, ops, functional as F
    x = torch.zeros(2, 8, 8, 4)
    w = torch.zeros(3, 3, 4, 4)
    with pytest.raises(UnboundLocalError):          # layers.py:17-25 leaves conv_2d unbound for unknown padding strings
        L.conv2d(x, w, 1.0, padding="REFLECT")
    with pytest.raises(ValueError):
        L.conv2d(x, w, 1.0, strides=[1, 2, 1, 1])
    with pytest.raises(ValueError):
        L.simple_concat2d(torch.zeros(2, 8, 8, 1), torch.zeros(2, 4, 8, 1))
    with pytest.raises(ValueError):
        L.crop_and_concat(torch.zeros(2, 4, 8, 1), torch.zeros(2, 8, 8, 3))           # x1 smaller than x2: nothing to crop
    with pytest.raises(ValueError):
        L.cross_entropy(torch.zeros(2, 8, 8, 2), torch.zeros(2, 8, 8, 3))
    with pytest.raises(ValueError):
        L.max_pool2d(x, 0)
    with pytest.raises(ValueError):
        L.avg_pool2d(x, -1)
    with pytest.raises(ValueError):
        ops.PS(torch.zeros(2, 4, 4, 64), 8, n_channel=1, batch_size=3)
    with pytest.raises(ValueError):
        ops.PS(torch.zeros(1, 4, 5, 64), 8, n_channel=1, batch_size=1)
    assert F.same_pad(256, 3, 2) == (0, 1) and F.same_pad(128, 5, 2) == (1, 2) and F.same_pad(16, 5, 4) == (0, 1)
    g = F._geometry((2, 4, 4, 4), (3, 3, 4, 4), F.LayerCfg(stride=2, padding="SYMMETRIC"))
    assert g[0] == 1 and (g[1].H, g[1].Ho, g[1].pad_t) == (6, 2, 0)


def test_confusion_matrix_metrics_match_oracle():
    from pnp_b200.lib import _dice, _jaccard, _label_decomp
    from oracle import tf14_numpy as N
    rng = np.random.RandomState(0)
    lab, pred = rng.randint(0, 5, (2, 16, 16)), rng.randint(0, 5, (2, 16, 16))
    cm = np.zeros((5, 5), np.int64)
    np.add.at(cm, (lab.ravel(), pred.ravel()), 1)
    y = N.label_decomp(5, lab)
    assert np.array_equal(_label_decomp(5, lab), y)
    d, arr = N.dice_eval(pred, y.astype(np.float64), 5)
    assert np.allclose(_dice(cm), arr, atol=1e-6)
    inter = np.diag(cm).astype(np.float64)
    assert np.allclose(_jaccard(cm), inter / (cm.sum(0) + cm.sum(1) - inter))


def _dp_worker(rank, world, port, out):
    # host ranks over gloo: hide any GPU, which would otherwise have to exist once per LOCAL_RANK
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      CUDA_VISIBLE_DEVICES="")
    sys.path.insert(0, ROOT)
    import pnp_b200  # noqa: F401
    from pnp_b200 import parallel
    parallel.init_from_env(backend="gloo")
    dp = parallel.DataParallel()
    g = torch.full((2048,), float(rank + 1))
    scale = dp.allreduce(g)
    theta = torch.full((8,), float(rank))
    dp.broadcast_params(theta)
    out[rank] = (dp.world, dp.rank, scale, float(g[0]), float(theta[0]))
    dp.barrier()
    torch.distributed.destroy_process_group()


def test_data_parallel_gloo_world_size_2():
    """one all-reduce over the flat gradient arena; the optimizer's grad_scale = 1/N turns the sum into the average of the
    per-rank reference steps (SURVEY 8e parity definition)"""
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    out = mgr.dict()
    port = 29500 + os.getpid() % 2000
    mp.spawn(_dp_worker, args=(2, port, out), nprocs=2, join=True)
    for r in (0, 1):
        world, rank, scale, gsum, th = out[r]
        assert world == 2 and rank == r and scale == 0.5
        assert gsum == 3.0 and gsum * scale == 1.5      # (1 + 2) / 2
        assert th == 0.0                                # rank 0's parameters everywhere


def test_checkpoint_transplant_chain_baseline_to_gan(tmp_path):
    """SURVEY 8f #1: train_segmenter.py checkpoint -> `--phase pre-train` initialisation:
    restore(no_gan=True) takes only group*/output* conv weights (adversarial.py:514-532), load_batch_norm_weights maps the
    baseline's anonymous BatchNorm_k scopes onto group_g/pred_* in creation order (lists/old_bn_list -> lists/pred_bn_list,
    adversarial.py:743-765), adapt_copy_weights clones the MR front into the CT DAM (lists/half_zip_*_vars, :706-741)."""
    import pnp_b200
    from pnp_b200 import runtime as rt, source_segmenter as seg, adversarial as adv
    from pnp_b200.lib import _save
    from pnp_b200.train_gan import configure
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_var_names.json")))
    seg.Full_DRN(channels=3, n_class=5, batch_size=2, cost_kwargs={"cross_flag": True, "miu_cross": 1.0, "miu_dice": 1.0})
    rng = np.random.RandomState(3)
    base = {n: rng.randn(*v.shape).astype(np.float32) for n, v in rt.graph.vars.items()}
    rt.load_state_dict(base)
    ck = _save(rt.state_dict(), str(tmp_path / "model.cpkt"), global_step=7)
    assert ck.endswith("model.cpkt-7.npz")
    c, nc, tc = configure("pre-train")
    net = adv.Full_DRN(channels=3, n_class=5, batch_size=2, cost_kwargs=c, network_config=nc)
    before = {n: v.detach().clone() for n, v in rt.graph.vars.items()}
    net.restore(ck, no_gan=True)
    net.load_batch_norm_weights(ck)
    net.adapt_copy_weights()
    v = rt.graph.vars
    # conv weights of the frozen segmenter come from the baseline, name for name
    for n in base:
        if "/Variable" in n:
            assert np.array_equal(v[n].cpu().numpy(), base[n]), n
    # BN: old_bn_list[i] -> pred_bn_list[i]  (the reference's two lists are index-aligned)
    scope_of = {}
    for n in v:
        if "/pred_" in n:
            scope_of[n.split("/", 1)[1]] = n
    for old, new in zip(gold["old_bn_list"], gold["pred_bn_list"]):
        assert np.array_equal(v[scope_of[new]].cpu().numpy(), base[old]), (old, new)
    # DAM initialised from the MR front: half_zip_mri_vars[i] -> half_zip_ct_vars[i]
    for m, c_ in zip(gold["half_zip_mri_vars"], gold["half_zip_ct_vars"]):
        assert np.array_equal(v[c_].cpu().numpy(), v[m].cpu().numpy()), (m, c_)
    # critics untouched
    for n in v:
        if "cls" in n:
            assert torch.equal(v[n], before[n]), n


def test_tfrecord_reader_round_trip_and_reference_slicing(tmp_path):
    """SURVEY 8f #2: the reference's TFRecord schema (README.md:49-64) decoded without TensorFlow; label = middle slice"""
    from pnp_b200 import tfrecord as tfr
    assert tfr.crc32c(b"123456789") == 0xE3069283                      # CRC-32C check value
    rng = np.random.RandomState(0)
    files = []
    truth = []
    for i in range(5):
        img = rng.randn(256, 256, 3).astype(np.float32)
        lab = rng.randint(0, 5, (256, 256, 3)).astype(np.float32)
        p = str(tmp_path / ("s%d.tfrecords" % i))
        tfr.write_record(p, [tfr.encode_example(img, lab)])
        files.append(p)
        truth.append((img, lab))
    ex = tfr.parse_example(next(tfr.read_records(files[2])))
    assert ex["dsize_dim0"] == [256] and ex["dsize_dim2"] == [3] and ex["lsize_dim1"] == [256] and len(ex["data_vol"]) == 256 * 256 * 3 * 4
    x, y = tfr.decode_slice(next(tfr.read_records(files[2])))
    assert np.array_equal(x, truth[2][0]) and np.array_equal(y, truth[2][1][:, :, 1].astype(np.int64))
    src = tfr.TFRecordSource(files, batch_size=3, seed=1)
    xb, yb = src.next()
    assert tuple(xb.shape) == (3, 256, 256, 3) and xb.dtype == torch.float32 and tuple(yb.shape) == (3, 256, 256) and yb.dtype == torch.int64
    xb2, _ = src.next()                                                    # wraps around the 5-file list
    assert tuple(xb2.shape) == (3, 256, 256, 3)
    # corruption is detected
    raw = bytearray(open(files[0], "rb").read())
    raw[100] ^= 0xFF
    open(files[0], "wb").write(bytes(raw))
    with pytest.raises(IOError):
        list(tfr.read_records(files[0]))


def test_io_library_exports_every_declared_symbol_and_crc32c_known_answers():
    """include/pnp_io.h <-> libpnp_io.so <-> _io.SIGNATURES, and the CRC32C known-answer vectors of RFC 3720 B.4 on BOTH
    code paths (SSE4.2 instruction / slicing-by-8 tables)"""
    from pnp_b200 import _io
    hdr = open(os.path.join(ROOT, "include", "pnp_io.h")).read()
    declared = sorted(set(re.findall(r"\b(pnp_[a-z0-9_]+)\s*\(", hdr)))
    lib = ctypes.CDLL(_io.LIB_PATH)
    assert declared and not [n for n in declared if not hasattr(lib, n)]
    assert set(declared) == set(_io.SIGNATURES), set(declared) ^ set(_io.SIGNATURES)
    kat = [(b"123456789", 0xE3069283), (bytes(32), 0x8A9136AA), (b"\xff" * 32, 0x62A8AB43), (bytes(range(32)), 0x46DD794E),
           (bytes(range(31, -1, -1)), 0x113FDB5C), (b"", 0x00000000)]
    for data, want in kat:
        assert _io.lib.pnp_crc32c(data, len(data)) == want, (data[:8], hex(want))
        assert _io.lib.pnp_crc32c_sw(data, len(data)) == want
    rng = np.random.RandomState(3)
    for n in (1, 7, 8, 9, 63, 1000, 65537):          # unaligned heads / tails
        buf = rng.bytes(n + 3)
        for off in (0, 1, 3):
            view = buf[off:off + n]
            assert _io.lib.pnp_crc32c(view, n) == _io.lib.pnp_crc32c_sw(view, n)
    assert _io.lib.pnp_masked_crc32c(b"123456789", 9) == ((((0xE3069283 >> 15) | (0xE3069283 << 17)) & 0xFFFFFFFF) + 0xA282EAD8) & 0xFFFFFFFF


def test_native_tfrecord_decoder_matches_the_python_parser_and_rejects_corruption(tmp_path):
    """pnp_tfrecord_load_file (C: framing + CRC + protobuf + decode_raw + middle-slice label) == the hand-written Python parser
    that is itself pinned to the reference's next_batch (test_reference_graph_trace.py); multi-record files; error codes"""
    from pnp_b200 import tfrecord as tfr, _io
    rng = np.random.RandomState(1)
    exs = [(rng.randn(256, 256, 3).astype(np.float32), rng.randint(0, 5, (256, 256, 3)).astype(np.float32)) for _ in range(3)]
    multi = str(tmp_path / "multi.tfrecords")
    tfr.write_record(multi, [tfr.encode_example(i, l) for i, l in exs])
    raw = open(multi, "rb").read()
    assert _io.lib.pnp_tfrecord_count(raw, len(raw)) == 3
    for k, payload in enumerate(tfr.read_records(multi)):
        xi, yi = tfr.decode_slice(payload)
        xn, yn = tfr.load_slice(multi, k)
        assert np.array_equal(xi, xn) and np.array_equal(yi, yn) and yn.dtype == np.int64
        assert np.array_equal(yn, exs[k][1][:, :, 1].astype(np.int64))
    with pytest.raises(IOError, match="index"):
        tfr.load_slice(multi, 3)
    bad = bytearray(raw)
    bad[5000] ^= 0x01
    p2 = str(tmp_path / "bad.tfrecords")
    open(p2, "wb").write(bytes(bad))
    with pytest.raises(IOError, match="CRC"):
        tfr.load_slice(p2, 0)
    tfr.load_slice(p2, 0, check_crc=False)                   # the flipped bit sits inside the image bytes: decodable without the check
    open(p2, "wb").write(raw[:100000])
    with pytest.raises(IOError, match="truncated"):
        tfr.load_slice(p2, 0)
    with pytest.raises(IOError, match="open"):
        tfr.load_slice(str(tmp_path / "missing.tfrecords"), 0)
    other = str(tmp_path / "other.tfrecords")                # a valid record that does not follow the schema
    tfr.write_record(other, [b"\x0a\x02\x0a\x00"])
    with pytest.raises(IOError, match="schema"):
        tfr.load_slice(other, 0)


def test_threaded_tfrecord_source_shuffles_and_delivers_every_example(tmp_path):
    """4 reader threads + shuffle buffer (tf.train.shuffle_batch semantics): every file is delivered, batches are assembled in
    alternating pinned buffers, a reader error surfaces in next()"""
    from pnp_b200 import tfrecord as tfr
    files = []
    for i in range(12):
        img = np.full((256, 256, 3), float(i), np.float32)
        lab = np.full((256, 256, 3), float(i % 5), np.float32)
        p = str(tmp_path / ("e%02d.tfrecords" % i))
        tfr.write_record(p, [tfr.encode_example(img, lab)])
        files.append(p)
    src = tfr.TFRecordSource(files, batch_size=4, seed=5, num_threads=4, capacity=8, min_after_dequeue=4)
    seen, orders = [], []
    for _ in range(9):                                        # 36 examples = 3 epochs of 12
        x, y = src.next()
        ids = [int(v) for v in x[:, 0, 0, 0]]
        assert all(int(y[j, 0, 0]) == ids[j] % 5 for j in range(4))
        seen += ids
        orders.append(ids)
    src.close()
    assert set(seen) == set(range(12)) and max(seen.count(i) for i in range(12)) <= 4
    assert orders[0] != sorted(orders[0]) or orders[1] != sorted(orders[1])            # shuffled
    # synchronous mode is deterministic
    a = tfr.TFRecordSource(files, 4, seed=7, num_threads=0)
    b = tfr.TFRecordSource(files, 4, seed=7, num_threads=0)
    assert torch.equal(a.next()[0], b.next()[0])
    os.remove(files[3])
    bad = tfr.TFRecordSource(files, 4, seed=5, num_threads=2, capacity=8, min_after_dequeue=4)
    with pytest.raises(IOError):
        for _ in range(8):
            bad.next()
    bad.close()


def test_conv_routing_table_matches_the_kernel_contract():
    """host-side routing (functional._tc_candidate) against the channel contract documented in include/pnp_b200.h:
    forward / data gradient on tcgen05 when Cin and Cout are each 64k, 32 or 16; weight gradient when Cin in {32, 64k}
    and Cout = 64k; everything else (3/5/40-channel ends) on the general fp32 kernels."""
    from pnp_b200 import functional as F
    from pnp_b200._C import ConvGeom

    def g(cin, cout, k=3, s=1):
        return ConvGeom(8, 64, 64, cin, 64 // s, 64 // s, cout, k, k, s, 1, 1, 1)

    assert F.TC_K32 and F.TC_K16
    F._tc_declined.clear()
    yes = [("fwd", 512, 512), ("dgrad", 512, 2560), ("wgrad", 64, 64), ("fwd", 32, 64), ("dgrad", 32, 64), ("wgrad", 32, 64),
           ("fwd", 16, 16), ("dgrad", 16, 32), ("fwd", 16, 32), ("fwd", 64, 320), ("wgrad", 128, 256)]
    no = [("fwd", 3, 16), ("fwd", 40, 5), ("dgrad", 40, 5), ("fwd", 5, 16), ("wgrad", 16, 16), ("wgrad", 16, 32), ("wgrad", 32, 32),
          ("fwd", 48, 64), ("fwd", 64, 24)]
    for kind, ci, co in yes:
        assert F._tc_candidate(kind, g(ci, co)), (kind, ci, co)
    for kind, ci, co in no:
        assert not F._tc_candidate(kind, g(ci, co)), (kind, ci, co)
    assert not F._tc_candidate("fwd", g(64, 64, k=7))            # more than 25 taps
    # a shape the library declined once is not offered again
    F._tc_declined.add(F._gkey("fwd", g(16, 64)))
    assert not F._tc_candidate("fwd", g(16, 64))
    F._tc_declined.clear()
    # producers emit operand planes exactly for the tensors a tcgen05 convolution can consume
    assert [bool(F._want_planes(c)) for c in (16, 32, 64, 320, 5, 40, 48)] == ([True, True, True, True, False, False, False]
                                                                                if F._tc_mode() else [False] * 7)


def _bucket_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import pnp_b200  # noqa: F401
    from pnp_b200 import parallel, optim
    torch.manual_seed(0)
    vs = [torch.zeros(n) for n in (3000, 10, 5000, 700, 1, 2048, 900)]
    for i, v in enumerate(vs):
        v.pnp_name = "v%d" % i
    arena = optim.Arena(vs)
    dp = parallel.DataParallel()
    red = dp.attach(arena, n_buckets=3)
    assert red is not None and len(red.bounds) >= 2 and red.bounds[0][0] == 0 and red.bounds[-1][1] == arena.total
    res = []
    for step in range(3):
        arena.grad.zero_()
        dp.begin_backward(arena)
        # "backward": variables complete from the back, v5 receives two contributions per step (a shared critic weight)
        for i in (6, 5, 5, 4, 3, 2, 1, 0):
            vs[i].grad.add_(float(rank + 1) * (i + 1 + step))
            v = vs[i]
            v._pnp_grad_hook(v)
            if step > 0 and i == 2:
                launched_early = list(red.launched)
        scale = dp.finish_backward(arena)
        res.append([float(v.grad.flatten()[0]) for v in vs])
    # passive mode: local gradients stay local until finish
    arena.grad.zero_()
    dp.begin_backward(arena, overlap=False)
    for i in (6, 5, 5, 4, 3, 2, 1, 0):
        vs[i].grad.add_(float(rank + 1))
        vs[i]._pnp_grad_hook(vs[i])
    local = float(vs[6].grad[0])
    dp.finish_backward(arena)
    out[rank] = (res, scale, launched_early, local, float(vs[6].grad[0]), red.expected)
    # a step with an extra contribution must raise instead of reducing a half-written bucket
    dp.begin_backward(arena)
    err = None
    try:
        for i in (6, 6):
            vs[i]._pnp_grad_hook(vs[i])
        for i in (6,):
            vs[i]._pnp_grad_hook(vs[i])
    except RuntimeError as e:
        err = str(e)
    out["err%d" % rank] = err
    dist.barrier()
    dist.destroy_process_group()


def test_bucketed_overlapped_allreduce_gloo_world_size_2():
    """parallel.BucketedAllReduce: calibration step = one call; later steps launch each bucket as soon as its last contribution
    is in (before the 'backward' has finished), results equal the plain sum; passive mode keeps local gradients"""
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_bucket_worker, args=(2, 29700 + os.getpid() % 2000, out), nprocs=2, join=True)
    for r in (0, 1):
        res, scale, launched_early, local, after, expected = out[r]
        assert scale == 0.5 and sum(expected.values()) == 8
        for step in range(3):
            for i in range(7):
                mult = 2 if i == 5 else 1
                assert res[step][i] == 3.0 * mult * (i + 1 + step), (step, i, res[step][i])
        assert any(launched_early), "no bucket was reduced before the backward pass ended"
        assert local == float(r + 1) and after == 3.0
        assert out["err%d" % r] is not None and "more gradient contributions" in out["err%d" % r]


def test_entry_scripts_read_the_reference_list_files(tmp_path):
    """train_segmenter.py:60-61 / train_gan.py:69-72: `_read_lists` on ./lists/*_list (None when the file is absent, as in lib.py:11-12);
    a present list selects the TFRecord source of that stream -- training AND validation --, an absent one the synthetic source, and a
    list that points at missing data stops the run instead of silently training on synthetic slices."""
    import pnp_b200  # noqa: F401
    from pnp_b200 import tfrecord as tfr, source_segmenter as S, adversarial as A
    from pnp_b200.lib import _read_lists
    from pnp_b200.train_segmenter import resolve_lists
    from pnp_b200.train_gan import configure
    rng = np.random.RandomState(4)
    lists = tmp_path / "lists"
    lists.mkdir()
    truth = {}
    for name, n in (("mr_train_list", 3), ("mr_val_list", 2), ("ct_train_list", 3)):
        files = []
        for i in range(n):
            img = rng.randn(256, 256, 3).astype(np.float32)
            lab = rng.randint(0, 5, (256, 256, 3)).astype(np.float32)
            p = str(tmp_path / ("%s_%d.tfrecords" % (name, i)))
            tfr.write_record(p, [tfr.encode_example(img, lab)])
            files.append(p)
            truth[p] = img
        (lists / name).write_text("\n".join(files) + "\n\n")              # trailing blank lines are skipped (len < 3)
    assert _read_lists(str(lists / "ct_val_list")) is None
    assert _read_lists(str(lists / "mr_val_list")) == [str(tmp_path / ("mr_val_list_%d.tfrecords" % i)) for i in range(2)]
    mr_train, mr_val, ct_train, ct_val = resolve_lists(*[str(lists / n) for n in ("mr_train_list", "mr_val_list", "ct_train_list",
                                                                                  "ct_val_list")], False)
    assert len(mr_train) == 3 and len(mr_val) == 2 and len(ct_train) == 3 and ct_val == []
    assert resolve_lists(str(lists / "mr_train_list"), True) == [[]]                           # --synthetic
    (lists / "broken_list").write_text(str(tmp_path / "gone.tfrecords") + "\n")
    with pytest.raises(IOError, match="does not exist"):
        resolve_lists(str(lists / "broken_list"), False)

    # ---- the segmenter loop draws its training batches from train_list and its validation batches from val_list
    net = S.Full_DRN(3, 5, 2, cost_kwargs={"cross_flag": True, "miu_cross": 1.0, "dice_flag": True, "miu_dice": 1.0})
    tr = S.Trainer(net, train_list=mr_train, val_list=mr_val, num_cls=5, batch_size=2, opt_kwargs={"learning_rate": 1e-3}, optimizer="adam")
    seen = {"train": [], "val": []}
    tr.feed = lambda images, raw: (images, raw)
    tr.train_step = lambda x, y, keep_prob=0.75: seen["train"].append(x.clone()) or (0.0, 0.0)
    tr.output_minibatch_stats = lambda x, y, step=None, log_dir=None: 0.0
    tr.val_stats = lambda x, y, step=None, log_dir=None, detail=False: seen["val"].append(x.clone()) or {}
    tr.train(output_path=str(tmp_path / "seg"), training_iters=3, epochs=1, display_step=2)
    imgs = lambda lst: [truth[p] for p in lst]
    member = lambda x, pool: any(np.array_equal(x.cpu().numpy(), im) for im in pool)
    assert len(seen["train"]) == 3 and len(seen["val"]) == 2
    assert all(member(b[k], imgs(mr_train)) for b in seen["train"] for k in range(2))
    assert all(member(b[k], imgs(mr_val)) for b in seen["val"] for k in range(2))

    # ---- the GAN loop: MR from its lists, CT training from its list, CT validation (no list) from the synthetic stream
    ck, nc, tc = configure("pre-train")
    tc.update(training_iters=3, epochs=1)
    anet = A.Full_DRN(3, 5, 2, cost_kwargs=ck, network_config=nc)
    atr = A.Trainer(anet, mr_train, mr_val, ct_train, ct_val, num_cls=5, batch_size=2, opt_kwargs={"learning_rate": 3e-4}, train_config=tc)
    got = {"d": [], "mon": []}
    atr.d_step = lambda mr, ct, keep_prob=0.75, apply=True: got["d"].append((mr.clone(), ct.clone()))
    atr.g_step = lambda ct, keep_prob=0.75, apply=True: None
    atr.output_minibatch_stats = lambda step, ct, cty, mr, mry, log_dir=None, detail=False: got["mon"].append((detail, ct.clone(), mr.clone()))
    atr.train(output_path=str(tmp_path / "gan"), restore=False, training_iters=3, epochs=1, display_step=2)
    assert len(got["d"]) == 2 and len(got["mon"]) == 4
    assert all(member(mr[k], imgs(mr_train)) and member(ct[k], imgs(ct_train)) for mr, ct in got["d"] for k in range(2))
    for detail, ct, mr in got["mon"]:
        assert all(member(mr[k], imgs(mr_val) if detail else imgs(mr_train)) for k in range(2))
        assert all(member(ct[k], imgs(ct_train)) != detail for k in range(2))            # validation CT: synthetic, not from a list
