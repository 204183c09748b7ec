"""-m gpu: the CUDA path (through the C ABI) against the CPU oracle, bit-exact."""
import numpy as np
import pytest

from draco_sharp_b200 import _native as N
from draco_sharp_b200 import synth_gen as G

from common import cloud, compare_with_oracle, gpu_decode_all

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("scheme", [1, 0, -1])
def test_positions_small_sizes(gpu_decoder, scheme):
    bufs = [cloud(n, seed=10 + n, scheme=scheme) for n in (0, 1, 2, 3, 4, 5, 7, 8, 33, 100, 1000, 4099)]
    gpu = gpu_decode_all(gpu_decoder, bufs)
    assert compare_with_oracle(gpu, bufs) == len(bufs)


@pytest.mark.parametrize("scheme", [1, 0, -1])
def test_positions_normals_colors(gpu_decoder, scheme):
    bufs = [cloud(n, seed=77 + n, scheme=scheme, normal_bits=10, colors=1) for n in (1, 6, 257, 5000)]
    bufs += [cloud(3000, seed=5, scheme=scheme, pos_bits=0, normal_bits=7, colors=0),
             cloud(3000, seed=6, scheme=scheme, pos_bits=0, normal_bits=0, colors=1),
             cloud(2000, seed=7, scheme=scheme, pos_bits=22, normal_bits=12, colors=1),
             cloud(2000, seed=8, scheme=scheme, pos_bits=1, normal_bits=2, colors=1)]
    gpu = gpu_decode_all(gpu_decoder, bufs)
    assert compare_with_oracle(gpu, bufs) == len(bufs)


def test_config2_shape_batch(gpu_decoder):
    """BASELINE config 2 shape at a size the oracle finishes in seconds: 48 clouds x 100k points, 14-bit."""
    bufs = [cloud(100000, seed=0xD5AC0000 + k, scheme=1) for k in range(48)]
    gpu = gpu_decode_all(gpu_decoder, bufs, want=("out", "qints"))
    assert compare_with_oracle(gpu, bufs) == len(bufs)


def test_ragged_batch_mixed_schemes(gpu_decoder):
    rng = np.random.default_rng(3)
    bufs = []
    for k in range(40):
        n = int(rng.integers(0, 20000))
        bufs.append(cloud(n, seed=1000 + k, scheme=int(rng.integers(-1, 2)), normal_bits=int(rng.choice([0, 8, 10])),
                          colors=int(rng.integers(0, 2)), pos_bits=int(rng.choice([0, 8, 11, 14, 16, 20]))))
    gpu = gpu_decode_all(gpu_decoder, bufs)
    assert compare_with_oracle(gpu, bufs) == len(bufs)


def test_wide_alphabets(gpu_decoder):
    """Precisions 15..20 (u32 tables, global-memory tables): large deltas over wide quantisation."""
    bufs = [cloud(60000, seed=40 + i, scheme=1, pos_bits=pb, rho=rho)
            for i, (pb, rho) in enumerate([(16, (999, 1000)), (20, (9999, 10000)), (18, (9999, 10000)), (14, (199, 200))])]
    gpu = gpu_decode_all(gpu_decoder, bufs)
    assert compare_with_oracle(gpu, bufs) == len(bufs)


def test_malformed_buffers_status_parity(gpu_decoder):
    """Truncated and bit-flipped buffers: per-buffer status codes (the reference's exception sites) must agree
    with the oracle, and one bad buffer must not poison its neighbours."""
    rng = np.random.default_rng(11)
    good = [cloud(3000, seed=90, scheme=1, normal_bits=10, colors=1), cloud(3000, seed=91, scheme=0, colors=1)]
    bufs = []
    for g in good:
        bufs.append(g)
        for cut in (0, 3, 5, 9, 11, 16, 30, 40, 60, 100, len(g) // 2, len(g) - 9, len(g) - 1):
            bufs.append(g[:cut].copy())
        for _ in range(60):
            b = g.copy()
            pos = int(rng.integers(0, min(len(b), 1400)))
            b[pos] ^= np.uint8(1 << int(rng.integers(0, 8)))
            bufs.append(b)
    gpu = gpu_decode_all(gpu_decoder, bufs, want=("out",))
    n_ok = compare_with_oracle(gpu, bufs)
    assert n_ok >= 2


def test_full_size_checksums(gpu_decoder):
    """Size-independent property at a large batch: the word checksum of every decoded attribute equals the
    checksum of the generator's source values pushed through the reference dequantisation formula."""
    sp = G.make_spec(100000, seed=0xD5AC0000, scheme=1, colors=1)
    arena, offs, lens, sums, schemes, used = G.synth_batch(sp, 256)
    batch = gpu_decoder.index_arena(arena, offs, lens)
    out, _ = gpu_decoder.decode(batch)
    assert batch.points == 256 * 100000
    for k in range(256):
        assert batch.status(k) == 0
        a0 = batch.attr_info(k, 0)
        a1 = batch.attr_info(k, 1)
        assert G.word_checksum(out[a0.out_off: a0.out_off + a0.out_bytes]) == int(sums[k, 0])
        assert G.word_checksum(out[a1.out_off: a1.out_off + a1.out_bytes]) == int(sums[k, 2])
    st = gpu_decoder.stats()
    assert st.n_launches >= 1
    batch.free()


def test_resident_decode_into_torch_tensor(gpu_decoder):
    """Split form: upload once, decode into caller-owned device memory (a torch tensor), twice, same bytes."""
    import torch
    sp = G.make_spec(20000, seed=5, scheme=-1, normal_bits=10, colors=1)
    arena, offs, lens, sums, schemes, used = G.synth_batch(sp, 32)
    batch = gpu_decoder.index_arena(arena, offs, lens)
    gpu_decoder.upload(batch)
    out = torch.zeros(batch.out_bytes, dtype=torch.uint8, device="cuda")
    gpu_decoder.decode_resident(batch, dev_out=out.data_ptr())
    first = out.cpu().numpy().copy()
    out.zero_()
    gpu_decoder.decode_resident(batch, dev_out=out.data_ptr())
    assert np.array_equal(first, out.cpu().numpy())
    bufs = [arena[int(o): int(o + l)] for o, l in zip(offs, lens)]
    host, _ = gpu_decoder.decode(gpu_decoder.index(bufs))
    for k in range(32):
        for a in range(3):
            ai = batch.attr_info(k, a)
            assert np.array_equal(first[ai.out_off: ai.out_off + ai.out_bytes], host[ai.out_off: ai.out_off + ai.out_bytes])
    batch.free()


@pytest.mark.parametrize("scheme", [-1, 0])
@pytest.mark.parametrize("slices", [3, 8])
def test_pipeline_slices_match_single_shard(gpu_decoder, scheme, slices):
    """The same device listed K times in dcb_create = K pipeline slices (contiguous buffer runs, own streams, own
    arenas): every decoded byte and status equals the single-shard decode."""
    import draco_sharp_b200 as D
    sp = G.make_spec(20000, seed=0xD5AC0100, scheme=scheme, normal_bits=10, colors=1)
    arena, offs, lens, sums, schemes, used = G.synth_batch(sp, 37)
    arena = arena.copy()
    arena[int(offs[5]) + 40] ^= 0x55  # one damaged buffer: must fail alone, in its own slice
    one = gpu_decoder.index_arena(arena, offs, lens)
    ref, _ = gpu_decoder.decode(one)
    dec = D.DracoBatchDecoder([0] * slices)
    try:
        many = dec.index_arena(arena, offs, lens)
        out, _ = dec.decode(many)
        assert many.out_bytes == out.nbytes
        devs = set()
        for k in range(37):
            assert many.status(k) == one.status(k)
            devs.add(many.buffer_info(k).device)
            if one.status(k):
                continue
            for a in range(3):
                x, y = one.attr_info(k, a), many.attr_info(k, a)
                assert x.out_bytes == y.out_bytes
                assert np.array_equal(ref[x.out_off: x.out_off + x.out_bytes], out[y.out_off: y.out_off + y.out_bytes]), (k, a)
        assert len(devs) == slices
        many.free()
    finally:
        dec.close()
        one.free()


def test_library_shards_a_batch_across_distinct_devices(gpu_decoder):
    """dcb_create with DISTINCT device ids (SURVEY 8e): the library's own sharding -- longest-processing-time-first by
    compressed bytes, one host thread per physical device, no collective -- against the single-device decode.  Needs a
    machine with at least two GPUs; skipped where there is one."""
    import draco_sharp_b200 as D
    from draco_sharp_b200 import _native as Nn
    n_dev = Nn.lib().dcb_device_count()
    if n_dev < 2:
        pytest.skip("needs at least two GPUs")
    for scheme in (-1, 0):
        sp = G.make_spec(30000, seed=0xD5AC0200 + scheme, scheme=scheme, normal_bits=10, colors=1)
        arena, offs, lens, sums, schemes, used = G.synth_batch(sp, 61)
        arena = arena.copy()
        arena[int(offs[7]) + 40] ^= 0x55
        one = gpu_decoder.index_arena(arena, offs, lens)
        ref, _ = gpu_decoder.decode(one)
        dec = D.DracoBatchDecoder(list(range(n_dev)))
        try:
            many = dec.index_arena(arena, offs, lens)
            out, _ = dec.decode(many)
            devs = set()
            for k in range(61):
                assert many.status(k) == one.status(k)
                devs.add(many.buffer_info(k).device)
                if one.status(k):
                    continue
                for a in range(3):
                    x, y = one.attr_info(k, a), many.attr_info(k, a)
                    assert np.array_equal(ref[x.out_off: x.out_off + x.out_bytes], out[y.out_off: y.out_off + y.out_bytes]), (k, a)
            assert len(devs) == n_dev
            many.free()
        finally:
            dec.close()
            one.free()


def test_uniform_lut_fallback_path_is_bit_exact_too():
    """DCB_NO_SPLIT=1 forces every Raw stream through the uniform-LUT probe (the path tables take when they cannot
    satisfy the two-region LUT); the switch is read once per process, so the parity cases re-run in a child."""
    import os
    import subprocess
    import sys
    if os.environ.get("DCB_NO_SPLIT"):
        pytest.skip("already the child")
    env = dict(os.environ, DCB_NO_SPLIT="1", DCB_NO_DIRECT="1")  # small batches would take the direct slot LUT otherwise
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(here, "test_gpu_parity.py"), "-q", "-x", "-m", "gpu", "-k",
                        "positions_small_sizes or positions_normals_colors or ragged_batch or wide_alphabets"],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


def _rerun_in_child(extra_env, select):
    import os
    import subprocess
    import sys
    if os.environ.get("DCB_TEST_CHILD"):
        pytest.skip("already the child")
    env = dict(os.environ, DCB_TEST_CHILD="1", **extra_env)
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "pytest", here, "-q", "-x", "-m", "gpu", "-k", select],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


_PATH_CASES = ("positions_small_sizes or positions_normals_colors or ragged_batch or wide_alphabets or crafted_streams or "
               "malformed_buffers or house_positions or grid_meshes or parallelogram_random")


def test_two_level_tables_single_warp_kernels_are_bit_exact():
    """Small batches are planned with the direct slot LUT (few streams per SM); DCB_NO_DIRECT=1 sends the same cases
    through the two-level tables and the one-warp-per-CTA kernels, the path of the big batches (BASELINE configs[1])."""
    _rerun_in_child({"DCB_NO_DIRECT": "1"}, _PATH_CASES)


def test_two_level_tables_warp_pair_kernels_are_bit_exact():
    """DCB_RANS_PC=1 + DCB_NO_DIRECT=1: chain / consumer warp pairs over the two-level tables (kept as an experiment
    path: measured slower than one warp per sub-partition when the SM is full of streams)."""
    _rerun_in_child({"DCB_NO_DIRECT": "1", "DCB_RANS_PC": "1"}, _PATH_CASES)


def test_bucket_record_kernels_are_bit_exact():
    """DCB_REC=1 + DCB_NO_DIRECT=1: the bucket-record tables of dcb_rans_rec.cu (one dependent shared-memory access per
    symbol; taken for every group whose tables have the shape, the others keep the two-level kernels)."""
    _rerun_in_child({"DCB_NO_DIRECT": "1", "DCB_REC": "1"}, _PATH_CASES)


def test_split_layout_of_the_warp_pair_kernels_is_bit_exact():
    """DCB_SPLIT=1: chain warps on sub-partitions 0..2, every consumer warp on sub-partition 3 (both pair kernels)."""
    _rerun_in_child({"DCB_NO_DIRECT": "1", "DCB_REC": "1", "DCB_SPLIT": "1"}, "positions_small_sizes or positions_normals_colors or ragged_batch or crafted_streams")
    _rerun_in_child({"DCB_NO_DIRECT": "1", "DCB_RANS_PC": "1", "DCB_SPLIT": "1"}, "positions_small_sizes or positions_normals_colors or ragged_batch or crafted_streams")
