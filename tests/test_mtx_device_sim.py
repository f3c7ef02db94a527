""".mtx ingest on the device on the CPU emulation (tests/cusim): the kernels and the host orchestration of
osp_readcoo_device run without a GPU and must give the triplets of the host loader osp_readcoo, as raw 32-bit words.
The cases are tests/test_gpu_mtx_device.py's (which runs them on a B200); the out-of-memory and leak checks need the
emulated device's allocation counter and run here only."""
import pytest

import outerspace_b200 as osp
from outerspace_b200 import api
import test_engine_sim as es
import test_gpu_mtx_device as gm
import test_host_loaders as hl


@pytest.fixture(scope="module", autouse=True)
def emulated_library(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("cusim_mtx") / "libosp_b200_cusim.so")
    es._build_emulation(out)
    saved = (api._LIB_PATH, api._lib)
    api._LIB_PATH, api._lib = out, None
    try:
        yield api.load_library()
    finally:
        api._LIB_PATH, api._lib = saved


@pytest.fixture(scope="module")
def engine(emulated_library):
    eng = osp.Engine(0)
    yield eng
    eng.close()


test_fuzz_texts_match_the_host_loader = gm.test_fuzz_texts_match_the_host_loader
test_every_odd_value = gm.test_every_odd_value
test_line_shapes = gm.test_line_shapes
test_long_comment_and_wide_lines = gm.test_long_comment_and_wide_lines
test_indices_at_the_edges = gm.test_indices_at_the_edges
test_significant_digits_and_exponents = gm.test_significant_digits_and_exponents
test_nul_bytes_in_lines = gm.test_nul_bytes_in_lines
test_no_few_and_only_slow_lines = gm.test_no_few_and_only_slow_lines
test_garbage_line_and_missing_file = gm.test_garbage_line_and_missing_file
test_host_coo_has_no_device_pointers = gm.test_host_coo_has_no_device_pointers
test_to_csr_matches_host_coo2csr = gm.test_to_csr_matches_host_coo2csr
test_mtx_to_device_operands_to_product = gm.test_mtx_to_device_operands_to_product


def test_device_out_of_memory_is_reported_not_fatal(emulated_library, monkeypatch, tmp_path):
    """A device too small for the text, the per-line scratch, the slow lines or the triplets: OSP_ERR_OOM from whichever
    allocation fails, nothing leaked, and the context works afterwards."""
    path = str(tmp_path / "fuzz.mtx")
    hl._write(path, 3000, 7)
    with open(path, "rb") as f:
        text = f.read()
    rc, want, nrow, ncol = gm.host_readcoo(text, True)
    assert rc == 0
    eng = osp.Engine(0)
    try:
        warm = eng.readcoo_buffer_device(text, sym=True)            # the arena and the pool of the context, at full size
        warm.free()
        base = es._live_bytes(emulated_library)
        failures, messages = 0, set()
        # every 16 KB, and byte by byte where the text fits but its few bytes of tile counts do not
        for extra in [k << 14 for k in range(75)] + list(range(len(text) - 256, len(text) + 256, 8)) + [4 << 20]:
            monkeypatch.setenv("CUSIM_DEVICE_MB", repr((base + extra) / (1 << 20)))
            for reader in (lambda: eng.readcoo_buffer_device(text, sym=True), lambda: eng.readcoo_device(path, sym=True)):
                try:
                    dev = reader()
                except osp.OspError as e:
                    assert e.code == api.OSP_ERR_OOM, str(e)
                    failures += 1
                    messages.add(str(e))
                    assert es._live_bytes(emulated_library) == base, f"leak after: {e}"
                    continue
                gm.same_triplets(dev, want, nrow, ncol, f"device with {extra} bytes to spare")
                dev.free()
                assert es._live_bytes(emulated_library) == base
        assert failures >= 4
        for what in ("text", "tile counts", "line scratch", "slow lines", "slow entries", "triplet allocation"):
            assert any(f"osp_readcoo_device: {what}" in m for m in messages), (what, messages)
        monkeypatch.delenv("CUSIM_DEVICE_MB")
        gm.check_text(eng, text)
    finally:
        eng.close()


def test_device_coo_is_freed_with_its_context(emulated_library):
    before = es._live_bytes(emulated_library)
    eng = osp.Engine(0)
    dev = eng.readcoo_buffer_device(b"3 3 2\n1 1 2\n3 2 -1\n")     # noqa: F841 -- left alive on purpose
    res = dev.to_csr(3)                                              # noqa: F841
    assert es._live_bytes(emulated_library) > before
    eng.close()
    assert es._live_bytes(emulated_library) == before

