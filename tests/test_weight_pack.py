"""CPU checks of the packed weight table (dvd_b200/weights.py): it holds every pack the tensor modes read and nothing else, and the
library rejects a bf16x3 table that lacks one of the packs only bf16x3 reads.  No GPU: the table is packed on the CPU and the library
calls return before any launch."""
import ctypes as C

import pytest
import torch

LIVE_PACKED_BYTES = 1_235_526_176          # synthetic live-only state dict, every precision's packs


@pytest.fixture(scope="module")
def packed():
    from dvd_b200.weights import PackedWeights
    from oracle import synth
    return PackedWeights(synth.make_state_dict(1234, live_only=True), torch.device("cpu"))


def test_table_holds_what_the_tensor_modes_read(packed):
    T = packed.table
    pairs = [T.emb[i] for i in range(1, 5)] + [T.xattn_in, T.xattn_out, T.blk_qkv, T.blk_proj, T.blk_fc1, T.blk_fc2]
    pairs += [m for L in T.dec for m in (L.fc, L.conv2, L.qkv_ln, L.conv1_ln)] + list(T.pyr_h)
    for m in pairs:                                          # run on 16-bit pairs by bf16x3 (and on the hi by bf16)
        assert m.bf16 and m.bf16_lo
    for L in T.dec:
        assert L.qkv_colsum and L.qkv_cvec and L.conv1_colsum and L.conv1_cvec
    for m in [L.qkv for L in T.dec] + [L.conv1 for L in T.dec] + list(T.pyr):
        assert m.bf16 and not m.bf16_lo                      # bf16 reads the hi; bf16x3 reads qkv_ln, conv1_ln and pyr_h instead
    assert sum(t.nbytes for t in packed.keep) == LIVE_PACKED_BYTES


def _drop_pyr_h(T):
    T.pyr_h[6].bf16_lo = None


def _drop_qkv_ln(T):
    T.dec[0].qkv_ln.bf16 = None


def _drop_conv1_cvec(T):
    T.dec[5].conv1_cvec = None


@pytest.mark.parametrize("field, drop", [("pyr_h[6].bf16_lo", _drop_pyr_h), ("dec[0].qkv_ln.bf16", _drop_qkv_ln),
                                         ("dec[5].conv1_cvec", _drop_conv1_cvec)])
def test_bf16x3_rejects_a_table_without_its_packs(packed, field, drop):
    """Both entry points name the missing field before they look at their inputs (NULL here, so no call can reach a launch; the
    table's pointers are host pointers and no call may ever get a complete one)."""
    from dvd_b200 import _lib
    lib = _lib.lib()
    T = _lib.Weights.from_buffer_copy(packed.table)
    drop(T)
    ws, docs, n_hyp = C.c_void_p(1 << 20), 1, 2             # 256-byte aligned, never dereferenced
    ws_bytes = lib.dvd_workspace_bytes(docs, n_hyp, _lib.PREC_BF16X3)

    def static(prec):
        return lib.dvd_static_forward(C.byref(T), ws, ws_bytes, docs, n_hyp, prec, None, None, None, None, None)

    def step(prec):
        return lib.dvd_denoise_step(C.byref(T), ws, ws_bytes, docs, n_hyp, prec, None, None, None, 1, None, 1.0, 0.0, None, None, None)

    for call in (static, step):
        assert call(_lib.PREC_BF16X3) == -1
        assert field in lib.dvd_last_error().decode()
        assert call(_lib.PREC_BF16) == -1                    # bf16 reads none of these packs: it gets as far as the NULL inputs
        assert "null" in lib.dvd_last_error().decode()
