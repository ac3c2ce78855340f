"""CPU checks of ngcf_spmm's argument validation: every rejected argument is refused with its own message before any
CUDA call, so these run without a device.  (The return code alone would not show that: any CUDA call made without a
device fails too.)  The GPU side of the contract is tests/test_spmm_contract_gpu.py."""
import ctypes

import pytest

from seoul_tourism_recommendation_ngcf_b200 import _lib

P = 1 << 12                                        # a dummy device address, 16-byte aligned; never dereferenced


def _csr(n_rows=0, n_hub=0):
    """An ngcf_csr whose pointers are dummies.  n_rows == 0: a call that passes validation returns before any CUDA
    call, so a check that is missing shows as a return of 0 here."""
    s = _lib.NgcfCsr()
    s.n_rows = n_rows
    for f in ("rowptr", "ent", "tiles", "hub_of_row", "hub_chunk_ptr", "chunk_ptr", "hub_ent", "chunk_row",
              "chunk_tiles", "hub_rows", "hub_done", "tile_hubmask"):
        setattr(s, f, P if (f in ("rowptr", "ent") or n_hub) else None)
    s.n_hub = s.n_chunks = s.n_chunk_tiles = n_hub
    return s


def _args(**kw):
    a = dict(csr=_csr(), X=P, ldx=64, d=64, addend=None, ld_add=0, slot=None, gsum=None, ld_gsum=0, hub_partial=None,
             drop_p=0.0, seed=0, seed_dev=None, layer=0, transposed=0, row_offset=0, keep_bits=None, c_ent=None,
             c_cnt=None, Y=2 * P, ldy=64)
    a.update(kw)
    return a


def _spmm(a):
    lib = _lib.load()
    return lib.ngcf_spmm(ctypes.byref(a["csr"]), a["X"], a["ldx"], a["d"], a["addend"], a["ld_add"], a["slot"],
                         a["gsum"], a["ld_gsum"], a["hub_partial"], a["drop_p"], a["seed"], a["seed_dev"], a["layer"],
                         a["transposed"], a["row_offset"], a["keep_bits"], a["c_ent"], a["c_cnt"], a["Y"], a["ldy"],
                         None)


def test_valid_arguments_on_an_empty_csr_return_before_any_cuda_call():
    assert _spmm(_args()) == 0
    assert _spmm(_args(ldx=(1 << 30) - 4, addend=2 * P, ld_add=64, slot=3 * P, gsum=4 * P, ld_gsum=88)) == 0
    assert _spmm(_args(addend=3 * P, ld_add=100)) == 0           # an out-of-place addend may have its own pitch


@pytest.mark.parametrize("kw,msg", [
    (dict(X=None), b"null pointer"),
    (dict(Y=None), b"null pointer"),
    (dict(d=0), b"width 0"),
    (dict(d=129), b"width 129"),
    (dict(ldx=63), b"leading dimension"),
    (dict(ldy=63), b"leading dimension"),
    (dict(ldx=1 << 30), b"below 2^30"),                          # ldx * 4 would wrap the 32-bit byte stride
    (dict(ldx=(1 << 30) + 4), b"below 2^30"),
    (dict(addend=2 * P, ld_add=68), b"in-place addend"),         # addend == Y with a pitch other than ldy
    (dict(drop_p=1.0), b"drop_p"),
    (dict(drop_p=-0.5), b"drop_p"),
    (dict(layer=8), b"layer 8"),
    (dict(layer=-1), b"layer -1"),
    (dict(row_offset=-1), b"row_offset -1"),
    (dict(row_offset=1 << 31), b"row_offset"),
    (dict(slot=3 * P), b"slot given without gsum"),
    (dict(c_ent=3 * P), b"c_ent and c_cnt go together"),
    (dict(c_cnt=3 * P), b"c_ent and c_cnt go together"),
    (dict(csr=_csr(n_hub=1)), b"hub_partial scratch missing"),
    (dict(csr=_csr(n_rows=10), d=65, ldx=65, ldy=65, c_ent=3 * P, c_cnt=4 * P), b"compacted survivor lists"),
    (dict(csr=_csr(n_rows=10), ldx=66, c_ent=3 * P, c_cnt=4 * P), b"compacted survivor lists"),   # not a vector pitch
], ids=[
    "null_X", "null_Y", "d0", "d129", "ldx_below_d", "ldy_below_d", "ldx_2pow30", "ldx_2pow30_plus4",
    "inplace_addend_pitch", "drop_p_1", "drop_p_negative", "layer8", "layer_negative", "row_offset_negative",
    "row_offset_2pow31", "slot_without_gsum", "c_ent_without_c_cnt", "c_cnt_without_c_ent",
    "hubs_without_hub_partial", "compacted_at_d65", "compacted_at_odd_ldx"
])
def test_spmm_rejects_bad_arguments_before_any_cuda_call(kw, msg):
    assert _spmm(_args(**kw)) != 0
    err = _lib.load().ngcf_last_error()
    assert b"spmm" in err and msg in err, err
