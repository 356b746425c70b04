"""CPU checks of samd_draft_assemble's host-side validation: a bad shape is refused with a clear samd_last_error()
message before anything touches a device."""
import ctypes as C

import pytest


def _args(**kw):
    from samd_b200 import _cabi as K
    a = K.AssembleArgs()
    a.batch, a.n_nodes, a.n_paths, a.depth, a.kv_len, a.mask_dtype, a.draft_stride = 4, 16, 16, 16, 64, K.DTYPE_FP16, 16
    fake = 4096                                             # never dereferenced: validation happens first
    a.draft_dev = a.draft_len_dev = a.cache_len_dev = fake
    a.out_tokens_dev = a.out_position_ids_dev = a.out_n_nodes_dev = a.out_n_paths_dev = a.out_retrieve_dev = fake
    a.out_mask_dev = fake
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("bad, msg", [
    (dict(n_nodes=0), "n_nodes"), (dict(n_nodes=257, kv_len=300), "n_nodes"), (dict(n_paths=0), "n_paths"),
    (dict(depth=0), "depth"), (dict(kv_len=15), "kv_len"), (dict(mask_dtype=7), "dtype"), (dict(batch=0), "batch"),
    (dict(draft_dev=None), "sequence drafts"), (dict(out_mask_dev=None), "output"),
    (dict(tree_tokens_dev=4096), "tree drafts need"),
    (dict(tree_tokens_dev=4096, type_dev=4096, tree_parents_dev=4096, tree_depth_dev=4096, tree_n_dev=4096,
          tree_retrieve_dev=4096, tree_shape_dev=4096, tree_stride=17, tree_max_paths=16, tree_max_depth=16), "tree_stride"),
    (dict(tree_tokens_dev=4096, type_dev=4096, tree_parents_dev=4096, tree_depth_dev=4096, tree_n_dev=4096,
          tree_retrieve_dev=4096, tree_shape_dev=4096, tree_stride=16, tree_max_paths=17, tree_max_depth=16), "P x D"),
])
def test_draft_assemble_validates_on_the_host(bad, msg):
    from samd_b200 import _cabi as K
    rc = K.lib().samd_draft_assemble(C.byref(_args(**bad)), None)
    assert rc != 0
    assert msg in K.lib().samd_last_error().decode()
