"""``mfrec.lib.als_implicit`` on a B200: alternating least squares for implicit-feedback WRMF.

``als_wrmf`` keeps the reference's signature (mfrec/lib/als_implicit.pyx:211-225); ``m`` and
``m_inv`` are scratch matrices there and are accepted and ignored here; ``u`` and ``v`` are updated
in place; returns ``None``.  With more than one entry in ``options["devices"]`` the call is split
over those devices (``mfrec_train_als_wrmf_multi``) and gives the one-device result bit for bit.
``als_wrmf_dense`` (the dense-matrix development variant, :68-205) is out of scope."""
import numpy as np

from mfrec_b200 import _native
from mfrec_b200.lib._buffers import buffer_arg, options


def als_wrmf(nbr_epochs, dim, u, v, m, m_inv, ratings_users_row, ratings_users_col, ratings_items_row,
             ratings_items_col, nbr_users, nbr_items, c_pos=1, k=0.015, verbose=0):
    dim = int(dim)
    buffer_arg(u, "u", np.float64, 2)
    buffer_arg(v, "v", np.float64, 2)
    for name, a in (("ratings_users_row", ratings_users_row), ("ratings_users_col", ratings_users_col),
                    ("ratings_items_row", ratings_items_row), ("ratings_items_col", ratings_items_col)):
        buffer_arg(a, name, np.int32, 1, writable=False)
    if dim != u.shape[0] or dim != v.shape[0]:
        raise ValueError("dim=%d does not match the factor arrays (%d, %d features)" % (dim, u.shape[0], v.shape[0]))
    if u.shape[1] != int(nbr_items) or v.shape[1] != int(nbr_users):
        raise ValueError("u / v do not have nbr_items / nbr_users columns")
    if verbose:
        for epoch in range(int(nbr_epochs)):
            print('Epoch : ' + str(epoch))
    if len(options["devices"]) > 1:
        _native.train_als_wrmf_multi(options["devices"], int(nbr_epochs), dim, u, v, ratings_users_row,
                                     ratings_users_col, ratings_items_row, ratings_items_col, int(nbr_users),
                                     int(nbr_items), c_pos, k)
        return None
    _native.train_als_wrmf(int(nbr_epochs), dim, u, v, ratings_users_row, ratings_users_col,
                           ratings_items_row, ratings_items_col, int(nbr_users), int(nbr_items), c_pos, k,
                           ctx=_native.default_context(options["device"]))
    return None


def als_wrmf_dense(*_a, **_k):
    raise NotImplementedError("als_wrmf_dense is a development variant of the reference on a dense "
                              "users x items matrix and is not part of the B200 path; see DESIGN.md")
