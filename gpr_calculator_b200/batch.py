"""Device-side assembly of covariance rows from a batch of descriptors.

``SO3.calculate_batch(structures, to_host=False)`` leaves x / dxdr / seq on the device; this module
gathers them into the packed layout of the reference (utilities.py:340-390) without a host round
trip: energy item = all atoms of a structure, force item of atom i = every `seq` row with
seq[:, 1] == i, in increasing row order (gaussianprocess.py:857-861, utilities.py:114-117).
"""
import torch


def rows_from_batch(r, centres=None, stress=False):
    """r: dict returned by SO3.calculate_batch(..., to_host=False).

    centres: None (every atom is a force centre) or a list with, per structure, the local atom ids to
    keep (e.g. the atoms not held by FixAtoms), in increasing order.
    stress=True appends the 6 Voigt columns of rdxdr (xx, yy, zz, xy, xz, yz — gaussianprocess.py:862-864) to
    dXdR (9 columns; the descriptor must have been created with stress=True).
    Returns (energy tuple (X [A,d], ELE [A], indices [S]), force tuple (X [R,d], dXdR [R,d,3 or 9], ELE [R],
    indices [NF]) or None when no force centre is kept); tensors live on the device.
    """
    x, dxdr, seq = r['x'], r['dxdr'], r['seq']
    atom_ptr, seq_ptr, numbers = r['atom_ptr'].long(), r['seq_ptr'].long(), r['numbers']
    dev = x.device
    A = x.shape[0]
    S = atom_ptr.numel() - 1
    counts = atom_ptr[1:] - atom_ptr[:-1]
    E = (x, numbers.to(torch.int32), [int(v) for v in counts.cpu()])
    if dxdr is None:
        return E, None
    struct_of = torch.repeat_interleave(torch.arange(S, device=dev), counts)
    centre = torch.repeat_interleave(torch.arange(A, device=dev), seq_ptr[1:] - seq_ptr[:-1])   # global centre atom of row q
    gj = atom_ptr[struct_of[centre]] + seq[:, 1]                                                 # global force atom of row q
    order = torch.sort(gj, stable=True).indices
    n_rows = torch.bincount(gj, minlength=A)
    if centres is not None:
        keep = torch.zeros(A, dtype=torch.bool, device=dev)
        ids = [int(atom_ptr[k]) + int(i) for k, c in enumerate(centres) for i in c]
        if len(ids) == 0:
            return E, None
        keep[torch.as_tensor(ids, dtype=torch.long, device=dev)] = True
        order = order[keep[gj[order]]]
        n_rows = n_rows[keep]
    cen = centre[order]
    dX = dxdr[order]
    if stress:
        if r.get('rdxdr') is None:
            raise ValueError("stress rows need a descriptor created with stress=True (rdxdr)")
        voigt = r['rdxdr'][order].reshape(dX.shape[0], dX.shape[1], 9)[:, :, [0, 4, 8, 1, 2, 5]]
        dX = torch.cat((dX, voigt), dim=2)
    F = (x[cen], dX, numbers[cen].to(torch.int32), [int(v) for v in n_rows.cpu()])
    return E, F


def virial_rows_from_batch(r):
    """Rows of the total stress of every structure of the batch (descriptor created with stress=True).

    The stress rows of rows_from_batch(stress=True) summed over all force items of a structure equal, centre by centre,
    one row per atom with dxdr = sum over that atom's `seq` rows of rdxdr (gprb_virial_rows): the covariance is linear
    in dxdr once x is fixed (DESIGN.md §2).  Returns (energy tuple as rows_from_batch, stress tuple (X [A,d], V [A,d,6],
    ELE [A], indices = atoms per structure)) with V's columns in the order xx, yy, zz, xy, xz, yz."""
    from . import _lib
    from .device import ptr, stream
    if r.get('rdxdr') is None:
        raise ValueError("stress rows need a descriptor created with stress=True (rdxdr)")
    x = r['x']
    atom_ptr = r['atom_ptr'].long()
    E = (x, r['numbers'].to(torch.int32), [int(v) for v in (atom_ptr[1:] - atom_ptr[:-1]).cpu()])
    A, d = x.shape
    seq_ptr = r['seq_ptr'].to(torch.int32).contiguous()
    rdxdr = r['rdxdr'].contiguous()
    V = torch.empty((A, d, 6), dtype=torch.float64, device=x.device)
    _lib.call("gprb_virial_rows", A, d, ptr(seq_ptr), ptr(rdxdr), ptr(V), stream())
    return E, (x, V, E[1], E[2])
