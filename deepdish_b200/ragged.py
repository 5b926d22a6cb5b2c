"""Ragged detection batches (host side; no CUDA needed).

The reference hands ``Tracker.update`` a Python list of ``Detection`` objects per stream (deepdish.py:1014).  Its
batched equivalent on the wire between host and device is ONE contiguous blob per block of streams::

    i32 offsets[n + 1]                 stream s owns entries offsets[s] .. offsets[s + 1]
    (pad to 16 bytes)
    f64 tlwh[N][4]   f32 conf[N]   i32 label[N]          N = offsets[n]
    (pad to 16 bytes)
    f32 feat[N][128]
    (pad to 16 bytes)                  only when the batch carries frame presence:
    u8 present[n]                      nonzero = the stream has a frame this tick; an absent stream owns no entries

holding only the detections that exist -- what ``dd_engine_step_host`` / ``dd_engine_step_host_present`` /
``dd_unpack_detections`` read (include/deepdish_b200.h).  ``section_offsets`` is the single definition of the layout.
"""
import numpy as np

FEAT_DIM = 128


def section_offsets(n_streams, n_total, present=False):
    """Byte offsets (tlwh, conf, label, feat) -- with ``present``: (tlwh, conf, label, feat, present) -- and the total
    size of a blob with n_total detections."""
    o_tlwh = (4 * (n_streams + 1) + 15) // 16 * 16
    o_conf = o_tlwh + 32 * n_total
    o_label = o_conf + 4 * n_total
    o_feat = (o_label + 4 * n_total + 15) // 16 * 16
    end = o_feat + 4 * FEAT_DIM * n_total
    if not present:
        return (o_tlwh, o_conf, o_label, o_feat), end
    o_present = (end + 15) // 16 * 16
    return (o_tlwh, o_conf, o_label, o_feat, o_present), o_present + n_streams


def pack(tlwh, conf, label, feat, count, out=None, present=None):
    """Padded arrays of a block of streams (tlwh [n,D,4] f64, conf [n,D] f32, label [n,D] i32, feat [n,D,128] f32,
    count [n]) -> (blob u8 ndarray, total bytes, section offsets).  ``out``: a writable u8 buffer to fill (e.g. the
    numpy view of a pinned torch tensor); allocated when None.
    ``present`` (bool-like [n], optional): frame presence of each stream.  The blob then ends with the presence section
    and five section offsets are returned; an absent stream owns no entries and its count is ignored.  With None the
    blob and the four offsets are those of a batch without presence."""
    count = np.asarray(count, dtype=np.int64)
    n, D = conf.shape
    if present is not None:
        present = np.asarray(present).astype(bool)
        if present.shape != (n,):
            raise ValueError("present must have shape (%d,), got %s" % (n, present.shape))
        count = np.where(present, count, 0)
    if count.size and (int(count.max()) > D or int(count.min()) < 0):
        raise ValueError("detection counts must lie in [0, %d]" % D)
    offs = np.zeros(n + 1, dtype=np.int32)
    offs[1:] = np.cumsum(count)
    N = int(offs[-1])
    sections, total = section_offsets(n, N, present is not None)
    o_tlwh, o_conf, o_label, o_feat = sections[:4]
    b = np.zeros(max(total, 16), dtype=np.uint8) if out is None else out
    if b.size < total:
        raise ValueError("output buffer too small (%d < %d bytes)" % (b.size, total))
    sel = np.arange(D)[None, :] < count[:, None]
    b[:4 * (n + 1)].view(np.int32)[:] = offs
    b[o_tlwh:o_conf].view(np.float64)[:] = np.asarray(tlwh, np.float64)[sel].reshape(-1)
    b[o_conf:o_label].view(np.float32)[:] = np.asarray(conf, np.float32)[sel]
    b[o_label:o_label + 4 * N].view(np.int32)[:] = np.asarray(label, np.int32)[sel]
    b[o_feat:o_feat + 4 * FEAT_DIM * N].view(np.float32)[:] = np.asarray(feat, np.float32)[sel].reshape(-1)
    if present is not None:
        b[o_feat + 4 * FEAT_DIM * N:sections[4]] = 0
        b[sections[4]:total] = present
    return b, total, sections


def unpack(blob, n_streams, max_dets, present=False):
    """Inverse of ``pack`` on the host (what the device kernels do): -> padded (tlwh, conf, label, feat, count);
    ``present=True`` reads a blob packed with presence and appends its bool presence [n_streams] to the tuple."""
    offs = np.asarray(blob[:4 * (n_streams + 1)]).view(np.int32)
    N = int(offs[-1])
    sections, total = section_offsets(n_streams, N, present)
    o_tlwh, o_conf, o_label, o_feat = sections[:4]
    count = np.diff(offs).astype(np.int32)
    tlwh = np.zeros((n_streams, max_dets, 4)); conf = np.zeros((n_streams, max_dets), np.float32)
    label = np.zeros((n_streams, max_dets), np.int32); feat = np.zeros((n_streams, max_dets, FEAT_DIM), np.float32)
    sel = np.arange(max_dets)[None, :] < count[:, None]
    tlwh[sel] = np.asarray(blob[o_tlwh:o_conf]).view(np.float64).reshape(-1, 4)
    conf[sel] = np.asarray(blob[o_conf:o_label]).view(np.float32)
    label[sel] = np.asarray(blob[o_label:o_label + 4 * N]).view(np.int32)
    feat[sel] = np.asarray(blob[o_feat:o_feat + 4 * FEAT_DIM * N]).view(np.float32).reshape(-1, FEAT_DIM)
    if present:
        return tlwh, conf, label, feat, count, np.asarray(blob[sections[4]:total]) != 0
    return tlwh, conf, label, feat, count
