"""repeat_mask(): per-base repeat masks of many records, the union of the rows scan_batch finds (DESIGN.md section 6,
"Masks").

mask[p] is True if and only if some row (s, e, motif) that api.detect_repeats gives for the record holding base p has
s <= p - record start < e.  The rows are painted by crf_mask_rows on the device; from a CUDA tensor neither the bases, the
rows nor the mask leave HBM.
"""
import sys

import numpy as np

from . import api, batch

#: what the last repeat_mask() call did: the device loads of its scan_batch and the rows it painted
last_stats = {}


def repeat_mask(bases, offsets, filter_settings, device=None, **knobs):
    """Per-base repeat mask of the records bases[offsets[r]:offsets[r+1]] under filter_settings (full mode).

    Takes what batch.scan_batch takes and refuses what it refuses (NotImplementedError for interval attributes,
    min_repeats == 1 and a record longer than one device load).  Host input returns a numpy bool array of len(bases); a
    CUDA torch.uint8 tensor returns a CUDA torch.bool tensor of the same length on the same device, with the same stream
    rule as scan_batch: the caller's current stream is synchronised before the library reads, and the library's stream is
    synchronised before this returns.  Positions outside every record are False."""
    record, start, end, _ = batch.scan_batch(bases, offsets, filter_settings, device, **knobs)
    torch = sys.modules.get("torch")
    on_device = torch is not None and isinstance(bases, torch.Tensor)
    if on_device:
        offsets = offsets.cpu().numpy() if isinstance(offsets, torch.Tensor) else offsets
        n_bases = bases.numel()
    else:
        n_bases = bases.size if isinstance(bases, np.ndarray) else len(bases)
    dst = np.asarray(offsets).astype(np.uint64)[:-1]
    n_rows = int(record.numel() if on_device else record.size)
    last_stats.clear()
    last_stats.update(loads=batch.last_stats["loads"], rows=n_rows)
    if on_device:
        ctx = api.get_context(bases.device.index if device is None else device)
        words = torch.empty((n_bases + 31) // 32, dtype=torch.int32, device=bases.device)
        torch.cuda.current_stream(bases.device).synchronize()        # the row columns may come from torch.cat on it
        ctx.mask_rows(record.data_ptr(), start.data_ptr(), end.data_ptr(), dst, n_bases, n_rows=n_rows,
                      mask=words.data_ptr())
        shifts = torch.arange(8, dtype=torch.uint8, device=bases.device)
        bits = (words.view(torch.uint8).unsqueeze(1) >> shifts) & 1          # little-endian: bit p of the mask is base p
        return bits.view(-1)[:n_bases].view(torch.bool)
    words = api.get_context(device).mask_rows(record, start, end, dst, n_bases)
    return np.unpackbits(words.view(np.uint8), count=n_bases, bitorder="little").view(bool)
