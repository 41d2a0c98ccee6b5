"""Driver used under ncu / for timing: co-transition counting on synthetic contact-map
families (BASELINE config 4 shape).  Prints the sort and the counting kernel separately."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from cherryml_b200 import _lib
from cherryml_b200.counting._device import build_bucket_table_tiles, count_raw, sorted_grid
from cherryml_b200.synthetic import as_device_batch, quantization_grid, synthetic_co

fams = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
device = torch.device("cuda", 0)
grid = quantization_grid()
K = len(grid)
gd = torch.from_numpy(sorted_grid(grid)).to(device)
dev = as_device_batch(synthetic_co(fams, 1024, 300, seed=11, device=device), device)
tab = build_bucket_table_tiles(dev, gd, K)
lib = _lib.load()
order = torch.empty(dev.n_pairs, dtype=torch.int32, device=device)
recs = torch.empty(dev.n_pairs * 16, dtype=torch.uint8, device=device)
ws = torch.empty(2 * (K + 2), dtype=torch.int32, device=device)
raw = torch.zeros((K, 400, 400), dtype=torch.int32, device=device)
st = _lib.current_stream_ptr()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
for it in range(reps + 1):
    ev[0].record()
    _lib.check(lib.cherry_sort_pairs_by_bucket(_lib.ptr(tab), dev.r_pad, dev.n_pairs, K, _lib.ptr(dev.fams),
                                               _lib.ptr(dev.pair_a), _lib.ptr(dev.pair_b), _lib.ptr(dev.pair_fam),
                                               _lib.ptr(order), _lib.ptr(recs), _lib.ptr(ws), st), "sort")
    ev[1].record()
    _lib.check(lib.cherry_count_co(_lib.ptr(dev.msa), _lib.ptr(recs), _lib.ptr(ws), dev.n_pairs,
                                   dev.max_row_stride, K, 20, _lib.ptr(raw), st), "count")
    ev[2].record()
    torch.cuda.synchronize()
    if it == 0:
        continue
    ms_sort, ms = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
    print(f"families {fams} items {dev.n_sites_examined} sort_ms {ms_sort:.3f} count_ms {ms:.3f} "
          f"items/s {dev.n_sites_examined / ms * 1e3:.3e} residue GB/s {dev.msa.numel() / ms / 1e6:.1f} "
          f"counted {int(raw.sum(dtype=torch.int64).item())}")
