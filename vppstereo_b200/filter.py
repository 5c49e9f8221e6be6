"""Drop-in for the reference's filter.py occlusion heuristic, the producer of the VPP occlusion mask (test.py:154):

    from vppstereo_b200.filter import occlusion_heuristic     # instead of  from filter import occlusion_heuristic (test.py:17)
    mask_occ = occlusion_heuristic(hints)[1]

Same signature and return value as filter.py:246-292: `(dmap, conf_map)` = the hints that survive the warp / weighted
window / un-warp round trip (gaps of one pixel linearly filled) and the binary mask (0 = visible hint, 1 elsewhere).
numpy in -> numpy out; CUDA tensors ([H,W] or a batch [N,H,W]) in -> CUDA tensors out, so the mask can go straight into
`vpp(..., g_occ=mask)` without a host hop.  Maps are float32 (what test.py passes); other dtypes are converted.
"""
from . import _lib

__all__ = ["occlusion_heuristic"]


def occlusion_heuristic(dmap, rx=9, ry=7, l=2, g=0.4375, th_conf=1, th_filter=0.1):
    torch = _lib.require_cuda()
    host = not _lib.is_tensor(dmap)
    d = _lib.as_device(dmap, torch.float32)
    if d.dim() not in (2, 3):
        raise ValueError("dmap must be [H,W] or [N,H,W]")
    H, W = d.shape[-2:]
    n = d.shape[0] if d.dim() == 3 else 1
    out = torch.empty_like(d)
    conf = torch.empty(d.shape, dtype=torch.uint8, device=d.device)
    with torch.cuda.device(d.device):
        ws = _lib.workspace(_lib.lib().vppb200_occlusion_workspace_bytes(H, W, n), d.device, tag="occ")
        _lib.call("vppb200_occlusion_heuristic", _lib.ptr(d), _lib.ptr(out), _lib.ptr(conf), W, H, int(rx), int(ry), float(l),
                  float(g), float(th_conf), float(th_filter), _lib.ptr(ws), ws.numel(), n, _lib.stream_ptr(d.device),
                  what="occlusion_heuristic")
    if host:
        return out.cpu().numpy(), conf.cpu().numpy()
    return out, conf
