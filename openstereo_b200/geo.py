"""Host-side mirror of the reference's combined geometry-encoding volume (SURVEY.md section 8(f) row 1).

``CombinedGeoEncodingVolume(init_fmap1, init_fmap2, geo_volume, num_levels=2, radius=4)`` and ``obj(disp, coords)`` have
the reference's signature and return value (stereo/modeling/models/stereobase/gru_blocks.py:169-229;
``Combined_Geo_Encoding_Volume`` stereo/modeling/models/igev/geometry.py:7-66 is the same class under IGEV's name).  What
differs is the data layout: the geometry volume stays (B, C, D, H, W) -- no (B*H*W, C, 1, D) permuted copy -- the pyramid
is built by the pair-average kernel, and one gather kernel per GRU iteration writes the (B, L*(C+1)*(2r+1), H, W) feature
map directly instead of grid tensors + 2L grid_sample calls + cat + permute.  CUDA only: there is no CPU fallback.
"""
import torch

from . import ops


class CombinedGeoEncodingVolume:
    def __init__(self, init_fmap1, init_fmap2, geo_volume, num_levels=2, radius=4):
        if not (geo_volume.is_cuda and init_fmap1.is_cuda and init_fmap2.is_cuda):
            raise RuntimeError("CombinedGeoEncodingVolume: CUDA tensors required (the reference class serves CPU tensors)")
        self.num_levels, self.radius = int(num_levels), int(radius)
        corr = self.corr(init_fmap1.float(), init_fmap2.float())                   # (B, H, W1, 1, W2)
        b, h, w1, _, w2 = corr.shape
        self.geo_volume_pyramid = [geo_volume.float().contiguous()]               # native (B, C, D, H, W)
        self.init_corr_pyramid = [corr.reshape(b, h, w1, w2)]
        for _ in range(self.num_levels - 1):
            self.geo_volume_pyramid.append(ops.avgpool_pairs(self.geo_volume_pyramid[-1], 2))
            self.init_corr_pyramid.append(ops.avgpool_pairs(self.init_corr_pyramid[-1], 3))

    def __call__(self, disp, coords):
        return ops.geo_lookup(self.geo_volume_pyramid, self.init_corr_pyramid, disp, coords, self.radius)

    @staticmethod
    def corr(fmap1, fmap2):
        """All-pairs row correlation (gru_blocks.py:222-229): a batched fp32 GEMM, left to cuBLAS."""
        b, _, h, w1 = fmap1.shape
        w2 = fmap2.shape[-1]
        with torch.autocast("cuda", enabled=False):                 # fp32 also when the model is evaluated under autocast
            corr = torch.einsum('aijk,aijh->ajkh', fmap1, fmap2)
        return corr.reshape(b, h, w1, 1, w2).contiguous()


Combined_Geo_Encoding_Volume = CombinedGeoEncodingVolume          # IGEV's spelling (igev/geometry.py:7)
context_upsample = ops.context_upsample
