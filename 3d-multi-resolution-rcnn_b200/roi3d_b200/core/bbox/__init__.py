from .assigners import AssignResult, MaxIoUAssigner
from .geometry import bbox_overlaps
from .samplers import RandomSampler, SamplingResult
from .transforms import bbox2delta3d, bbox2roi3D, bbox2roi3D_padded, delta2bbox3D

__all__ = ['bbox2roi3D', 'bbox2roi3D_padded', 'delta2bbox3D', 'bbox2delta3d', 'bbox_overlaps', 'MaxIoUAssigner',
           'AssignResult', 'RandomSampler', 'SamplingResult']
