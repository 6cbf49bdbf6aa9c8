"""
String enums of the reference's public API for the kernel-model path.

Mirrors /root/reference/homonim/enums.py:22-53 (same member names and string values, so that
``Model('gain-offset')`` / ``ProcCrs('ref')`` and YAML/CLI strings written for homonim keep working).
"""
from enum import Enum


class Model(str, Enum):
    """ Linear model variants for correcting to surface reflectance (reference enums.py:22-42). """
    gain = 'gain'
    """ Gain-only model: ``ref ~ gain * src``. """
    gain_blk_offset = 'gain-blk-offset'
    """ Gain-only model fitted to a source block that was first offset-normalised against the reference. """
    gain_offset = 'gain-offset'
    """ Full linear model: ``ref ~ gain * src + offset``. """


class ProcCrs(str, Enum):
    """ Pixel grid in which the models are fitted (reference enums.py:45-53). """
    auto = 'auto'
    """ The coarser of the source and reference grids. """
    src = 'src'
    """ The source image grid. """
    ref = 'ref'
    """ The reference image grid. """


class Resampling(str, Enum):
    """
    Resampling methods understood by the B200 path.  Stand-in for ``rasterio.enums.Resampling`` on the
    ``downsampling`` / ``upsampling`` config keys (reference kernel_model.py:98-136): members compare equal to their
    names, and ``Resampling.coerce`` accepts rasterio's enum members, names or this enum.
    """
    nearest = 'nearest'
    bilinear = 'bilinear'
    cubic = 'cubic'
    cubic_spline = 'cubic_spline'
    lanczos = 'lanczos'
    average = 'average'
    mode = 'mode'
    max = 'max'
    min = 'min'
    med = 'med'
    q1 = 'q1'
    q3 = 'q3'

    @classmethod
    def coerce(cls, value) -> 'Resampling':
        if isinstance(value, cls):
            return value
        name = getattr(value, 'name', value)
        return cls(str(name))
