from . import WaveGrowthModels2D  # noqa: F401
from .WaveGrowthModels2D import WaveGrowth2D  # noqa: F401
from .WaveGrowthModels2DEnsemble import WaveGrowth2DEnsemble  # noqa: F401
