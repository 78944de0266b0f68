from .fftpower import FFTPower, FFTBase, ProjectedFFTPower, project_to_basis
from .fftcorr import FFTCorr
from .fftrecon import FFTRecon
from .fof import FOF
from .paircount import SimulationBoxPairCount, SimulationBox2PCF
from .convpower import ConvolvedFFTPower, FKPCatalog, FKPWeightFromNbar, FKPCatalogMesh

FKPPower = ConvolvedFFTPower

__all__ = ['FFTCorr', 'FOF', 'SimulationBoxPairCount', 'SimulationBox2PCF', 'FFTRecon', 'FFTPower', 'ProjectedFFTPower', 'FFTBase', 'project_to_basis', 'ConvolvedFFTPower', 'FKPPower', 'FKPCatalog',
           'FKPWeightFromNbar', 'FKPCatalogMesh']
