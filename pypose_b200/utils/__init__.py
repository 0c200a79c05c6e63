from .io import read_bal, read_g2o
from .stepper import ReduceToBason
