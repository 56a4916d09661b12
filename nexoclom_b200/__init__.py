"""nexoclom_b200 -- B200-native hot path of the nexoclom exosphere model.

Public API mirrors the reference's ``nexoclom/__init__.py:9-14``.  Importing the
package needs neither PostgreSQL nor astropy; creating an ``Output`` /
``ModelImage`` / ``ModelImageCube`` / ``ModelDensity`` / ``ModelDeposition`` /
``ModelIonization`` / ``ModelTrajectoryImage`` / ``ModelTrajectoryDensity`` / ``LOSResult`` /
``LOSSpectrum`` needs the built CUDA library and a
GPU (there is no CPU fallback).
"""
from .Input import Input
from .Output import Output
from .ModelImage import ModelImage
from .ModelImageCube import ModelImageCube
from .ModelDensity import ModelDensity
from .ModelDeposition import ModelDeposition
from .ModelIonization import ModelIonization
from .ModelTrajectory import ModelTrajectoryImage, ModelTrajectoryDensity
from .LOSResult import LOSResult
from .LOSSpectrum import LOSSpectrum
from .LOSResultFitted import LOSResultFitted
from .solarsystem import SSObject
from .input_classes import InputError

__all__ = ['Input', 'Output', 'ModelImage', 'ModelImageCube', 'ModelDensity', 'ModelDeposition',
           'ModelIonization', 'ModelTrajectoryImage', 'ModelTrajectoryDensity', 'LOSResult', 'LOSSpectrum', 'LOSResultFitted', 'SSObject', 'InputError']
__version__ = '0.1.0'
