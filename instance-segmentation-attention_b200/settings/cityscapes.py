"""Cityscapes-shaped settings (1024x2048 net input, up to 64 instances) for BASELINE.json config 4.
No such class exists in the reference; fields follow settings/CVPPP."""
from .cvppp import ModelSettings as _CVPPPModelSettings
from .cvppp import TrainingSettings as _CVPPPTrainingSettings


class ModelSettings(_CVPPPModelSettings):

    def __init__(self):
        super(ModelSettings, self).__init__()
        self.MAX_N_OBJECTS = 64
        self.IMAGE_HEIGHT = 1024
        self.IMAGE_WIDTH = 2048
        self.MEAN = [0.485, 0.456, 0.406]
        self.STD = [0.229, 0.224, 0.225]
        self.D_MODEL = 32
        self.D_K = 16
        self.D_V = 16
        self.N_OBJECTS_PREDICTION = 64


class TrainingSettings(_CVPPPTrainingSettings):

    def __init__(self):
        super(TrainingSettings, self).__init__()
        self.MAX_N_OBJECTS = 64
        self.IMAGE_HEIGHT = 1024
        self.IMAGE_WIDTH = 2048
        # street scenes have an up: horizontal flips only
        self.VERTICAL_FLIPPING = False
        self.TRANSPOSING = False
        self.ROTATION_90X = False
        self.ROTATION = False
