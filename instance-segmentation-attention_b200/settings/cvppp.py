"""CVPPP settings: field names and values of
/root/reference/code/settings/CVPPP/data_settings.py:15-19, model_settings.py:12-29,
training_settings.py:10-60 (the hard-coded /media/snowday paths are dropped)."""
import os


class DataSettings(object):

    def __init__(self):
        self.BASE_PATH = os.path.abspath(os.path.join(os.path.dirname(__file__), os.path.pardir, os.path.pardir))
        self.CLASS_WEIGHTS = None
        self.MAX_N_OBJECTS = 32
        self.N_CLASSES = 1 + 1


class ModelSettings(DataSettings):

    def __init__(self):
        super(ModelSettings, self).__init__()
        self.MEAN = [0.521697844321, 0.389775426267, 0.206216114391]
        self.STD = [0.212398291819, 0.151755427041, 0.113022107204]
        self.MODEL_NAME = 'ReSeg'
        self.USE_INSTANCE_SEGMENTATION = True
        self.USE_COORDINATES = False
        self.IMAGE_HEIGHT = 256
        self.IMAGE_WIDTH = 256
        self.DELTA_VAR = 0.5
        self.DELTA_DIST = 1.5
        self.NORM = 2
        # attention / embedding widths (reference: lib/archs/modules/config.py:22-26)
        self.N_HEAD = 2
        self.D_MODEL = 24
        self.D_K = 12
        self.D_V = 12
        self.D_INNER = 40
        self.N_RENET_UNITS = 100
        self.N_OBJECTS_PREDICTION = 16   # lib/model.py:496 hard-codes 16
        # trained instance-count head (archs.ReSeg(count_head=True)): each image is clustered with its own predicted count
        # instead of N_OBJECTS_PREDICTION
        self.COUNT_HEAD = False


class TrainingSettings(ModelSettings):

    def __init__(self):
        super(TrainingSettings, self).__init__()
        self.TRAINING_LMDB = os.path.join(self.BASE_PATH, 'data', 'processed', 'CVPPP', 'lmdb', 'training-lmdb')
        self.VALIDATION_LMDB = os.path.join(self.BASE_PATH, 'data', 'processed', 'CVPPP', 'lmdb', 'validation-lmdb')
        self.TRAIN_CNN = True
        self.OPTIMIZER = 'Adadelta'
        self.LEARNING_RATE = 1
        self.LR_DROP_FACTOR = 0.5
        self.LR_DROP_PATIENCE = 25
        self.WEIGHT_DECAY = 0.001
        self.CLIP_GRAD_NORM = 10.0
        self.HORIZONTAL_FLIPPING = True
        self.VERTICAL_FLIPPING = True
        self.TRANSPOSING = True
        self.ROTATION_90X = True
        self.ROTATION = True
        self.COLOR_JITTERING = False
        self.GRAYSCALING = False
        self.CHANNEL_SWAPPING = False
        self.GAMMA_ADJUSTMENT = False
        self.RESOLUTION_DEGRADING = False
        self.CRITERION = 'Multi'
        self.OPTIMIZE_BG = False
        self.CENTER_CUT = True
        self.SEED = 23
        self.USE_WAE = False
        self.load_model_path = ''
        self.load_decoder_model_path = ''
