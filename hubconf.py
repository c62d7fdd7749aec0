"""torch.hub entry points -- same names, defaults and `dependencies` contract as the reference's hubconf.py:1-34."""
dependencies = ['torch', 'numpy']      # the reference also lists scipy / sklearn / cv2 / ...: their arithmetic runs in libttk here

import os
import sys
import zipfile

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from upliftingtabletennis_b200.interface import BallDetector, TableDetector, TableTennisPipeline, _get_weights_path  # noqa: E402

IMAGES_ZIP_URL = "https://mediastore.rz.uni-augsburg.de/get/51XbRH38ZY/"
IMAGES_ZIP_FILENAME = "example_images.zip"


def ball_detection(model_name='segformerpp_b2', dtype=None, **kwargs):
    """Loads the Ball Detection Model.  B200 kernels exist for 'wasb' and 'vitpose'; the reference's default name is kept, but
    segformer++ is not part of the reference repository and raises NotImplementedError before anything is downloaded.
    dtype: 'tf32' (WASB default: tensor cores at the precision class of the reference's cuDNN convolutions), 'tf32x3' (ViTPose
    default, WASB on request: float32-class results on the tensor cores), 'fp32' (SIMT), 'bf16', 'fp16' (WASB / HRNet only: the bf16 kernels
    with fp16 storage)."""
    return BallDetector(model_name=model_name, dtype=dtype)


def table_detection(model_name='segformerpp_b2', dtype=None, **kwargs):
    """Loads the Table Detection Model.  B200 kernels exist for 'hrnet' and 'vitpose'.  dtype: as for ball_detection."""
    return TableDetector(model_name=model_name, dtype=dtype)


def full_pipeline(dtype=None, **kwargs):
    """Loads the End-to-End Pipeline (Ball + Table + Uplifting).  kwargs: ball_model / ball_model_aux / table_model / table_model_aux."""
    return TableTennisPipeline(dtype=dtype, **kwargs)


def download_example_images(local_folder='example_images'):
    """hubconf.py:34-88: fetch and unpack the example frames (needs network)."""
    if os.path.exists(local_folder) and len(os.listdir(local_folder)) > 0:
        print(f"Images already present in '{local_folder}'. Skipping download.")
        return local_folder
    os.makedirs(local_folder, exist_ok=True)
    zip_path = os.path.join(local_folder, IMAGES_ZIP_FILENAME)
    if not os.path.exists(zip_path):
        try:
            torch.hub.download_url_to_file(IMAGES_ZIP_URL, zip_path, progress=True)
        except Exception as e:
            if os.path.exists(zip_path):
                os.remove(zip_path)
            raise RuntimeError(f"Failed to download images: {e}")
    try:
        with zipfile.ZipFile(zip_path, 'r') as zip_ref:
            zip_ref.extractall(local_folder)
    except Exception as e:
        raise RuntimeError(f"Failed to extract images: {e}")
    if os.path.exists(zip_path):
        os.remove(zip_path)
    return local_folder
