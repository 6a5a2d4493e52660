"""B200 implementation of the parts of `icon_registration==1.1.2` the reference calls
(oai_analysis/registration.py:2-4,20,25; oai_analysis/dask_processing.py:51-53,77,85):
pretrained_models.OAI_knees_gradICON_model, itk_wrapper.register_pair, and the networks/wrappers behind them."""
from . import itk_wrapper, losses, networks, pretrained_models  # noqa: F401
