from .AFs import AF_EI, AF_HF, AF_HF_Engineering, AF_LF, AF_LF_Engineering  # noqa: F401
from .BO_GP_plus import (BO, Visualize_BO, acquisition_table_argmax, prepare_candidate_table,  # noqa: F401
                         prepare_candidate_table_on_device,
                         score_prepared, to_device)
from .qbatch import (optimize_acquisition_qbatch, optimize_gibbon, optimize_knowledge_gradient,  # noqa: F401
                     optimize_posterior_mean)
