from jamie_b200.evaluation import (foscttm, label_transfer_accuracy, imputation_auroc, imputation_correlation,  # noqa: F401
                                   kneighbors, knn_impute, mean_feature_r, silhouette_samples, silhouette_score,
                                   test_closer, test_LabelTA)
