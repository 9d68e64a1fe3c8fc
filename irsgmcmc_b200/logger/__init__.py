from .writers import (load_im_from_disk, load_field_from_disk, load_landmarks_from_disk, save_displacement_mean_and_std_dev,
                      save_field_to_disk, save_grid_to_disk, save_im_to_disk, save_landmarks_to_disk, save_sample,
                      save_variational_posterior_mean)
